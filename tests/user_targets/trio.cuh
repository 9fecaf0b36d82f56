// trio: K independent Student-t(nu) coordinates with scales s[K], then u = log sigma with sigma ~ Gamma(a, b), then
// z = logit p with p ~ Beta(alpha, beta).  D = K + 2.  Unconstrained scale, Jacobians included:
//   sigma^(a-1) e^(-b sigma) d sigma = e^(a u - b e^u) du,   p^(alpha-1) (1-p)^(beta-1) dp = p^alpha (1-p)^beta dz.
// Exact moments (oracle/user_models.py): E[u] = psi(a) - log b, Var u = psi'(a); E[z] = psi(alpha) - psi(beta),
// Var z = psi'(alpha) + psi'(beta); Var t_k = s_k^2 nu / (nu - 2).
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const int K = (int)d.size(field::s);
        const auto nu = d.real(field::nu)[0];
        const auto s = d.real(field::s);
        T lp{};
        for (int k = 0; k < K; ++k) {
            const T r = x[k] / s[k];
            lp -= 0.5 * (nu + 1) * log1p(r * r / nu);
        }
        const T u = x[K], z = x[K + 1];
        return lp + d.real(field::a)[0] * u - d.real(field::b)[0] * exp(u)
               + d.real(field::alpha)[0] * log_inv_logit(z) + d.real(field::beta)[0] * log_inv_logit(-z);
    }
};
