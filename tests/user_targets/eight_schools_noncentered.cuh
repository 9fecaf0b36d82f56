// posteriordb eight_schools_noncentered, restated from its Stan program; params [theta_trans_1..J, mu, u = log tau]
//   parameters { vector[J] theta_trans; real mu; real<lower=0> tau; }
//   model { theta_trans ~ normal(0, 1); y ~ normal(theta_trans * tau + mu, sigma); mu ~ normal(0, 5);
//           tau ~ cauchy(0, 5); }
// The half-Cauchy term on the unconstrained scale is -log1p(tau^2 / 25) + u = -log1p_exp(2u - log 25) + u.
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const int J = (int)d.integer(field::J)[0];
        const auto y = d.real(field::y);
        const auto sigma = d.real(field::sigma);
        const T mu = x[J], u = x[J + 1];
        const T tau = exp(u);
        T lp{};
        for (int j = 0; j < J; ++j) {
            const T tt = x[j];
            const T r = (y[j] - mu - tau * tt) / sigma[j];
            lp -= 0.5 * (tt * tt + r * r);
        }
        return lp - mu * mu / 50.0 - log1p_exp(2.0 * u - 3.2188758248682006) + u;
    }
};
