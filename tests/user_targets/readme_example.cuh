// The example of README.md, "Your own target": x[0] = t, x[1] = u = log sigma, x[2] = z = logit p
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const auto nu = d.real(field::nu)[0];               // field:: constants are generated from the data keys
        const T t = x[0], u = x[1], z = x[2];
        return -0.5 * (nu + 1) * log1p(t * t / nu)
               + d.real(field::a)[0] * u - d.real(field::b)[0] * exp(u)
               + d.real(field::alpha)[0] * log_inv_logit(z) + d.real(field::beta)[0] * log_inv_logit(-z);
    }
};
