// posteriordb arma11 (Stan User's Guide ARMA(1,1)), restated from its Stan program; params [mu, a, b, v] with
// phi = tanh(a / 2), theta = tanh(b / 2), sigma = e^v
//   model { nu[1] = mu + phi * mu; err[1] = y[1] - nu[1];
//           for (t in 2:T) { nu[t] = mu + phi * y[t - 1] + theta * err[t - 1]; err[t] = y[t] - nu[t]; }
//           mu ~ normal(0, 10); phi ~ normal(0, 2); theta ~ normal(0, 2); sigma ~ cauchy(0, 5); err ~ normal(0, sigma); }
// log(d phi / da) = log 2 - |a| - 2 log1p(e^-|a|): finite where log(1 - phi^2) would round to -inf.
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T jacobian(const T& a) {
        using namespace klhr::ad;
        return 0.6931471805599453 - fabs(a) - 2.0 * log1p(exp(-fabs(a)));
    }
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const int n = (int)d.size(field::y);
        const auto y = d.real(field::y);
        const T mu = x[0], a = x[1], b = x[2], v = x[3];
        const T phi = tanh(0.5 * a), th = tanh(0.5 * b);
        T err = y[0] - mu * (1.0 + phi);
        T ss = err * err;
        for (int t = 1; t < n; ++t) {
            err = (y[t] - mu) - phi * y[t - 1] - th * err;
            ss += err * err;
        }
        return -mu * mu / 200.0 - (phi * phi + th * th) / 8.0 - log1p_exp(2.0 * v - 3.2188758248682006)
               + (1 - n) * v - 0.5 * exp(-2.0 * v) * ss + jacobian<T, X, Data>(a) + jacobian<T, X, Data>(b);
    }
};
