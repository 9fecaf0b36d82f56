// Bayesian logistic regression, restated from its Stan program; params [alpha, beta_1..K]
//   data { int<lower=0> N; int<lower=1> K; matrix[N, K] x; array[N] int<lower=0, upper=1> y; }
//   model { alpha ~ normal(0, 2.5); beta ~ normal(0, 2.5); y ~ bernoulli_logit(alpha + x * beta); }
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const int N = (int)d.integer(field::N)[0], K = (int)d.integer(field::K)[0];
        const auto xm = d.real(field::x);
        const auto y = d.integer(field::y);
        T lp{};
        for (int k = 0; k <= K; ++k) lp -= x[k] * x[k] / 12.5;
        for (int i = 0; i < N; ++i) {
            T eta = x[0];
            for (int k = 0; k < K; ++k) eta += xm[(size_t)i * K + k] * x[k + 1];
            lp += y[i] * eta - log1p_exp(eta);
        }
        return lp;
    }
};
