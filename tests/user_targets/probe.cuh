// probe: lp = sum_k w_k f_k(x_k), one AD primitive per coordinate (D = 12), weights w from the data.  With w one-hot
// and a one-node line fit, the KL objective exposes f_k, f_k' and f_k'' of one primitive (tests/test_gpu_user_model.py).
struct Target {
    template <typename T, typename X, typename Data>
    __device__ static T log_density(const X& x, const Data& d) {
        using namespace klhr::ad;
        const auto w = d.real(field::w);
        return w[0] * exp(x[0]) + w[1] * log(x[1]) + w[2] * log1p(x[2]) + w[3] * expm1(x[3]) + w[4] * sqrt(x[4])
               + w[5] * square(x[5]) + w[6] * pow(x[6], 2.5) + w[7] * tanh(x[7]) + w[8] * log1p_exp(x[8])
               + w[9] * log_inv_logit(x[9]) + w[10] * fabs(x[10]) + w[11] * (1.0 / x[11]);
    }
};
