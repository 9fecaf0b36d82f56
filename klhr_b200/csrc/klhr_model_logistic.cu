// klhr_b200 -- step/eval kernel instantiations for one Stan target (one translation unit
// per model so the build parallelises).  See klhr_models.cuh for the density itself.
#include "klhr_chain.cuh"
#include "klhr_mh.cuh"
#include "klhr_slice.cuh"

namespace klhr {
using M64_logistic_regression = LogisticRegression<double>;
using M32_logistic_regression = LogisticRegression<float>;
KLHR_DEFINE_MODEL(logistic_regression, M64_logistic_regression, M32_logistic_regression)
KLHR_DEFINE_MODEL_CHAIN(logistic_regression, M64_logistic_regression, M32_logistic_regression)
KLHR_DEFINE_MODEL_MH(logistic_regression, M64_logistic_regression, M32_logistic_regression)
KLHR_DEFINE_MODEL_SLICE(logistic_regression, M64_logistic_regression, M32_logistic_regression)
}  // namespace klhr
