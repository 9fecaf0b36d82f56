// klhr_b200 -- step/eval kernel instantiations for one Stan target (one translation unit
// per model so the build parallelises).  See klhr_models.cuh for the density itself.
#include "klhr_chain.cuh"
#include "klhr_mh.cuh"
#include "klhr_slice.cuh"

namespace klhr {
using M64_arma11 = Arma11<double>;
using M32_arma11 = Arma11<float>;
KLHR_DEFINE_MODEL(arma11, M64_arma11, M32_arma11)
KLHR_DEFINE_MODEL_CHAIN(arma11, M64_arma11, M32_arma11)
KLHR_DEFINE_MODEL_MH(arma11, M64_arma11, M32_arma11)
KLHR_DEFINE_MODEL_SLICE(arma11, M64_arma11, M32_arma11)
}  // namespace klhr
