// klhr_b200 -- step/eval kernel instantiations for one Stan target (one translation unit
// per model so the build parallelises).  See klhr_models.cuh for the density itself.
// Both parametrisations of eight schools share this unit: they are small and read the same data.
#include "klhr_chain.cuh"
#include "klhr_mh.cuh"
#include "klhr_slice.cuh"

namespace klhr {
using M64_eight_schools_nc = EightSchoolsNC<double>;
using M32_eight_schools_nc = EightSchoolsNC<float>;
KLHR_DEFINE_MODEL(eight_schools_nc, M64_eight_schools_nc, M32_eight_schools_nc)
KLHR_DEFINE_MODEL_CHAIN(eight_schools_nc, M64_eight_schools_nc, M32_eight_schools_nc)
KLHR_DEFINE_MODEL_MH(eight_schools_nc, M64_eight_schools_nc, M32_eight_schools_nc)
KLHR_DEFINE_MODEL_SLICE(eight_schools_nc, M64_eight_schools_nc, M32_eight_schools_nc)

using M64_eight_schools_c = EightSchoolsC<double>;
using M32_eight_schools_c = EightSchoolsC<float>;
KLHR_DEFINE_MODEL(eight_schools_c, M64_eight_schools_c, M32_eight_schools_c)
KLHR_DEFINE_MODEL_CHAIN(eight_schools_c, M64_eight_schools_c, M32_eight_schools_c)
KLHR_DEFINE_MODEL_MH(eight_schools_c, M64_eight_schools_c, M32_eight_schools_c)
KLHR_DEFINE_MODEL_SLICE(eight_schools_c, M64_eight_schools_c, M32_eight_schools_c)
}  // namespace klhr
