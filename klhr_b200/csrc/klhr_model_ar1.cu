// klhr_b200 -- the launcher table of one Stan target, which instantiates every kernel for it (one translation unit
// per model so the build parallelises).  See klhr_models.cuh for the density itself.
#include "klhr_target.cuh"

namespace klhr {
extern const klhr_user_table_t kAr1Launchers = TargetLaunchers<AR1<double>, AR1<float>>::table;
}  // namespace klhr
