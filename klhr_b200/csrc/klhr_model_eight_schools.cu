// klhr_b200 -- the launcher table of one Stan target, which instantiates every kernel for it (one translation unit
// per model so the build parallelises).  See klhr_models.cuh for the density itself.
// Both parametrisations of eight schools share this unit: they are small and read the same data.
#include "klhr_target.cuh"

namespace klhr {
extern const klhr_user_table_t kEightSchoolsNCLaunchers =
    TargetLaunchers<EightSchoolsNC<double>, EightSchoolsNC<float>>::table;
extern const klhr_user_table_t kEightSchoolsCLaunchers =
    TargetLaunchers<EightSchoolsC<double>, EightSchoolsC<float>>::table;
}  // namespace klhr
