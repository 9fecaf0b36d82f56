/* Entry point of a user target library: a shared object compiled from one user-written CUDA target
 * (klhr_b200/csrc/klhr_user.cuh, KLHR_DEFINE_USER_TARGET).  Its launcher table is handed to klhr_user_register of
 * libklhr_sm100.so (include/klhr_sm100.h), which then runs KLHR_MODEL_USER descriptors of that slot through it. */
#ifndef KLHR_USER_H_
#define KLHR_USER_H_

#include "klhr_sm100.h"

#ifdef __cplusplus
extern "C" {
#endif

const klhr_user_table_t* klhr_user_table(void);

#ifdef __cplusplus
}
#endif
#endif /* KLHR_USER_H_ */
