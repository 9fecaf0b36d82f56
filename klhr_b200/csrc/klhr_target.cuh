// klhr_b200 -- TargetLaunchers<M64, M32>::table: the launcher table of one target.  Taking it instantiates every kernel
// (octet step, chain, eval, KL, MH, slice) for M64 in fp64 and M32 in fp32.  klhr_api.cu runs built-in targets
// (klhr_model_*.cu) and user targets (klhr_user.cuh) alike through such a table.
#pragma once
#include "klhr_chain.cuh"
#include "klhr_mh.cuh"
#include "klhr_slice.cuh"

namespace klhr {

template <class M64, class M32>
struct TargetLaunchers {
    static int step(const void* a, int dtype, int family, int replay, int accum, void* st, void* info) {
        const StepArgs& s = *static_cast<const StepArgs*>(a);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        LaunchInfo* li = static_cast<LaunchInfo*>(info);
        return dtype == KLHR_F64 ? launch_step_typed<double, M64>(s, family, replay, accum, stream, li)
                                 : launch_step_typed<float, M32>(s, family, replay, accum, stream, li);
    }
    static int chain(const void* a, int dtype, int family, int replay, void* st, void* info) {
        const StepArgs& s = *static_cast<const StepArgs*>(a);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        LaunchInfo* li = static_cast<LaunchInfo*>(info);
        return dtype == KLHR_F64 ? launch_chain_typed<double, M64>(s, family, replay, stream, li)
                                 : launch_chain_typed<float, M32>(s, family, replay, stream, li);
    }
    static int eval(const void* mp, int dtype, const void* theta, void* lp, void* grad, int64_t B, void* st) {
        const ModelParams& m = *static_cast<const ModelParams*>(mp);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        return dtype == KLHR_F64 ? launch_eval_typed<double, M64>(m, theta, lp, grad, B, stream)
                                 : launch_eval_typed<float, M32>(m, theta, lp, grad, B, stream);
    }
    static int kl(const void* a, int dtype, int family, void* st) {
        const KlArgs& k = *static_cast<const KlArgs*>(a);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        return dtype == KLHR_F64 ? launch_kl_typed<double, M64>(k, family, stream)
                                 : launch_kl_typed<float, M32>(k, family, stream);
    }
    static int mh(const void* a, int dtype, void* st) {
        const MhArgs& m = *static_cast<const MhArgs*>(a);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        return dtype == KLHR_F64 ? launch_mh_typed<double, M64>(m, stream) : launch_mh_typed<float, M32>(m, stream);
    }
    static int slice(const void* a, int dtype, int replay, void* st) {
        const SliceArgs& s = *static_cast<const SliceArgs*>(a);
        const cudaStream_t stream = static_cast<cudaStream_t>(st);
        return dtype == KLHR_F64 ? launch_slice_typed<double, M64>(s, replay, stream)
                                 : launch_slice_typed<float, M32>(s, replay, stream);
    }
    static constexpr klhr_user_table_t table = {
        KLHR_ABI_VERSION, (int32_t)sizeof(StepArgs), (int32_t)sizeof(SliceArgs), (int32_t)sizeof(MhArgs),
        (int32_t)sizeof(KlArgs), (int32_t)sizeof(ModelParams), step, chain, eval, kl, mh, slice};
};

}  // namespace klhr
