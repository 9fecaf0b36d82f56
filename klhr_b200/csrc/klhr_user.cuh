// klhr_b200 -- UserModel<R, Target>: a target written by the user as one templated device function, run by every
// kernel the built-in targets run on (chain, octet step, slice, MH, eval, KL).
//
// The user's contract (README, "Your own target"):
//   struct Target {
//       template <typename T, typename X, typename Data>
//       __device__ static T log_density(const X& x, const Data& d);   // log density on the unconstrained scale
//   };
// x[i] is coordinate i of the point (T is R, klhr::ad::Dual<R> or klhr::ad::Tay2<R>); d.real(k)[i] is value i of data
// field k in R, d.size(k) its length and d.integer(k)[i] its values as int64_t when they are integers.  The field
// constants field::<key> are generated from the data keys (sorted, numbered from 0).
//
// Data of a KLHR_MODEL_USER descriptor (i1 = F fields):
//   data0  every field's values, flattened in C order and concatenated in field order, in the arithmetic type R;
//   data1  int64: a header of 3 F entries, (offset into data0, length, offset into data1 or -1) per field, then the
//          values of the integer fields.  Integer fields are in both buffers, so d.real(k) works for every field.
//
// The line restriction.  eval runs log_density once on Tay2<R> through a lazy accessor: x[i] is
// {theta_i + y rho_i, rho_i, 0}, so l(y), l'(y) and l''(y) come out of one pass and no D-vector is stored per chain;
// Coef keeps the theta and rho row pointers (kCoefKeepsRows) and l(0).  A closed-form model pays O(D) once per draw
// and O(1) per evaluation; a user model pays a whole log_density per evaluation, at about three times the arithmetic
// of a plain pass (the second-order chain rule of every operation).
//
// The gradient (log_density_gradient, the sinh family's gradient clip) runs one Dual<R> pass per component, lane k of
// the G lanes of a chain owning the components i = k mod G, plus one plain pass for the value on every lane (so the
// value is uniform and bitwise the log_density value).  With the exact clip of the sinh family (D <= 16) that is D Dual
// passes and one plain pass on every evaluation where it is active.
#pragma once
#include "klhr_ad.cuh"
#include "klhr_target.cuh"
#include "../../include/klhr_user.h"

namespace klhr {

// A data field, indexed like a pointer.  Every read is an explicit global load (__ldg): Coef holds these pointers next
// to the theta / rho row pointers, which are shared memory in most kernels, and with plain dereferences nvcc has been
// seen to infer the shared space for the data pointers too and emit shared-memory loads from global addresses.
template <typename V>
struct UserField {
    const V* p;
    __device__ __forceinline__ V operator[](int64_t i) const { return __ldg(p + i); }
};

template <typename R>
struct UserData {
    const R* re;
    const int64_t* tab;
    __device__ __forceinline__ UserField<R> real(int k) const { return {re + __ldg(tab + 3 * k)}; }
    __device__ __forceinline__ int64_t size(int k) const { return __ldg(tab + 3 * k + 1); }
    __device__ __forceinline__ UserField<int64_t> integer(int k) const { return {tab + __ldg(tab + 3 * k + 2)}; }
};

// the point theta
template <typename R>
struct UserRow {
    const R* th;
    __device__ __forceinline__ R operator[](int i) const { return th[i]; }
};

// theta + y rho as a second-order Taylor variable in y
template <typename R>
struct UserLine {
    const R* th;
    const R* rh;
    R y;
    __device__ __forceinline__ ad::Tay2<R> operator[](int i) const { return {th[i] + y * rh[i], rh[i], R(0)}; }
};

// theta with the tangent e_k
template <typename R>
struct UserTangent {
    const R* th;
    int k;
    __device__ __forceinline__ ad::Dual<R> operator[](int i) const { return {th[i], i == k ? R(1) : R(0)}; }
};

template <typename R, typename Target>
struct UserModel {
    using Self = UserModel<R, Target>;
    static constexpr bool kDenseCta = false;
    static constexpr bool kCoefKeepsRows = true;
    struct Coef { const R* th; const R* rh; UserData<R> d; R l0; };
    __device__ static __forceinline__ UserData<R> data_(const ModelParams& mp) {
        return {reinterpret_cast<const R*>(mp.p0), reinterpret_cast<const int64_t*>(mp.p1)};
    }
    // every lane runs the t = 0 pass: a uniform result without shuffles
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int, unsigned, const ModelParams& mp) {
        Coef c;
        c.th = th; c.rh = rh; c.d = data_(mp);
        c.l0 = Target::template log_density<R>(UserRow<R>{th}, c.d);
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const ad::Tay2<R> l = Target::template log_density<ad::Tay2<R>>(UserLine<R>{c.th, c.rh, y}, c.d);
        return jet_guard<R>(l.v - c.l0, l.d, l.s);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned, const ModelParams& mp) {
        const UserData<R> d = data_(mp);
        if (g)
            for (int i = lane; i < mp.D; i += G)
                g[i] = Target::template log_density<ad::Dual<R>>(UserTangent<R>{th, i}, d).d;
        return Target::template log_density<R>(UserRow<R>{th}, d);
    }
};

}  // namespace klhr

// Instantiates every kernel for UserModel<double, Target> and UserModel<float, Target> and exports the launcher table
// (include/klhr_user.h).  The generated translation unit of a user target ends with this macro.
#define KLHR_DEFINE_USER_TARGET(TARGET)                                                                        \
    extern "C" __attribute__((visibility("default"))) const klhr_user_table_t* klhr_user_table(void) {         \
        return &klhr::TargetLaunchers<klhr::UserModel<double, TARGET>, klhr::UserModel<float, TARGET>>::table; \
    }
