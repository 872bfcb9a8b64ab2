// smb200_plugin.cuh -- device side of a USER-DEFINED Op struct (compile with nvcc for sm_100a).
//
// The reference's recipe for adding an operation (README.md:86-133, "Extending with Custom
// Operations") is: (1) an Op struct with `apply`, (2) its `apply_simd` specialisations, (3) an
// operator that calls element_wise_op<T, MyOp<T>>.  On the device, step (2) becomes a
// `__device__ apply_device` and one registration -- no change to libsmb200.so:
//
//     // my_op.h (shared by host and device code)
//     template<typename T> struct MyOp {
//         static T apply(const T &a, const T &b) { return (a + b) * 2; }          // the definition (host oracle)
//         static int device_op() { return smb::op_id("MyOp"); }                    // looked up by name, see helpers.h
//     #ifdef __CUDACC__
//         static __device__ __forceinline__ T apply_device(T a, T b) { return (a + b) * 2; }
//     #endif
//     };
//     // my_op_device.cu (nvcc -gencode arch=compute_100a,code=sm_100a)
//     #include <smb200_plugin.cuh>
//     #include "my_op.h"
//     SMB_REGISTER_DEVICE_OP("MyOp", float, MyOp<float>);
//     SMB_REGISTER_DEVICE_OP("MyOp", int32_t, MyOp<int32_t>);
//
// The macros instantiate THIS library's kernel templates (k_stream: 128-bit streams; k_row: broadcast
// with fast-divmod index math; k_generic: arbitrary strides) over a functor that calls apply_device, and
// hand three launchers to smb_register_op (include/smb200.h).  element_wise_op / array_scalar_op with
// that Op then take every path a built-in op takes: views, host operands (staged), device sets, async.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <smb200.h>
#include "../simplemath_b200/csrc/smb_kernels.cuh"

namespace smb {
namespace plugin {

template<typename T> struct dtype_of;
template<> struct dtype_of<float> { static constexpr int value = SMB_F32; };
template<> struct dtype_of<double> { static constexpr int value = SMB_F64; };
template<> struct dtype_of<int32_t> { static constexpr int value = SMB_I32; };

// The functors the kernel templates apply: element index unused (only int pow needs it).
template<typename T, typename Op> struct BinFn {
    uint64_t lane_end;
    __device__ __forceinline__ T operator()(T a, T b, uint64_t) const { return Op::apply_device(a, b); }
};
template<typename T, typename Op> struct ScalarRightFn { // the scalar is the RIGHT operand (calculate.h:159,167)
    T v;
    uint64_t lane_end;
    __device__ __forceinline__ T operator()(T a, T, uint64_t) const { return Op::apply_device(a, v); }
};

// The plugin's translation unit carries its own (static) CUDA runtime, whose idea of the calling thread's
// current device is separate from the library's: make the launch device current here for the launch.
struct DeviceGuard {
    int saved = -1;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&saved) != cudaSuccess) saved = -1;
        if (saved != device) cudaSetDevice(device); else saved = -1;
    }
    ~DeviceGuard() { if (saved >= 0) cudaSetDevice(saved); }
};

inline unsigned grid_for(uint64_t items, uint64_t per_block, int sm_count, int ctas_per_sm) {
    uint64_t blocks = (items + per_block - 1) / per_block;
    if (blocks == 0) blocks = 1;
    if (ctas_per_sm > 0 && blocks > (uint64_t)sm_count * (uint64_t)ctas_per_sm) blocks = (uint64_t)sm_count * (uint64_t)ctas_per_sm;
    return (unsigned)(blocks < 0x7fffffffull ? blocks : 0x7fffffffull);
}

// Dense streams: vector kernel when the three addresses share a 16-byte phase (a short scalar head
// is peeled), the element-wise kernel otherwise -- the same dispatch as the built-in ops.
template<typename T, typename Fn, bool HAS_B>
inline int stream(const smb_launch_env *env, const T *a, const T *b, T *out, uint64_t n, Fn fn) {
    if (n == 0) return 0;
    const DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)env->stream;
    constexpr int VB = 16, UNROLL = 4;
    const uintptr_t ma = (uintptr_t)a % VB, mb = HAS_B ? (uintptr_t)b % VB : ma, mo = (uintptr_t)out % VB;
    if (ma == mb && ma == mo && ma % sizeof(T) == 0) {
        uint64_t head = ma ? (VB - ma) / sizeof(T) : 0;
        if (head > n) head = n;
        if (head) k_stream_unaligned<T, Fn, HAS_B><<<1, kBlock, 0, s>>>(a, b, out, head, 0, fn);
        const uint64_t rest = n - head;
        if (rest) {
            constexpr uint64_t per_block = (uint64_t)kBlock * UNROLL * (VB / sizeof(T));
            k_stream<T, Fn, HAS_B, VB, UNROLL><<<grid_for(rest, per_block, env->sm_count, 0), kBlock, 0, s>>>(
                a + head, HAS_B ? b + head : nullptr, out + head, rest, head, fn, kPdlWaitFirst);
        }
    } else {
        k_stream_unaligned<T, Fn, HAS_B><<<grid_for(n, kBlock, env->sm_count, 32), kBlock, 0, s>>>(a, b, out, n, 0, fn);
    }
    return (int)cudaGetLastError();
}

template<typename T, typename Op>
int launch_contiguous(const smb_launch_env *env, const void *a, const void *b, void *out, uint64_t n) {
    return stream<T, BinFn<T, Op>, true>(env, (const T *)a, (const T *)b, (T *)out, n, BinFn<T, Op>{0});
}
template<typename T, typename Op>
int launch_scalar(const smb_launch_env *env, const void *a, const void *scalar, void *out, uint64_t n) {
    return stream<T, ScalarRightFn<T, Op>, false>(env, (const T *)a, nullptr, (T *)out, n, ScalarRightFn<T, Op>{*(const T *)scalar, 0});
}
template<typename T, typename Op>
int launch_strided(const smb_launch_env *env, const void *a, const void *b, void *out, const void *table, int table_bytes,
                   int generic, int wide, int vector_bytes, int a_reused, int b_reused) {
    if (table_bytes != (int)sizeof(BcastTable)) return (int)cudaErrorInvalidValue; // header / library mismatch
    const BcastTable t = *(const BcastTable *)table;
    const DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)env->stream;
    using Fn = BinFn<T, Op>;
    const Fn fn{0};
    const T *pa = (const T *)a, *pb = (const T *)b;
    T *po = (T *)out;
    if (generic) {
        const unsigned grid = grid_for(t.count, kBlock, env->sm_count, 32);
        if (wide) k_generic<T, Fn, true><<<grid, kBlock, 0, s>>>(pa, pb, po, t, fn);
        else k_generic<T, Fn, false><<<grid, kBlock, 0, s>>>(pa, pb, po, t, fn);
    } else {
        constexpr int UNROLL = 2;
        const uint64_t nvec = t.count / (uint64_t)(vector_bytes / (int)sizeof(T));
        const unsigned grid = grid_for(nvec, (uint64_t)kBlock * UNROLL, env->sm_count, a_reused && b_reused ? 32 : 0);
        if (vector_bytes == 16) {
            if (wide) k_row<T, Fn, 16, true, UNROLL><<<grid, kBlock, 0, s>>>(pa, pb, po, t, a_reused, b_reused, fn);
            else k_row<T, Fn, 16, false, UNROLL><<<grid, kBlock, 0, s>>>(pa, pb, po, t, a_reused, b_reused, fn);
        } else {
            if (wide) k_row<T, Fn, (int)sizeof(T), true, UNROLL><<<grid, kBlock, 0, s>>>(pa, pb, po, t, a_reused, b_reused, fn);
            else k_row<T, Fn, (int)sizeof(T), false, UNROLL><<<grid, kBlock, 0, s>>>(pa, pb, po, t, a_reused, b_reused, fn);
        }
    }
    return (int)cudaGetLastError();
}

// Registers Op's device launchers for element type T under `name`; returns the op id (>= SMB_OP_USER).
template<typename T, typename Op>
int register_op(const char *name) {
    smb_user_op u;
    u.contiguous = &launch_contiguous<T, Op>;
    u.scalar = &launch_scalar<T, Op>;
    u.strided = &launch_strided<T, Op>;
    return smb_register_op(name, dtype_of<T>::value, &u);
}

} // namespace plugin
} // namespace smb

#define SMB_PLUGIN_CAT2(a, b) a##b
#define SMB_PLUGIN_CAT(a, b) SMB_PLUGIN_CAT2(a, b)
// At namespace scope of a .cu file: registers at load time (before main, or when the shared object is loaded).
#define SMB_REGISTER_DEVICE_OP(NAME, T, ...) \
    static const int SMB_PLUGIN_CAT(smb_registered_op_, __COUNTER__) = ::smb::plugin::register_op<T, __VA_ARGS__>(NAME)
