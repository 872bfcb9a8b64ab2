// smb_kernels.cuh -- the sm_100a kernels that replace the reference's three CPU
// loops (include/math/calculate.h):
//
//   k_stream   <- handle_contiguous_arrays (:101-134) and array_scalar_op (:137-169)
//                 dense streams, 128/256-bit vector loads+stores, grid-stride.
//   k_row      <- element_wise_op general loop (:47-98) when, after coalescing,
//                 both operands have inner stride 0 or 1: vectorised along the
//                 inner dim, outer index -> offset by fast-divmod.
//   k_generic  <- the same loop for arbitrary element strides (scalar gathers,
//                 coalesced stores).
//
// All are HBM-bound (0.08-0.25 flop/byte); no tensor cores, no TMEM.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "smb_math.cuh"
#include "smb_plan.h"

namespace smb {

constexpr int kBlock = 256; // threads per CTA of every kernel in this file
#ifndef SMB_STREAM_LOAD_HINT
#define SMB_STREAM_LOAD_HINT true // dense streams: L1::no_allocate loads (false: default caching loads)
#endif
#ifndef SMB_STREAM_STORE_HINT
#define SMB_STREAM_STORE_HINT true
#endif
// The pow tile body is one long basic block; without a fence ptxas sinks the next tile's loads
// to its end (no prefetch left) and holds every store until then.  A warp-level barrier is one
// instruction it will not move memory operations across.
#ifndef SMB_POW_SCHED_FENCE
#define SMB_POW_SCHED_FENCE() __syncwarp()
#endif
#ifndef SMB_POW64_MIN_BLOCKS
#define SMB_POW64_MIN_BLOCKS 3 // resident CTAs per SM the f64 pow kernel is compiled for
#endif
#ifndef SMB_POW_MIN_BLOCKS
#define SMB_POW_MIN_BLOCKS 3 // resident CTAs per SM the f32 pow kernel is compiled for
#endif
#ifndef SMB_DOT_MIN_BLOCKS
// k_dot: the 4-byte instantiations fit four CTAs per SM as they are; capping the f64 one to 64 registers for a fourth
// CTA was tried and lost (5.70 -> 5.32 TB/s: the spills cost more than the extra CTA hides), so it keeps its 70.
#define SMB_DOT_MIN_BLOCKS(T) (sizeof(T) == 8 ? 3 : 4)
#endif

// ---------------------------------------------------------------------------
// 16-byte and 32-byte global vector access with streaming cache hints.
// 256-bit LDG/STG is new with sm_100 (SASS LDG.E.256 / STG.E.256).
// Streaming operands are read once: L1 no-allocate + L2 evict-first keep them
// from displacing reused (broadcast) operands.
template<int BYTES> struct alignas(BYTES) RawVec { uint32_t w[BYTES / 4]; };

template<int BYTES, bool STREAMING> struct VecIO;

template<> struct VecIO<16, true> {
    static __device__ __forceinline__ RawVec<16> load(const void *p) {
        RawVec<16> v;
        asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ void store(void *p, const RawVec<16> &v) {
        asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};"
                     :: "l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
    }
};
// Same access without .nc: an ordinary (coherent) load, which ptxas will not move across a warp
// barrier -- used to pin the pow kernel's prefetch at the top of its tile.
__device__ __forceinline__ RawVec<16> load_stream_pinned(const RawVec<16> *p) {
    RawVec<16> v;
    asm volatile("ld.global.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ RawVec<32> load_stream_pinned(const RawVec<32> *p) {
    RawVec<32> v;
    asm volatile("ld.global.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]), "=r"(v.w[4]), "=r"(v.w[5]), "=r"(v.w[6]), "=r"(v.w[7])
                 : "l"(p) : "memory");
    return v;
}
template<> struct VecIO<16, false> {
    static __device__ __forceinline__ RawVec<16> load(const void *p) {
        RawVec<16> v;
        asm volatile("ld.global.nc.v4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ void store(void *p, const RawVec<16> &v) {
        asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};"
                     :: "l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
    }
};
template<> struct VecIO<32, true> {
    static __device__ __forceinline__ RawVec<32> load(const void *p) {
        RawVec<32> v;
        asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]),
                       "=r"(v.w[4]), "=r"(v.w[5]), "=r"(v.w[6]), "=r"(v.w[7]) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ void store(void *p, const RawVec<32> &v) {
        asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                     :: "l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]),
                        "r"(v.w[4]), "r"(v.w[5]), "r"(v.w[6]), "r"(v.w[7]) : "memory");
    }
};
template<> struct VecIO<32, false> {
    static __device__ __forceinline__ RawVec<32> load(const void *p) {
        RawVec<32> v;
        asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]),
                       "=r"(v.w[4]), "=r"(v.w[5]), "=r"(v.w[6]), "=r"(v.w[7]) : "l"(p));
        return v;
    }
    static __device__ __forceinline__ void store(void *p, const RawVec<32> &v) {
        asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                     :: "l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]),
                        "r"(v.w[4]), "r"(v.w[5]), "r"(v.w[6]), "r"(v.w[7]) : "memory");
    }
};

template<typename T, int BYTES> union Pack {
    RawVec<BYTES> raw;
    T e[BYTES / sizeof(T)];
    __device__ __forceinline__ Pack() {}
};

// ---------------------------------------------------------------------------
// mbarrier + 1-D bulk copy (TMA engine, SASS UBLKCP): used to stage the pow lookup tables in shared
// memory with one instruction instead of a load/store loop.
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(smem)), "l"(gmem), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}

// ---------------------------------------------------------------------------
// Programmatic dependent launch (griddepcontrol, sm_90+).  Every participating kernel lets the next
// launch on its stream become resident as soon as all of its own CTAs have started
// (launch_dependents first thing), and waits for the PREVIOUS launch to complete and flush either
// before its first global access (kPdlWaitFirst: the host saw a data hazard, or the stream is not
// the library's own) or just before it exits (no hazard: the two grids overlap, and this grid's
// completion still implies the previous one's).  Both instructions are no-ops in a launch without
// the programmatic-stream-serialisation attribute.  The host side is in smb_runtime.inl (pdl_decide).
constexpr uint32_t kPdlWaitFirst = 1u;
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// A launch that must wait for its predecessors lets ITS dependents in only after the wait has returned: the host drops its
// record of earlier launches' operand ranges at such a launch ("when its work starts, everything before it is done"), and a
// dependent admitted before the wait could start -- and read what an earlier, still running grid writes -- while this grid is
// still blocked in griddepcontrol.wait.
__device__ __forceinline__ void pdl_enter(uint32_t flags) {
    if (flags & kPdlWaitFirst) { pdl_wait(); pdl_launch_dependents(); }
    else pdl_launch_dependents();
}
__device__ __forceinline__ void pdl_exit(uint32_t flags) {
    if (!(flags & kPdlWaitFirst)) pdl_wait();
}

// ---------------------------------------------------------------------------
// Functors: what a launch applies to (a[i], b[i]).  `lane` tells the i32 pow
// instantiation whether flat element i is one the reference computes in an
// AVX2 lane (wrapping) or with scalar Op::apply (through double); see
// smb_math.cuh.  Every other (Op, T) ignores it.
template<int OP, typename T> struct BinaryFn {
    uint64_t lane_end; // elements with flat index < lane_end use lane semantics
    __device__ __forceinline__ T operator()(T a, T b, uint64_t) const { return DevOp<OP, T>::apply(a, b); }
};
template<> struct BinaryFn<OP_POW, int32_t> {
    uint64_t lane_end;
    __device__ __forceinline__ int32_t operator()(int32_t a, int32_t b, uint64_t i) const {
        return i < lane_end ? powi_lane(a, b) : powi_scalar(a, b);
    }
};

// array (op) scalar: the scalar is the RIGHT operand (calculate.h:159,167).
template<int OP, typename T> struct ScalarFn {
    T v;
    uint64_t lane_end;
    __device__ __forceinline__ T operator()(T a, T, uint64_t) const { return DevOp<OP, T>::apply(a, v); }
};
template<> struct ScalarFn<OP_POW, int32_t> {
    int32_t v;
    uint64_t lane_end;
    __device__ __forceinline__ int32_t operator()(int32_t a, int32_t, uint64_t i) const {
        return i < lane_end ? powi_lane(a, v) : powi_scalar(a, v);
    }
};
// sm::pow(arr, y) for float: pairs of elements go through the table-driven
// packed core (smb_math.cuh); whatever it declines -- specials, denormal inputs,
// results near overflow / underflow -- takes the FP64 reference-accuracy path,
// kept out of line so the hot loop stays small.
__device__ __noinline__ float pow_f32_slow(float x, PowExpF32 pe) { return pow_f32(x, pe); }

static __device__ const PowTabLog d_pow_log_tab[SMB_POW_LOG_ENTRIES] = SMB_POW_LOG_TABLE_INIT;   // small-y: {invc, -log2 invc}
static __device__ const PowTabLog d_pow_logc_tab[SMB_POW_LOG_ENTRIES] = SMB_POW_LOGC_TABLE_INIT; // large-y: {c, log2 c}
static __device__ const PowTabExp d_pow_exp_tab[SMB_POW_EXP_ENTRIES] = SMB_POW_EXP_TABLE_INIT;

// The replicated shared-memory layout of the two f32 pow tables, kept ready-made in global memory
// ([0] small-y, [1] large-y; 24 KB each, L2 resident) so that a CTA stages them with ONE bulk copy
// instead of ~60 instructions per thread -- which is what lets the pow grid be many waves deep
// (a few tiles per CTA).  Built once per device by k_pow_image_init (smb_runtime.inl: init_ctx).
static __device__ __align__(128) SmbPowTabs g_pow_image[2];
__global__ void k_pow_image_init() {
    const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
    for (int v = 0; v < 2; ++v) {
        const PowTabLog *src = v == 0 ? d_pow_log_tab : d_pow_logc_tab;
        for (int i = t0; i < SMB_POW_LOG_ENTRIES * SMB_POW_LOG_STRIDE; i += stride) g_pow_image[v].log[i] = src[i / SMB_POW_LOG_STRIDE];
        for (int i = t0; i < SMB_POW_EXP_ENTRIES * SMB_POW_EXP_STRIDE; i += stride) g_pow_image[v].exp[i] = d_pow_exp_tab[i / SMB_POW_EXP_STRIDE];
    }
}

// The reference-accuracy path alone: exponents the fast core cannot take (|y| >= 2^64 or
// y * log2 x denormal), and the scalar-access kernels.
struct PowF32SlowFn {
    PowExpF32 pe;
    uint64_t lane_end;
    __device__ __forceinline__ float operator()(float a, float, uint64_t) const { return pow_f32_slow(a, pe); }
    static PowF32SlowFn make(float y, uint64_t lane_end_) { return PowF32SlowFn{classify_exp(y), lane_end_}; }
};
template<> struct ScalarFn<OP_POW, float> : PowF32SlowFn {};

// The host only launches this functor when pow_f32_fast_ok(pe); the variant (TIER, SIGN,
// Y_LT_1) is picked from the uniform exponent, see pow_f32_pair_fast.
template<int TIER, int SIGN, bool Y_LT_1> struct PowF32Fn {
    static constexpr bool PAIRWISE = true;    // stream_vec feeds two elements per call
    static constexpr bool POW_TABLES = true;  // k_stream stages the lookup tables in shared memory
    PowExpF32 pe;  // exponent classified once on the host
    uint64_t lane_end;
    PowLane lane;  // this thread's replica offsets into the shared-memory tables
    uint64_t *tab_bar; // mbarrier the table copy completes on
    __device__ __forceinline__ float operator()(float a, float, uint64_t) const { return pow_f32_slow(a, pe); }
    __device__ __forceinline__ float slow(float a) const { return pow_f32(a, pe); } // inlined, see pow_tile
    __device__ __forceinline__ float slow_call(float a) const { return pow_f32_slow(a, pe); } // out of line (ragged tile)
    // Two elements through the branch-free fast core; false = redo on the slow path.
    __device__ __forceinline__ bool pair(float a0, float a1, float &r0, float &r1) const {
        return pow_f32_pair_fast<TIER, SIGN, Y_LT_1>(a0, a1, pe.y, lane, nullptr, nullptr, &r0, &r1);
    }
    // Lookup tables, L2 -> shared memory once per CTA, each entry replicated across the lanes
    // of a wavefront (24 KB) so the per-lane lookups never conflict; see smb_math.cuh.
    // block_init only ISSUES the copy (one cp.async.bulk of the ready-made image); block_wait is
    // called after the CTA's first tile loads are in flight, so the two latencies overlap.
    __device__ __forceinline__ void block_init() {
        __shared__ __align__(8) uint64_t bar;
        if (threadIdx.x == 0) {
            mbar_init(&bar, 1);
            mbar_expect_tx(&bar, (uint32_t)sizeof(SmbPowTabs));
            bulk_g2s(&smb_s_pow, &g_pow_image[TIER != POW_TIER_LARGE ? 0 : 1], (uint32_t)sizeof(SmbPowTabs), &bar);
        }
        lane = pow_lane(threadIdx.x, lane.c);
        tab_bar = &bar;
        __syncthreads(); // the barrier is initialised before anyone waits on it
    }
    __device__ __forceinline__ void block_wait() {
        mbar_wait(tab_bar, 0);
        // the lookups name the table from inline PTX; tie them to the wait through the lane offsets
        asm volatile("" : "+r"(lane.log_off), "+r"(lane.exp_off) :: "memory");
    }
    static PowF32Fn make(float y, uint64_t lane_end_) {
        PowF32Fn fn;
        fn.pe = classify_exp(y);
        fn.lane_end = lane_end_;
        fn.lane = PowLane{0, 0, pow_consts()}; // offsets set per thread in block_init; the constants ride in as kernel parameters
        fn.tab_bar = nullptr;
        return fn;
    }
};
// sm::pow(a (op) b, y) in ONE pass at the pow kernel's speed (the ≤ 3-leaf contiguous case of a fused chain,
// smb_chain: leaf (op) leaf, then pow by a constant): the same functor with a binary pre-operator applied to the two
// loaded operands -- rounded to float by the same DevOp bodies the separate operator uses, so the result is
// bit-identical to `add` followed by the pow kernel.  The pre-operator is a run-time (uniform) code, not a template
// parameter: one instantiation per pow variant instead of six.
enum { PRE_ADD = 0, PRE_SUB = 1, PRE_MUL = 2, PRE_DIV = 3, PRE_RSUB = 4, PRE_RDIV = 5 };
template<int TIER, int SIGN, bool Y_LT_1> struct PowF32FnPre : PowF32Fn<TIER, SIGN, Y_LT_1> {
    static constexpr bool PREOP = true;
    static constexpr int UNROLL_OVERRIDE = 2; // two operand streams: half the vectors per thread keep the register buffers the same size
    int pre_op;
    __device__ __forceinline__ float pre(float a, float b) const {
        switch (pre_op) { // uniform
            case PRE_ADD: return DevOp<OP_ADD, float>::apply(a, b);
            case PRE_SUB: return DevOp<OP_SUB, float>::apply(a, b);
            case PRE_MUL: return DevOp<OP_MUL, float>::apply(a, b);
            case PRE_DIV: return DevOp<OP_DIV, float>::apply(a, b);
            case PRE_RSUB: return DevOp<OP_SUB, float>::apply(b, a);
            default: return DevOp<OP_DIV, float>::apply(b, a);
        }
    }
    __device__ __forceinline__ float operator()(float a, float b, uint64_t) const { return pow_f32_slow(pre(a, b), this->pe); }
    static PowF32FnPre make(float y, uint64_t lane_end_, int pre_op_) {
        PowF32FnPre fn;
        static_cast<PowF32Fn<TIER, SIGN, Y_LT_1> &>(fn) = PowF32Fn<TIER, SIGN, Y_LT_1>::make(y, lane_end_);
        fn.pre_op = pre_op_;
        return fn;
    }
};
template<typename Fn, typename = void> struct fn_preop : std::false_type {};
template<typename Fn> struct fn_preop<Fn, std::void_t<decltype(Fn::PREOP)>> : std::bool_constant<Fn::PREOP> {};
// sm::pow(a (op) constant, y) -- the same idea with ONE operand stream: the pre-operator combines the loaded element with a
// uniform constant (either operand order), so the kernel is the plain pow kernel plus one instruction per element.
template<int TIER, int SIGN, bool Y_LT_1> struct PowF32FnPre1 : PowF32Fn<TIER, SIGN, Y_LT_1> {
    static constexpr bool PREOP1 = true;
    // a + c, a - c, c - a and a * c are ONE fma with uniform operands -- fma(a, 1, c), fma(a, 1, -c), fma(a, -1, c),
    // fma(a, c, -0.0) round exactly like the add / subtract / multiply they stand for (signed zeros included) -- so the
    // pre-operator costs one instruction per element and no branch.  (The two divisions stay on the chain kernel: an
    // inlined, predicated division per element cost this kernel 8 %.)
    float pre_mul, pre_add;
    __device__ __forceinline__ float pre1(float a) const { return __fmaf_rn(a, pre_mul, pre_add); }
    __device__ __forceinline__ float operator()(float a, float, uint64_t) const { return pow_f32_slow(pre1(a), this->pe); }
    static PowF32FnPre1 make(float y, uint64_t lane_end_, int pre_op_, float c) { // PRE_ADD, PRE_SUB, PRE_RSUB or PRE_MUL
        PowF32FnPre1 fn;
        static_cast<PowF32Fn<TIER, SIGN, Y_LT_1> &>(fn) = PowF32Fn<TIER, SIGN, Y_LT_1>::make(y, lane_end_);
        fn.pre_mul = pre_op_ == PRE_MUL ? c : pre_op_ == PRE_RSUB ? -1.0f : 1.0f;
        fn.pre_add = pre_op_ == PRE_MUL ? -0.0f : pre_op_ == PRE_SUB ? -c : c;
        return fn;
    }
};
template<typename Fn, typename = void> struct fn_preop1 : std::false_type {};
template<typename Fn> struct fn_preop1<Fn, std::void_t<decltype(Fn::PREOP1)>> : std::bool_constant<Fn::PREOP1> {};
template<typename T, typename Fn> __device__ __forceinline__ T apply_pre1(const Fn &fn, T a) {
    if constexpr (fn_preop1<Fn>::value) return fn.pre1(a);
    else return a;
}

// sm::pow(arr, y) for double: table-driven fast core per element, double-double
// reference-accuracy path (out of line) for whatever it declines.
__device__ __noinline__ double pow_f64_slow(double x, PowExpF64 pe) { return pow_f64(x, pe); }

static __device__ const PowTabLog64 d_pow64_log_tab[SMB_POW_LOG_ENTRIES] = SMB_POW64_LOG_TABLE_INIT;
static __device__ const PowTabExp64 d_pow64_exp_tab[SMB_POW_EXP_ENTRIES] = SMB_POW64_EXP_TABLE_INIT;

template<bool SMALL_Y, bool ODD_Y> struct PowF64Fn {
    static constexpr bool CHECKED = true;
    static constexpr bool POW_TABLES = true;
    PowExpF64 pe;
    uint64_t lane_end;
    int fast_ok;
    uint64_t sign_reject;
    const PowTabLog64A *tab_a;
    const PowTabLog64B *tab_b;
    const PowTabExp64 *tab_exp;
    __device__ __forceinline__ double operator()(double a, double, uint64_t) const { return pow_f64_slow(a, pe); }
    __device__ __forceinline__ double slow(double a) const { return pow_f64(a, pe); } // inlined, see pow_tile
    __device__ __forceinline__ bool fast(double a, double &r) const {
        return pow_f64_fast<SMALL_Y, ODD_Y>(a, pe.y, sign_reject, tab_a, tab_b, tab_exp, &r) && fast_ok != 0;
    }
    __device__ __forceinline__ void block_wait() {}
    __device__ __forceinline__ void block_init() { // 40 KB, every entry replicated per wavefront lane
        __shared__ __align__(16) PowTabLog64A s_a[SMB_POW_LOG_ENTRIES * SMB_POW64_A_STRIDE];
        __shared__ __align__(16) PowTabLog64B s_b[SMB_POW_LOG_ENTRIES * SMB_POW64_B_STRIDE];
        __shared__ __align__(16) PowTabExp64 s_exp[SMB_POW_EXP_ENTRIES * SMB_POW64_EXP_STRIDE];
        for (int i = threadIdx.x; i < SMB_POW_LOG_ENTRIES * SMB_POW64_A_STRIDE; i += kBlock) {
            const PowTabLog64 e = d_pow64_log_tab[i / SMB_POW64_A_STRIDE];
            s_a[i].c = e.c;
            s_a[i].l_hi = e.l_hi;
        }
        for (int i = threadIdx.x; i < SMB_POW_LOG_ENTRIES * SMB_POW64_B_STRIDE; i += kBlock)
            s_b[i].l_lo = d_pow64_log_tab[i / SMB_POW64_B_STRIDE].l_lo;
        for (int i = threadIdx.x; i < SMB_POW_EXP_ENTRIES * SMB_POW64_EXP_STRIDE; i += kBlock)
            s_exp[i] = d_pow64_exp_tab[i / SMB_POW64_EXP_STRIDE];
        __syncthreads();
        tab_a = s_a + (threadIdx.x & (SMB_POW64_A_STRIDE - 1));
        tab_b = s_b + (threadIdx.x & (SMB_POW64_B_STRIDE - 1));
        tab_exp = s_exp + (threadIdx.x & (SMB_POW64_EXP_STRIDE - 1));
    }
    static PowF64Fn make(double y, uint64_t lane_end_) {
        PowF64Fn fn;
        fn.pe = classify_exp(y);
        fn.lane_end = lane_end_;
        fn.fast_ok = pow_f64_fast_ok(fn.pe) ? 1 : 0;
        fn.sign_reject = fn.pe.y_is_int ? 0ull : 0x8000000000000000ull;
        fn.tab_a = nullptr;
        fn.tab_b = nullptr;
        fn.tab_exp = nullptr;
        return fn;
    }
};
template<> struct ScalarFn<OP_POW, double> : PowF64Fn<false, true> {};
// sm::pow(a (op) b, y) and sm::pow(a (op) constant, y) for double: the f64 pow kernel with a pre-operator, like PowF32FnPre /
// PowF32FnPre1 (same DevOp rounding of the intermediate, same pow variant: bit-identical to the two eager operators).  Without them
// a double chain with a pow step runs the double-double reference path per element (k_chain has no f64 table staging) -- slower than
// the eager operators it was meant to fuse.
template<bool SMALL_Y, bool ODD_Y> struct PowF64FnPre : PowF64Fn<SMALL_Y, ODD_Y> {
    static constexpr bool PREOP = true;
    static constexpr int UNROLL_OVERRIDE = 2; // two operand streams: half the vectors per thread keep the register buffers the same size
    int pre_op;
    __device__ __forceinline__ double pre(double a, double b) const {
        switch (pre_op) { // uniform
            case PRE_ADD: return DevOp<OP_ADD, double>::apply(a, b);
            case PRE_SUB: return DevOp<OP_SUB, double>::apply(a, b);
            case PRE_MUL: return DevOp<OP_MUL, double>::apply(a, b);
            case PRE_DIV: return DevOp<OP_DIV, double>::apply(a, b);
            case PRE_RSUB: return DevOp<OP_SUB, double>::apply(b, a);
            default: return DevOp<OP_DIV, double>::apply(b, a);
        }
    }
    __device__ __forceinline__ double operator()(double a, double b, uint64_t) const { return pow_f64_slow(pre(a, b), this->pe); }
    static PowF64FnPre make(double y, uint64_t lane_end_, int pre_op_) {
        PowF64FnPre fn;
        static_cast<PowF64Fn<SMALL_Y, ODD_Y> &>(fn) = PowF64Fn<SMALL_Y, ODD_Y>::make(y, lane_end_);
        fn.pre_op = pre_op_;
        return fn;
    }
};
template<bool SMALL_Y, bool ODD_Y> struct PowF64FnPre1 : PowF64Fn<SMALL_Y, ODD_Y> {
    static constexpr bool PREOP1 = true;
    double pre_mul, pre_add; // a + c, a - c, c - a, a * c as ONE fma with uniform operands (see PowF32FnPre1)
    __device__ __forceinline__ double pre1(double a) const { return __fma_rn(a, pre_mul, pre_add); }
    __device__ __forceinline__ double operator()(double a, double, uint64_t) const { return pow_f64_slow(pre1(a), this->pe); }
    static PowF64FnPre1 make(double y, uint64_t lane_end_, int pre_op_, double c) { // PRE_ADD, PRE_SUB, PRE_RSUB or PRE_MUL
        PowF64FnPre1 fn;
        static_cast<PowF64Fn<SMALL_Y, ODD_Y> &>(fn) = PowF64Fn<SMALL_Y, ODD_Y>::make(y, lane_end_);
        fn.pre_mul = pre_op_ == PRE_MUL ? c : pre_op_ == PRE_RSUB ? -1.0 : 1.0;
        fn.pre_add = pre_op_ == PRE_MUL ? -0.0 : pre_op_ == PRE_SUB ? -c : c;
        return fn;
    }
};

template<typename Fn, typename = void> struct fn_pairwise : std::false_type {};
template<typename Fn> struct fn_pairwise<Fn, std::void_t<decltype(Fn::PAIRWISE)>> : std::bool_constant<Fn::PAIRWISE> {};
template<typename Fn, typename = void> struct fn_pow_tables : std::false_type {};
template<typename Fn> struct fn_pow_tables<Fn, std::void_t<decltype(Fn::POW_TABLES)>> : std::bool_constant<Fn::POW_TABLES> {};
// CHECKED functors offer `bool fast(a, r)`: a branch-free fast path that may decline.
template<typename Fn, typename = void> struct fn_checked : std::false_type {};
template<typename Fn> struct fn_checked<Fn, std::void_t<decltype(Fn::CHECKED)>> : std::bool_constant<Fn::CHECKED> {};

// Exact special forms of sm::pow(arr, y) for y in {2, 0.5, -1, 1}: one correctly
// rounded instruction instead of exp2(y*log2 x).  Chosen on the host
// (SMB_OPT_POW_SPECIALISE); the C99 special-case table still holds:
//   y = 2  : x*x            (pow(-0,2)=+0, pow(+-inf,2)=+inf, NaN -> NaN)
//   y = -1 : 1/x            (pow(+-0,-1)=+-inf, pow(+-inf,-1)=+-0)
//   y = 0.5: sqrt(x) except pow(-0,.5)=+0 and pow(-inf,.5)=+inf
//   y = 1  : x
enum { POWS_SQUARE = 0, POWS_RECIP = 1, POWS_SQRT = 2, POWS_IDENT = 3 };
template<int WHICH, typename T> struct PowSpecialFn {
    uint64_t lane_end;
    __device__ __forceinline__ T operator()(T a, T, uint64_t) const {
        if (WHICH == POWS_SQUARE) return DevOp<OP_MUL, T>::apply(a, a);
        if (WHICH == POWS_RECIP) return DevOp<OP_DIV, T>::apply((T)1, a);
        if (WHICH == POWS_SQRT) {
            if (a == (T)0) return (T)0;                 // +-0 -> +0
            if (a == -(T)INFINITY) return (T)INFINITY;  // -inf -> +inf
            if constexpr (sizeof(T) == 4) return __fsqrt_rn(a);
            else return __dsqrt_rn(a);
        }
        return a;
    }
};

// ---------------------------------------------------------------------------
// k_stream: out[i] = fn(a[i], b[i]) over dense streams.
//   VB     bytes per vector access (16 or 32)
//   UNROLL independent vectors in flight per thread per operand
//   HAS_B  false for array (op) scalar
// Work is cut into tiles of blockDim*UNROLL vectors; tile t is handled by block
// t mod gridDim (grid-stride), thread j of the block touching vectors
// j, j+blockDim, ... so every warp access is one fully coalesced 512 B / 1 KiB run.
// All loads of a tile are issued before the first use (memory-level parallelism).
// The ragged end (< one vector) is done by the last threads with scalar accesses.
// One vector of results from one vector (or two) of operands.
template<typename T, typename Fn, bool HAS_B, int VB>
__device__ __forceinline__ void stream_vec(const Pack<T, VB> &pa, const Pack<T, VB> &pb, Pack<T, VB> &r, uint64_t first_elem,
                                           const Fn &fn) {
    constexpr int EPV = VB / (int)sizeof(T);
    if constexpr (fn_pairwise<Fn>::value && (!HAS_B || fn_preop<Fn>::value) && (EPV % 2 == 0)) {
        // Pairwise functors (f32 pow): branch-free fast core on every pair, ONE check per vector;
        // a vector with any declined element is redone whole on the slow path (rare).  With a fused
        // pre-operator the pair is (a (op) b), exactly what the multi-tile loop feeds the core.
        Pack<T, VB> x;
#pragma unroll
        for (int k = 0; k < EPV; ++k) {
            if constexpr (fn_preop<Fn>::value) x.e[k] = fn.pre(pa.e[k], pb.e[k]);
            else x.e[k] = apply_pre1(fn, pa.e[k]);
        }
        bool ok = true;
#pragma unroll
        for (int k = 0; k < EPV; k += 2) ok &= fn.pair(x.e[k], x.e[k + 1], r.e[k], r.e[k + 1]);
        if (!ok) {
#pragma unroll
            for (int k = 0; k < EPV; ++k) r.e[k] = fn.slow_call(x.e[k]);
        }
    } else if constexpr (fn_checked<Fn>::value && (!HAS_B || fn_preop<Fn>::value)) {
        // (with a pre-operator too: the ragged tile must take the same fast / slow decision as the full tiles)
        bool ok = true;
#pragma unroll
        for (int k = 0; k < EPV; ++k) {
            T x;
            if constexpr (fn_preop<Fn>::value) x = fn.pre(pa.e[k], pb.e[k]);
            else x = apply_pre1(fn, pa.e[k]);
            ok &= fn.fast(x, r.e[k]);
        }
        if (!ok) {
#pragma unroll
            for (int k = 0; k < EPV; ++k) r.e[k] = fn(pa.e[k], HAS_B ? pb.e[k] : pa.e[k], 0);
        }
    } else {
#pragma unroll
        for (int k = 0; k < EPV; ++k) r.e[k] = fn(pa.e[k], HAS_B ? pb.e[k] : pa.e[k], first_elem + k);
    }
}

template<typename T, typename Fn, bool HAS_B, int VB, int UNROLL, bool GUARD>
__device__ __forceinline__ void stream_tile(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                            uint64_t v0, uint64_t nvec, uint64_t first, const Fn &fn) {
    constexpr int EPV = VB / (int)sizeof(T);
    Pack<T, VB> pa[UNROLL], pb[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint64_t v = v0 + (uint64_t)u * kBlock;
        if (!GUARD || v < nvec) {
            pa[u].raw = VecIO<VB, SMB_STREAM_LOAD_HINT>::load(reinterpret_cast<const RawVec<VB> *>(a) + v);
            if (HAS_B) pb[u].raw = VecIO<VB, SMB_STREAM_LOAD_HINT>::load(reinterpret_cast<const RawVec<VB> *>(b) + v);
        }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint64_t v = v0 + (uint64_t)u * kBlock;
        if (!GUARD || v < nvec) {
            Pack<T, VB> r;
            stream_vec<T, Fn, HAS_B, VB>(pa[u], pb[u], r, first + v * EPV, fn);
            VecIO<VB, SMB_STREAM_STORE_HINT>::store(reinterpret_cast<RawVec<VB> *>(out) + v, r.raw);
        }
    }
}

// One tile of a table-driven pow functor: the branch-free fast core on every vector, results
// stored under a predicate; the vectors it declined (specials, denormals, results near overflow --
// rare) are redone afterwards on the reference-accuracy path, ONE branch per tile.  Their input
// is re-read from memory rather than kept in registers; it has not been overwritten even when
// out aliases a, because the declined vector's store was skipped.
template<typename T, typename Fn, int VB, int UNROLL, bool PRE = false>
__device__ __forceinline__ void pow_tile(const Pack<T, VB> (&in)[UNROLL], [[maybe_unused]] const Pack<T, VB> (&in_b)[UNROLL],
                                         const T *__restrict__ a, [[maybe_unused]] const T *__restrict__ b, T *__restrict__ out,
                                         uint64_t v0, const Fn &fn) {
    constexpr int EPV = VB / (int)sizeof(T);
    bool ok[UNROLL], all = true;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        Pack<T, VB> r, x;
#pragma unroll
        for (int k = 0; k < EPV; ++k) {
            if constexpr (PRE) x.e[k] = fn.pre(in[u].e[k], in_b[u].e[k]);
            else x.e[k] = apply_pre1(fn, in[u].e[k]);
        }
        ok[u] = true;
        if constexpr (fn_pairwise<Fn>::value) {
#pragma unroll
            for (int k = 0; k < EPV; k += 2) ok[u] &= fn.pair(x.e[k], x.e[k + 1], r.e[k], r.e[k + 1]);
        } else {
#pragma unroll
            for (int k = 0; k < EPV; ++k) ok[u] &= fn.fast(x.e[k], r.e[k]);
        }
        if (ok[u]) VecIO<VB, true>::store(reinterpret_cast<RawVec<VB> *>(out) + v0 + (uint64_t)u * kBlock, r.raw);
        all &= ok[u];
        SMB_POW_SCHED_FENCE();
    }
    if (!all) {
        // ONE inlined copy of the reference-accuracy body in a rolled loop over the tile's elements:
        // a call here would make ptxas spill everything that lives across it (the prefetched tile).
        uint32_t bad = 0;
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) bad |= ok[u] ? 0u : 1u << u;
#pragma unroll 1
        for (int e = 0; e < UNROLL * EPV; ++e) {
            const int u = e / EPV;
            if ((bad >> u) & 1u) {
                const uint64_t i = (v0 + (uint64_t)u * kBlock) * EPV + (uint64_t)(e % EPV);
                if constexpr (PRE) out[i] = fn.slow(fn.pre(a[i], b[i]));
                else out[i] = fn.slow(apply_pre1(fn, a[i]));
            }
        }
    }
}

template<typename T, typename Fn, bool HAS_B, int VB, int UNROLL>
__global__ void __launch_bounds__(256, fn_pow_tables<Fn>::value ? (sizeof(T) == 4 ? SMB_POW_MIN_BLOCKS : SMB_POW64_MIN_BLOCKS) : 2) k_stream(const T *__restrict__ a, const T *__restrict__ b,
                                               T *__restrict__ out, uint64_t n, uint64_t first, Fn fn_in, uint32_t pdl) {
    constexpr int EPV = VB / (int)sizeof(T); // elements per vector
    Fn fn = fn_in;
    if (!(pdl & kPdlWaitFirst)) pdl_launch_dependents();
    if constexpr (fn_pow_tables<Fn>::value) fn.block_init(); // stage the lookup tables in shared memory (constant data: before the wait)
    if (pdl & kPdlWaitFirst) { pdl_wait(); pdl_launch_dependents(); } // dependents only after the wait, see pdl_enter
    const uint64_t nvec = n / EPV;
    constexpr uint64_t tile_vecs = (uint64_t)kBlock * UNROLL; // launches always use kBlock threads
    const uint64_t full_tiles = nvec / tile_vecs;
    // full tiles: no bounds checks in the loop body
    if constexpr (fn_pow_tables<Fn>::value && (!HAS_B || fn_preop<Fn>::value)) {
        constexpr bool PRE = fn_preop<Fn>::value;
        // Compute-heavy functor on a persistent grid: the next tile's loads are issued BEFORE this
        // tile's arithmetic (register double buffer), so HBM latency hides under ~500 issue slots of
        // math instead of stalling the warp (ncu: long_scoreboard was the top stall without it).
        // The two buffers swap roles every other tile (loop unrolled by two) -- copying one into
        // the other cost a MOV per element.
        Pack<T, VB> buf0[UNROLL], buf1[UNROLL];
        Pack<T, VB> bb0[PRE ? UNROLL : 1], bb1[PRE ? UNROLL : 1]; // the second operand's tiles (fused pre-operator only)
        const RawVec<VB> *av = reinterpret_cast<const RawVec<VB> *>(a);
        [[maybe_unused]] const RawVec<VB> *bv = reinterpret_cast<const RawVec<VB> *>(b);
        // one tile of loads into a buffer pair; the pow body needs operand b only with a pre-operator
#define SMB_POW_LOAD_TILE(BA, BB, TILE)                                                                     \
        _Pragma("unroll") for (int u = 0; u < UNROLL; ++u) {                                                \
            BA[u].raw = load_stream_pinned(av + (TILE) * tile_vecs + threadIdx.x + u * kBlock);             \
            if constexpr (PRE) BB[u].raw = load_stream_pinned(bv + (TILE) * tile_vecs + threadIdx.x + u * kBlock); \
        }
#define SMB_POW_RUN_TILE(BA, BB, TILE)                                                                      \
        do {                                                                                                \
            if constexpr (PRE) pow_tile<T, Fn, VB, UNROLL, true>(BA, BB, a, b, out, (TILE) * tile_vecs + threadIdx.x, fn); \
            else pow_tile<T, Fn, VB, UNROLL, false>(BA, BA, a, a, out, (TILE) * tile_vecs + threadIdx.x, fn); \
        } while (0)
        // CTA b owns `tpc` CONSECUTIVE tiles: the host sizes the grid so that tpc is a handful of tiles --
        // enough to amortise the table fill, few enough that the grid is many waves deep (a grid of
        // resident CTAs striding over everything measured 10-15 % slower on B200 for any 1-read-1-write
        // stream: profiles/r1_sweep_summary.md).
        const uint64_t tpc = (full_tiles + gridDim.x - 1) / gridDim.x;
        uint64_t tile = blockIdx.x * tpc;
        const uint64_t tiles_end = tile + tpc < full_tiles ? tile + tpc : full_tiles;
        if (tile < tiles_end) { SMB_POW_LOAD_TILE(buf0, bb0, tile) }
        fn.block_wait(); // the tables have landed (the copy overlapped the loads above)
#pragma unroll 1
        while (tile < tiles_end) {
            uint64_t next = tile + 1;
            if (next < tiles_end) { SMB_POW_LOAD_TILE(buf1, bb1, next) }
            SMB_POW_SCHED_FENCE();
            SMB_POW_RUN_TILE(buf0, bb0, tile);
            tile = next;
            if (tile >= tiles_end) break;
            next = tile + 1;
            if (next < tiles_end) { SMB_POW_LOAD_TILE(buf0, bb0, next) }
            SMB_POW_SCHED_FENCE();
            SMB_POW_RUN_TILE(buf1, bb1, tile);
            tile = next;
        }
#undef SMB_POW_LOAD_TILE
#undef SMB_POW_RUN_TILE
    } else {
#pragma unroll 1
        for (uint64_t tile = blockIdx.x; tile < full_tiles; tile += gridDim.x)
            stream_tile<T, Fn, HAS_B, VB, UNROLL, false>(a, b, out, tile * tile_vecs + threadIdx.x, nvec, first, fn);
    }
    // the ragged last tile goes to the block whose turn it would be
    if (full_tiles * tile_vecs < nvec && blockIdx.x == full_tiles % gridDim.x)
        stream_tile<T, Fn, HAS_B, VB, UNROLL, true>(a, b, out, full_tiles * tile_vecs + threadIdx.x, nvec, first, fn);
    // tail: n % EPV elements
    const uint64_t tail0 = nvec * EPV;
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gtid < n - tail0) {
        const uint64_t i = tail0 + gtid;
        out[i] = fn(a[i], HAS_B ? b[i] : a[i], first + i);
    }
    pdl_exit(pdl);
}

// Scalar-access variant for operands whose addresses do not share an alignment
// (views hand us interior pointers): element i by thread i, fully coalesced
// 4/8-byte accesses.
template<typename T, typename Fn, bool HAS_B>
__global__ void __launch_bounds__(256) k_stream_unaligned(const T *__restrict__ a, const T *__restrict__ b,
                                                         T *__restrict__ out, uint64_t n, uint64_t first, Fn fn) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = fn(a[i], HAS_B ? b[i] : a[i], first + i);
}

// ---------------------------------------------------------------------------
// Broadcast stride table.  Passed BY VALUE as a __grid_constant__ kernel
// parameter: kernel parameters live in the constant bank (c[0x0][...]), so every
// lane reads shape / stride / magic through the constant cache with uniform
// (broadcast) access -- the "stride table in constant memory" of the design --
// without a cudaMemcpyToSymbol round trip and without a global __constant__
// symbol that concurrent launches on different streams would race on.
struct BcastTable {
    int ndim;                        // coalesced rank >= 1
    uint32_t shape[SMB_MAX_NDIM];    // valid when !WIDE (all < 2^31)
    uint32_t mul[SMB_MAX_NDIM];      // fast-divmod magic per dim (divisor = shape[k])
    uint32_t shr[SMB_MAX_NDIM];
    uint64_t shape64[SMB_MAX_NDIM];
    uint64_t sa[SMB_MAX_NDIM];       // element strides, 0 on broadcast dims
    uint64_t sb[SMB_MAX_NDIM];
    uint64_t lin_base;               // first flat output index of this launch (sharding)
    uint64_t count;                  // elements this launch produces
    uint64_t lane_base;              // absolute flat index of lin_base (differs when a slab is staged)
};

__device__ __forceinline__ uint32_t fastdiv(uint32_t x, uint32_t d, uint32_t mul, uint32_t shr) {
    return d == 1 ? x : (__umulhi(x, mul) >> shr);
}

// flat index (relative to the full result) -> operand element offsets.
// Dims are peeled from the innermost outwards: idx_k = lin mod shape_k.
template<bool WIDE>
__device__ __forceinline__ void offsets_of(const BcastTable &t, uint64_t lin, uint64_t &oa, uint64_t &ob) {
    oa = 0;
    ob = 0;
    if (WIDE) {
        uint64_t rem = lin;
#pragma unroll
        for (int k = SMB_MAX_NDIM - 1; k >= 0; --k) {
            if (k < t.ndim) {
                uint64_t idx;
                if (k == 0) idx = rem;
                else { uint64_t q = rem / t.shape64[k]; idx = rem - q * t.shape64[k]; rem = q; }
                oa += idx * t.sa[k];
                ob += idx * t.sb[k];
            }
        }
    } else {
        uint32_t rem = (uint32_t)lin;
#pragma unroll
        for (int k = SMB_MAX_NDIM - 1; k >= 0; --k) {
            if (k < t.ndim) {
                uint32_t idx;
                if (k == 0) idx = rem;
                else { uint32_t q = fastdiv(rem, t.shape[k], t.mul[k], t.shr[k]); idx = rem - q * t.shape[k]; rem = q; }
                oa += (uint64_t)idx * t.sa[k];
                ob += (uint64_t)idx * t.sb[k];
            }
        }
    }
}

// k_row: inner strides in {0,1}.  Each thread produces UNROLL vectors of EPV consecutive
// outputs per iteration (host guarantees inner length, lin_base and the row bases are
// multiples of EPV and 16-byte aligned when EPV > 1); all operand loads of an iteration are
// issued before the first use.  An operand with inner stride 1 is read with one vector
// load; with inner stride 0 with one scalar load that is splat.  Operands with any zero
// stride are re-read by other threads, so they use the default (caching) load path; pure
// streams use the streaming hints.  (Staging the reused operand in shared memory measured
// slower on B200: DESIGN.md §4.2.)
template<typename T, typename Fn, int VB, bool WIDE, int UNROLL>
__global__ void __launch_bounds__(256) k_row(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                            const __grid_constant__ BcastTable t, int a_reused, int b_reused, Fn fn) {
    constexpr int EPV = VB / (int)sizeof(T);
    const uint64_t nvec = t.count / EPV; // host guarantees count % EPV == 0 when EPV > 1
    const int m = t.ndim;
    const bool ia = t.sa[m - 1] != 0, ib = t.sb[m - 1] != 0;
    constexpr uint64_t tile = (uint64_t)kBlock * UNROLL;
    for (uint64_t v0 = (uint64_t)blockIdx.x * tile + threadIdx.x; v0 < nvec; v0 += (uint64_t)gridDim.x * tile) {
        Pack<T, VB> pa[UNROLL], pb[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint64_t v = v0 + (uint64_t)u * kBlock;
            if (v < nvec) {
                uint64_t oa, ob;
                offsets_of<WIDE>(t, t.lin_base + v * EPV, oa, ob);
                if constexpr (EPV == 1) {
                    pa[u].e[0] = a[oa];
                    pb[u].e[0] = b[ob];
                } else {
                    if (ia) {
                        pa[u].raw = a_reused ? VecIO<VB, false>::load(a + oa) : VecIO<VB, true>::load(a + oa);
                    } else {
                        const T s = a[oa];
#pragma unroll
                        for (int k = 0; k < EPV; ++k) pa[u].e[k] = s;
                    }
                    if (ib) {
                        pb[u].raw = b_reused ? VecIO<VB, false>::load(b + ob) : VecIO<VB, true>::load(b + ob);
                    } else {
                        const T s = b[ob];
#pragma unroll
                        for (int k = 0; k < EPV; ++k) pb[u].e[k] = s;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint64_t v = v0 + (uint64_t)u * kBlock;
            if (v < nvec) {
                Pack<T, VB> r;
#pragma unroll
                for (int k = 0; k < EPV; ++k) r.e[k] = fn(pa[u].e[k], pb[u].e[k], t.lane_base + v * EPV + k);
                if constexpr (EPV == 1) out[v] = r.e[0];
                else VecIO<VB, true>::store(reinterpret_cast<RawVec<VB> *>(out) + v, r.raw);
            }
        }
    }
}

// k_outer: the "two operands, each broadcast along a different outer dim" pattern
// (BASELINE config C4: {D0,1,L} (op) {1,D1,L} -> {D0,D1,L}): out[i][j][k] = x[i][k] (op) y[j][k].
// The output is D1 (resp. D0) times larger than either operand, so the kernel is a store
// stream fed from L2; what can be saved is L2 -> SM read traffic.  Each thread keeps TI
// vectors of the dim-0 operand and TJ vectors of the dim-1 operand in registers and
// produces the TI x TJ block of output vectors from them: (TI+TJ) loads per TI*TJ stores
// instead of 2 per store (k_row).  A_ON_DIM0 says which reference operand varies with
// dim 0, so non-commutative ops keep their operand order.
// int32 a / b with the divisor's reciprocal precomputed in double and nudged up by 2^-50:
//   r = (1 / b) * (1 + 2^-50);  q = trunc(double(a) * r)
// Exact for every pair the reference defines (b != 0, not INT_MIN / -1): a true quotient that is
// not an integer is at least 1/|b| away from one, and the error of a*r is below 2^-18/|b|; a true
// quotient k that IS an integer comes out as k (1 + 2^-50 +- 2^-51.4) (r within an ulp of 1/b,
// one more half-ulp for the product), strictly beyond k by
// less than 2^-18, so truncation returns k.  Truncation itself avoids the (slow) F2I.F64:
// trunc(v) = rint(v - 0.5 sign(v)) for such v, fused into the product, and rint is the low word of
// (w + 1.5 * 2^52).  Per quotient: one LOP3 (the signed half), one DFMA, one DADD -- instead of
// the ~25-instruction software s32 division; worth it when a divisor is reused (k_outer).
__device__ __forceinline__ double idiv_recip(int32_t b) {
    // 1/b to within an ulp: MUFU.RCP64H seed (20 bits) and two Newton steps; b is a non-zero
    // integer, so none of __drcp_rn's special-case handling (and its branches) is needed.
    const double d = (double)b;
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = __fma_rn(r, __fma_rn(-d, r, 1.0), r);
    r = __fma_rn(r, __fma_rn(-d, r, 1.0), r);
    return __dmul_rn(r, 1.0 + 0x1p-50);
}
// high word of -0.5 * sign(r): XOR-ed with the dividend's sign bit it becomes -0.5 * sign(a / b)
__device__ __forceinline__ uint32_t idiv_half_hi(double r) { return ((uint32_t)__double2hiint(r) & 0x80000000u) ^ 0xbfe00000u; }
__device__ __forceinline__ int32_t idiv_by_recip(int32_t a, double a_as_double, double r, uint32_t half_hi) {
    const double half = __hiloint2double((int)(((uint32_t)a & 0x80000000u) ^ half_hi), 0);
    const double w = __fma_rn(a_as_double, r, half);
    return __double2loint(__dadd_rn(w, 6755399441055744.0));
}
template<typename T, typename Fn> struct is_int_div : std::false_type {};
template<> struct is_int_div<int32_t, BinaryFn<OP_DIV, int32_t>> : std::true_type {};

struct OuterParams {
    uint32_t d0, d1, len;   // (sub-)problem shape: d0 x d1 rows of `len` elements
    uint64_t s0, s1;        // element stride of the dim-0 / dim-1 operand between its rows
    uint64_t lane_base;     // absolute flat index of out[0] (int pow lane/scalar split)
};
template<typename T, typename Fn, int TI, int TJ, bool A_ON_DIM0>
__global__ void __launch_bounds__(256) k_outer(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                              const __grid_constant__ OuterParams p, Fn fn) {
    constexpr int EPV = 16 / (int)sizeof(T);
    const uint32_t k = (blockIdx.x * kBlock + threadIdx.x) * EPV;
    if (k >= p.len) return;
    const uint32_t j0 = blockIdx.y * TJ, i0 = blockIdx.z * TI;
    const T *x = A_ON_DIM0 ? a : b; // varies with dim 0
    const T *y = A_ON_DIM0 ? b : a; // varies with dim 1
    Pack<T, 16> xv[TI], yv[TJ];
#pragma unroll
    for (int ti = 0; ti < TI; ++ti)
        if (i0 + ti < p.d0) xv[ti].raw = VecIO<16, false>::load(x + (uint64_t)(i0 + ti) * p.s0 + k);
#pragma unroll
    for (int tj = 0; tj < TJ; ++tj)
        if (j0 + tj < p.d1) yv[tj].raw = VecIO<16, false>::load(y + (uint64_t)(j0 + tj) * p.s1 + k);
    if constexpr (is_int_div<T, Fn>::value) {
        // every divisor is used TI (TJ) times: one reciprocal each, then a multiply per quotient
        constexpr int ND = A_ON_DIM0 ? TJ : TI;
        double rc[ND][EPV];
        uint32_t hh[ND][EPV];
#pragma unroll
        for (int t = 0; t < ND; ++t) {
            if ((A_ON_DIM0 ? j0 : i0) + t < (A_ON_DIM0 ? p.d1 : p.d0)) {
#pragma unroll
                for (int e = 0; e < EPV; ++e) {
                    rc[t][e] = idiv_recip(A_ON_DIM0 ? yv[t].e[e] : xv[t].e[e]);
                    hh[t][e] = idiv_half_hi(rc[t][e]);
                }
            }
        }
        // outer loop over the dividend's vectors: each dividend is converted to double once too
        constexpr int NN = A_ON_DIM0 ? TI : TJ;
#pragma unroll
        for (int tn = 0; tn < NN; ++tn) {
            if ((A_ON_DIM0 ? i0 : j0) + tn >= (A_ON_DIM0 ? p.d0 : p.d1)) break;
            double num[EPV];
#pragma unroll
            for (int e = 0; e < EPV; ++e) num[e] = (double)(A_ON_DIM0 ? xv[tn].e[e] : yv[tn].e[e]);
#pragma unroll
            for (int td = 0; td < ND; ++td) {
                if ((A_ON_DIM0 ? j0 : i0) + td >= (A_ON_DIM0 ? p.d1 : p.d0)) break;
                const uint32_t i = i0 + (A_ON_DIM0 ? tn : td), j = j0 + (A_ON_DIM0 ? td : tn);
                const uint64_t lin = ((uint64_t)i * p.d1 + j) * p.len + k;
                Pack<T, 16> r;
#pragma unroll
                for (int e = 0; e < EPV; ++e)
                    r.e[e] = idiv_by_recip(A_ON_DIM0 ? xv[tn].e[e] : yv[tn].e[e], num[e], rc[td][e], hh[td][e]);
                VecIO<16, true>::store(out + lin, r.raw);
            }
        }
    } else {
#pragma unroll
        for (int ti = 0; ti < TI; ++ti) {
            if (i0 + ti >= p.d0) break;
#pragma unroll
            for (int tj = 0; tj < TJ; ++tj) {
                if (j0 + tj >= p.d1) break;
                const uint64_t lin = ((uint64_t)(i0 + ti) * p.d1 + (j0 + tj)) * p.len + k;
                Pack<T, 16> r;
#pragma unroll
                for (int e = 0; e < EPV; ++e)
                    r.e[e] = A_ON_DIM0 ? fn(xv[ti].e[e], yv[tj].e[e], p.lane_base + lin + e)
                                       : fn(yv[tj].e[e], xv[ti].e[e], p.lane_base + lin + e);
                VecIO<16, true>::store(out + lin, r.raw);
            }
        }
    }
}

// k_tile: a TRANSPOSED operand (what SMArray::transpose() hands to element_wise_op: stride 1
// along some earlier result dim, a large stride along the last).  Read directly, every
// warp would touch 32 different rows for 128 useful bytes; instead each CTA moves a 32x32 tile
// of that operand through shared memory -- global reads coalesced along the operand's own
// contiguous direction, the transpose done on chip -- and writes the result rows coalesced.
// The other operand is read directly (inner stride 0 or 1) or through a second tile when it
// is transposed too.  Leading dims are batches: their offsets come from the stride table by
// fast-divmod, once per CTA.
struct TileParams {
    uint32_t rows, cols;            // tile dims: rows = the dim the transposed operand is contiguous in, cols = last dim
    uint64_t a_r, a_c, b_r, b_c;    // element strides of each operand along rows / cols
    uint64_t o_r;                   // result stride along rows (cols are contiguous in the result)
    uint32_t nbatch_dims;           // every other dim, enumerated by blockIdx.z
    uint32_t bshape[SMB_MAX_NDIM], bmul[SMB_MAX_NDIM], bshr[SMB_MAX_NDIM];
    uint64_t ba[SMB_MAX_NDIM], bb[SMB_MAX_NDIM], bo[SMB_MAX_NDIM];
    uint64_t lane_base;
};
template<typename T, typename Fn, bool A_T, bool B_T, int TR, int TC, bool FULL>
__device__ __forceinline__ void tile_body(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                          const TileParams &p, const Fn &fn, uint32_t r0, uint32_t c0, uint64_t obase,
                                          T (*ta)[TR + 1], T (*tb)[TR + 1]) {
    static_assert(kBlock % TR == 0 && kBlock % TC == 0, "tile dims must divide the CTA size");
    constexpr int PER = TR * TC / kBlock;  // elements per thread
    constexpr int SSTEP = kBlock / TR;     // stage pass: thread -> (row tid % TR, col tid / TR + j * SSTEP)
    constexpr int PSTEP = kBlock / TC;     // produce pass: thread -> (col tid % TC, row tid / TC + j * PSTEP)
    const uint32_t slr = threadIdx.x % TR, slc = threadIdx.x / TR;
    const uint32_t plc = threadIdx.x % TC, plr = threadIdx.x / TC;
    // every global load of the tile is issued before the first use: the transposed operand along
    // its own contiguous direction (stage coordinates), a direct operand at the result's coordinates
    const T *as = a + (uint64_t)(r0 + slr) * p.a_r + (uint64_t)(c0 + slc) * p.a_c;
    const T *ap = a + (uint64_t)(r0 + plr) * p.a_r + (uint64_t)(c0 + plc) * p.a_c;
    const T *bs = b + (uint64_t)(r0 + slr) * p.b_r + (uint64_t)(c0 + slc) * p.b_c;
    const T *bp = b + (uint64_t)(r0 + plr) * p.b_r + (uint64_t)(c0 + plc) * p.b_c;
    const uint64_t a_step = A_T ? (uint64_t)SSTEP * p.a_c : (uint64_t)PSTEP * p.a_r;
    const uint64_t b_step = B_T ? (uint64_t)SSTEP * p.b_c : (uint64_t)PSTEP * p.b_r;
    const bool s_row_ok = FULL || r0 + slr < p.rows, p_col_ok = FULL || c0 + plc < p.cols;
    T va[PER], vb[PER];
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const bool s_ok = FULL || (s_row_ok && c0 + slc + j * SSTEP < p.cols);
        const bool p_ok = FULL || (p_col_ok && r0 + plr + j * PSTEP < p.rows);
        if (A_T ? s_ok : p_ok) va[j] = __ldg((A_T ? as : ap) + (uint64_t)j * a_step);
        if (B_T ? s_ok : p_ok) vb[j] = __ldg((B_T ? bs : bp) + (uint64_t)j * b_step);
    }
    if (A_T || B_T) {
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            if (A_T) ta[slc + j * SSTEP][slr] = va[j];
            if (B_T) tb[slc + j * SSTEP][slr] = vb[j];
        }
        __syncthreads();
    }
    T *o = out + obase + (uint64_t)(r0 + plr) * p.o_r + (c0 + plc);
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        if (FULL || (p_col_ok && r0 + plr + j * PSTEP < p.rows)) {
            const T x = A_T ? ta[plc][plr + j * PSTEP] : va[j];
            const T y = B_T ? tb[plc][plr + j * PSTEP] : vb[j];
            const uint64_t off = (uint64_t)j * PSTEP * p.o_r;
            o[off] = fn(x, y, p.lane_base + (uint64_t)(o + off - out));
        }
    }
}

template<typename T, typename Fn, bool A_T, bool B_T, int TR, int TC>
__global__ void __launch_bounds__(256) k_tile(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                             const __grid_constant__ TileParams p, Fn fn) {
    // tile: TR rows (the transposed operand's contiguous direction) x TC cols (the result's);
    // the +1 pad makes both the row-wise fill and the column-wise drain conflict-free
    __shared__ T ta[A_T ? TC : 1][TR + 1], tb[B_T ? TC : 1][TR + 1];
    const uint32_t c0 = blockIdx.x * TC, r0 = blockIdx.y * TR;
    uint64_t oa = 0, ob = 0, obase = 0;
    uint32_t rem = blockIdx.z;
#pragma unroll
    for (int k = SMB_MAX_NDIM - 1; k >= 0; --k) {
        if (k < (int)p.nbatch_dims) {
            const uint32_t q = k == 0 ? 0u : fastdiv(rem, p.bshape[k], p.bmul[k], p.bshr[k]);
            const uint32_t idx = k == 0 ? rem : rem - q * p.bshape[k];
            rem = q;
            oa += (uint64_t)idx * p.ba[k];
            ob += (uint64_t)idx * p.bb[k];
            obase += (uint64_t)idx * p.bo[k];
        }
    }
    if (r0 + TR <= p.rows && c0 + TC <= p.cols)
        tile_body<T, Fn, A_T, B_T, TR, TC, true>(a + oa, b + ob, out, p, fn, r0, c0, obase, ta, tb);
    else
        tile_body<T, Fn, A_T, B_T, TR, TC, false>(a + oa, b + ob, out, p, fn, r0, c0, obase, ta, tb);
}

// ---------------------------------------------------------------------------
// k_chain: a left-deep chain of Op structs in one pass (smb_chain),
//     acc = leaf_0;  acc = acc (op_i) leaf_i   [leaf_i (op_i) acc when swap_i]
// Every leaf is an array broadcast against the result (stride table, 0 on broadcast dims) or a
// constant.  EPV elements per thread along the inner dim: an inner-stride-1 leaf is one vector
// load, an inner-stride-0 leaf one scalar load splat (EPV == 1: any strides).  All leaves are
// loaded before the first operator is applied (the loops over steps are fully unrolled with
// uniform guards, so the leaf values sit in registers); each intermediate is rounded to T by the
// same DevOp bodies the single operators use, so the result is bit-identical to the unfused
// sequence.  HBM-bound: (array leaves + 1) * sizeof(T) bytes per element instead of
// 3 * sizeof(T) per operator.
struct ChainTable {
    int ndim, nsteps;
    uint32_t shape[SMB_MAX_NDIM], mul[SMB_MAX_NDIM], shr[SMB_MAX_NDIM];
    uint64_t shape64[SMB_MAX_NDIM];
    uint64_t stride[kChainMax][SMB_MAX_NDIM];
    const void *data[kChainMax];   // nullptr: constant leaf
    uint64_t cbits[kChainMax];     // the constant, as T, in the low bytes
    uint8_t op[kChainMax];         // CH_* step codes (the mirrored forms fold the swap flag in)
    uint64_t lin_base, count;      // flat output range of this launch
    uint64_t lane_end;             // int32 pow: flat indices below it use AVX2-lane semantics
    uint32_t tiles_per_cta;        // consecutive tiles per CTA (1; a few when the pow tables are staged)
    // f32 pow steps the table-driven core may take (POWFAST kernels): per step the two sign masks of
    // pow_f32_pair_fast<.., POW_SIGN_RUNTIME, ..>; pow_fast[s] == 0 keeps the reference-accuracy path
    uint8_t pow_fast[kChainMax];
    uint32_t pow_small;            // 1: the invc table image and the r-series core (every fast step has |y| <= 256)
    uint32_t pow_abs_mask[kChainMax], pow_sign_or[kChainMax];
    PowConsts pow_consts;
};
template<typename T> __device__ __forceinline__ T chain_const(uint64_t bits) {
    if constexpr (sizeof(T) == 8) return __longlong_as_double((long long)bits);
    else if constexpr (std::is_same<T, float>::value) return __uint_as_float((uint32_t)bits);
    else return (T)(uint32_t)bits;
}
// pow inside a chain is the reference-accuracy path, out of line: inlined at every step it would
// multiply the kernel's code size by the chain length for a case most chains do not contain.
template<typename T> __device__ __noinline__ T chain_pow(T a, T b, bool lane) {
    if constexpr (std::is_same<T, int32_t>::value) return lane ? powi_lane(a, b) : powi_scalar(a, b);
    else return DevOp<OP_POW, T>::apply(a, b);
}
// step codes: the four ops, the two non-commutative ones mirrored (leaf on the left), pow
enum { CH_ADD = 0, CH_SUB = 1, CH_MUL = 2, CH_DIV = 3, CH_POW = 4, CH_RSUB = 5, CH_RDIV = 6, CH_SQR = 7, CH_SQRT = 8 };
// pow(x, 0.5) exactly as the specialised sm::pow kernel computes it (PowSpecialFn<POWS_SQRT>); never reached for int32
// (out of line, like chain_pow: inlined, the correctly rounded square root's fix-up path cost the plain arithmetic chains three
// registers and 10 % -- 7.27 -> 6.50 TB/s on (a+b)*c)
template<typename T> __device__ __noinline__ T chain_sqrt(T a) {
    if constexpr (std::is_floating_point<T>::value) {
        if (a == (T)0) return (T)0;                 // +-0 -> +0
        if (a == -(T)INFINITY) return (T)INFINITY;  // -inf -> +inf
        if constexpr (sizeof(T) == 4) return __fsqrt_rn(a);
        else return __dsqrt_rn(a);
    } else {
        return a;
    }
}
// NS: compiled-in capacity of the chain (leaf registers); UNROLL: vectors per thread, all of whose
// leaf loads are issued before the first operator (UNROLL * NS independent loads in flight per
// thread -- a single vector per thread left HBM half idle).  One tile of 256 * UNROLL vectors per CTA.
// One tile (256 * UNROLL vectors) of leaf loads.  NDIM: the coalesced rank when it is 1 or 2 (the
// index and offset loops are then straight-line code on constant-bank operands -- with the rank a
// run-time value the guarded 6-dim loops were 58 instructions per element, most of them IMAD / MOV /
// ISETP / BRA), 0: any rank, guarded loops.
template<typename T, int EPV, bool WIDE, int NS, int UNROLL, int NDIM>
__device__ __forceinline__ void chain_load(const ChainTable &t, uint64_t tile, uint64_t nvec, T (&leaf)[UNROLL][NS][EPV]) {
    using Idx = typename std::conditional<WIDE, uint64_t, uint32_t>::type;
    constexpr int KMAX = NDIM ? NDIM : SMB_MAX_NDIM;
    const int ndim = NDIM ? NDIM : t.ndim;
    const uint64_t v0 = tile * (kBlock * UNROLL) + threadIdx.x;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint64_t v = v0 + (uint64_t)u * kBlock;
        if (v >= nvec) continue; // (its registers stay undefined; nothing of it is stored)
        const uint64_t lin = t.lin_base + v * EPV;
        // flat index -> per-dim indices, innermost first
        Idx idx[KMAX];
        Idx rem = (Idx)lin;
#pragma unroll
        for (int k = KMAX - 1; k >= 0; --k) {
            if (k < ndim) {
                if (k == 0) idx[k] = rem;
                else if (WIDE) { const uint64_t q = rem / t.shape64[k]; idx[k] = (Idx)(rem - q * t.shape64[k]); rem = (Idx)q; }
                else { const uint32_t q = fastdiv((uint32_t)rem, t.shape[k], t.mul[k], t.shr[k]); idx[k] = (Idx)((uint32_t)rem - q * t.shape[k]); rem = (Idx)q; }
            }
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            if (s < t.nsteps) {
                const T *base = static_cast<const T *>(t.data[s]);
                if (base == nullptr) {
#pragma unroll
                    for (int e = 0; e < EPV; ++e) leaf[u][s][e] = chain_const<T>(t.cbits[s]);
                } else {
                    uint64_t off = 0;
#pragma unroll
                    for (int k = 0; k < KMAX; ++k)
                        if (k < ndim) off += (uint64_t)idx[k] * t.stride[s][k];
                    if (EPV > 1 && t.stride[s][ndim - 1] == 1) {
                        Pack<T, 16> pk; // EPV * sizeof(T) == 16
                        pk.raw = VecIO<16, false>::load(base + off);
#pragma unroll
                        for (int e = 0; e < EPV; ++e) leaf[u][s][e] = pk.e[e];
                    } else {
                        const T x = __ldg(base + off);
#pragma unroll
                        for (int e = 0; e < EPV; ++e) leaf[u][s][e] = x;
                    }
                }
            }
        }
    }
}

// The operators of one tile and its stores: ONE uniform switch per step, straight-line code over
// every element the thread holds inside each case (a switch per element made the kernel
// branch-bound).
template<typename T, int EPV, int NS, int UNROLL, bool POWFAST>
__device__ __forceinline__ void chain_compute(const ChainTable &t, uint64_t tile, uint64_t nvec, const T (&leaf)[UNROLL][NS][EPV],
                                              T *__restrict__ out, [[maybe_unused]] const PowLane &lane) {
    const uint64_t v0 = tile * (kBlock * UNROLL) + threadIdx.x;
    T acc[UNROLL][EPV];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
#pragma unroll
        for (int e = 0; e < EPV; ++e) acc[u][e] = leaf[u][0][e];
#define SMB_CHAIN_CASE(CODE, EXPR)                                                       \
    case CODE:                                                                           \
        _Pragma("unroll") for (int u = 0; u < UNROLL; ++u)                               \
            _Pragma("unroll") for (int e = 0; e < EPV; ++e) {                            \
                const T x = acc[u][e], y = leaf[u][s][e];                                \
                acc[u][e] = EXPR;                                                        \
            }                                                                            \
        break;
#pragma unroll
    for (int s = 1; s < NS; ++s) {
        if (s < t.nsteps) {
            switch (t.op[s]) {
                SMB_CHAIN_CASE(CH_ADD, (DevOp<OP_ADD, T>::apply(x, y)))
                SMB_CHAIN_CASE(CH_SUB, (DevOp<OP_SUB, T>::apply(x, y)))
                SMB_CHAIN_CASE(CH_MUL, (DevOp<OP_MUL, T>::apply(x, y)))
                SMB_CHAIN_CASE(CH_DIV, (DevOp<OP_DIV, T>::apply(x, y)))
                SMB_CHAIN_CASE(CH_RSUB, (DevOp<OP_SUB, T>::apply(y, x)))
                SMB_CHAIN_CASE(CH_RDIV, (DevOp<OP_DIV, T>::apply(y, x)))
                default: // CH_POW and its two exact forms (rare: kept out of the compare chain of the arithmetic cases)
                    if (t.op[s] == CH_SQR || t.op[s] == CH_SQRT) {
                        const bool sq = t.op[s] == CH_SQR;
#pragma unroll
                        for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                            for (int e = 0; e < EPV; ++e) acc[u][e] = sq ? DevOp<OP_MUL, T>::apply(acc[u][e], acc[u][e]) : chain_sqrt<T>(acc[u][e]);
                        break;
                    }
#pragma unroll
                    for (int u = 0; u < UNROLL; ++u) {
                        const uint64_t lin = t.lin_base + (v0 + (uint64_t)u * kBlock) * EPV;
                        bool done = false;
                        if constexpr (POWFAST) {
                            if (t.pow_fast[s]) {
                                float r[EPV];
                                bool ok = true;
                                if (t.pow_small) { // every fast pow step of this chain has |y| <= 256: the r-series core
#pragma unroll
                                    for (int e = 0; e < EPV; e += 2)
                                        ok &= pow_f32_pair_fast<POW_TIER_MEDIUM, POW_SIGN_RUNTIME, false>(
                                            acc[u][e], acc[u][e + 1], leaf[u][s][0], lane, nullptr, nullptr, &r[e], &r[e + 1],
                                            t.pow_abs_mask[s], t.pow_sign_or[s]);
                                } else {
#pragma unroll
                                    for (int e = 0; e < EPV; e += 2)
                                        ok &= pow_f32_pair_fast<POW_TIER_LARGE, POW_SIGN_RUNTIME, false>(
                                            acc[u][e], acc[u][e + 1], leaf[u][s][0], lane, nullptr, nullptr, &r[e], &r[e + 1],
                                            t.pow_abs_mask[s], t.pow_sign_or[s]);
                                }
                                if (ok) {
#pragma unroll
                                    for (int e = 0; e < EPV; ++e) acc[u][e] = r[e];
                                    done = true;
                                }
                            }
                        }
                        if (!done) {
#pragma unroll
                            for (int e = 0; e < EPV; ++e) acc[u][e] = chain_pow<T>(acc[u][e], leaf[u][s][e], lin + e < t.lane_end);
                        }
                    }
                    break;
            }
        }
    }
#undef SMB_CHAIN_CASE
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint64_t v = v0 + (uint64_t)u * kBlock;
        if (v < nvec) {
            if (EPV > 1) {
                Pack<T, 16> r;
#pragma unroll
                for (int e = 0; e < EPV; ++e) r.e[e] = acc[u][e];
                VecIO<16, true>::store(out + v * EPV, r.raw);
            } else {
                out[v] = acc[u][0];
            }
        }
    }
}

// POWFAST (float, EPV == 4): the pow tables are staged per CTA (one bulk copy, overlapped with the
// first tile's loads) and a pow step goes through the FFMA2 core, two elements per call, the
// reference-accuracy path only for the vectors it declines -- sm::pow(a + b, e) in one pass.  Such a
// CTA runs several consecutive tiles to amortise the copy; plain chains run one tile per CTA.
template<typename T, int EPV, bool WIDE, int NS, int UNROLL, bool POWFAST, int NDIM>
__global__ void __launch_bounds__(256) k_chain(T *__restrict__ out, const __grid_constant__ ChainTable t) {
    const uint64_t nvec = t.count / EPV; // host guarantees count % EPV == 0
    const uint64_t ntiles = (nvec + kBlock * UNROLL - 1) / (kBlock * UNROLL);
    if constexpr (!POWFAST) {
        const uint64_t tile = blockIdx.x;
        if (tile >= ntiles) return;
        T leaf[UNROLL][NS][EPV];
        chain_load<T, EPV, WIDE, NS, UNROLL, NDIM>(t, tile, nvec, leaf);
        chain_compute<T, EPV, NS, UNROLL, false>(t, tile, nvec, leaf, out, PowLane{});
    } else {
        __shared__ __align__(8) uint64_t tab_bar;
        if (threadIdx.x == 0) {
            mbar_init(&tab_bar, 1);
            mbar_expect_tx(&tab_bar, (uint32_t)sizeof(SmbPowTabs));
            bulk_g2s(&smb_s_pow, &g_pow_image[t.pow_small ? 0 : 1], (uint32_t)sizeof(SmbPowTabs), &tab_bar);
        }
        PowLane lane = pow_lane(threadIdx.x, t.pow_consts);
        __syncthreads(); // the barrier is initialised before anyone waits on it
        uint64_t tile = (uint64_t)blockIdx.x * t.tiles_per_cta;
        const uint64_t tile_end = tile + t.tiles_per_cta < ntiles ? tile + t.tiles_per_cta : ntiles;
        if (tile >= tile_end) { // (the host never launches such a CTA) still let the bulk copy into our shared memory land
            mbar_wait(&tab_bar, 0);
            return;
        }
        // Occupancy (one vector per thread, four CTAs) hides the leaf loads; a register prefetch of the next tile
        // measured slower (profiles/r2_chain_pow_sweep.jsonl).
        bool first = true;
#pragma unroll 1
        for (; tile < tile_end; ++tile) {
            T leaf[UNROLL][NS][EPV];
            chain_load<T, EPV, WIDE, NS, UNROLL, NDIM>(t, tile, nvec, leaf);
            if (first) {
                mbar_wait(&tab_bar, 0); // the tables have landed (the copy overlapped the loads above)
                asm volatile("" : "+r"(lane.log_off), "+r"(lane.exp_off) :: "memory"); // ties the lookups to the wait
                first = false;
            }
            chain_compute<T, EPV, NS, UNROLL, true>(t, tile, nvec, leaf, out, lane);
        }
    }
}

// k_generic: arbitrary element strides; one output element per thread per
// iteration, coalesced stores, gathered loads.
template<typename T, typename Fn, bool WIDE>
__global__ void __launch_bounds__(256) k_generic(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                                const __grid_constant__ BcastTable t, Fn fn) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < t.count; i += stride) {
        const uint64_t lin = t.lin_base + i;
        uint64_t oa, ob;
        offsets_of<WIDE>(t, lin, oa, ob);
        out[i] = fn(a[oa], b[ob], t.lane_base + i);
    }
}

// ---------------------------------------------------------------------------
// k_sgather: small constant inner strides (w[:, ::2] + w[:, 1::2], every third column, ...).  k_generic reads
// such operands one 4-byte element per thread: the warp still pulls every sector of the rows it touches, but
// pays one load instruction, one index computation and one scalar store per ELEMENT.  Here a thread produces
// one 16-byte vector of consecutive outputs; an operand with inner stride S <= EPV is covered by at most
// S + 1 ALIGNED 16-byte loads (the span from its first to its last wanted element, aligned down by the
// operand's phase), and the wanted elements are picked in registers -- lane positions are compile-time
// constants, selected by ONE uniform switch on (stride, phase) per operand.  Every loaded vector contains
// at least one wanted element (S <= EPV), so nothing outside the operand's pages is touched.  Host
// guarantees: row length, range bounds and every outer stride are multiples of EPV (the phase is then the
// same for every vector), inner strides <= EPV, 16-byte aligned result.
// V32: the span is an even number of vectors starting on a 32-byte boundary (host-checked, uniform): one 256-bit load per
// vector PAIR (LDG.E.256, new with sm_100).  A warp's lanes sit S vectors apart, so 128-bit loads fill only every S-th
// 16 bytes of each L1 wavefront -- ncu had the LSU data pipe at 98 % on w[:, ::2] + w[:, 1::2] with DRAM at 65 %.
template<typename T, int S, int PH, bool V32>
__device__ __forceinline__ void sg_pick(const T *__restrict__ p_aligned, T (&v)[16 / sizeof(T)]) {
    constexpr int EPV = 16 / (int)sizeof(T);
    if constexpr (S == 0) {
        const T x = __ldg(p_aligned + PH);
#pragma unroll
        for (int e = 0; e < EPV; ++e) v[e] = x;
    } else {
        constexpr int NV = (PH + (EPV - 1) * S) / EPV + 1;
        if constexpr (V32 && NV % 2 == 0) {
            Pack<T, 32> pk[NV / 2];
#pragma unroll
            for (int k = 0; k < NV / 2; ++k) pk[k].raw = VecIO<32, false>::load(p_aligned + k * 2 * EPV);
#pragma unroll
            for (int e = 0; e < EPV; ++e) v[e] = pk[(PH + e * S) / (2 * EPV)].e[(PH + e * S) % (2 * EPV)];
        } else {
            Pack<T, 16> pk[NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) pk[k].raw = VecIO<16, false>::load(p_aligned + k * EPV);
#pragma unroll
            for (int e = 0; e < EPV; ++e) v[e] = pk[(PH + e * S) / EPV].e[(PH + e * S) % EPV];
        }
    }
}
template<typename T, int S, bool V32>
__device__ __forceinline__ void sg_load_phase(const T *__restrict__ p, int phase, T (&v)[16 / sizeof(T)]) {
    constexpr int EPV = 16 / (int)sizeof(T);
    const T *pa = p - phase;
    if constexpr (EPV == 4) {
        switch (phase) {
            case 0: sg_pick<T, S, 0, V32>(pa, v); break;
            case 1: sg_pick<T, S, 1, V32>(pa, v); break;
            case 2: sg_pick<T, S, 2, V32>(pa, v); break;
            default: sg_pick<T, S, 3, V32>(pa, v); break;
        }
    } else {
        if (phase == 0) sg_pick<T, S, 0, V32>(pa, v);
        else sg_pick<T, S, 1, V32>(pa, v);
    }
}
// wide32: the host found every vector span of this operand 32-byte aligned (even stride, base and outer strides on
// 32 bytes); only the strides whose spans can be an even number of vectors have a 256-bit form
template<typename T>
__device__ __forceinline__ void sg_load(const T *__restrict__ p, int stride, int phase, bool wide32, T (&v)[16 / sizeof(T)]) {
    constexpr int EPV = 16 / (int)sizeof(T);
    switch (stride) { // uniform
        case 0: sg_load_phase<T, 0, false>(p, phase, v); break;
        case 1: sg_load_phase<T, 1, false>(p, phase, v); break;
        case 2:
            if (wide32) sg_load_phase<T, 2, true>(p, phase, v);
            else sg_load_phase<T, 2, false>(p, phase, v);
            break;
        default:
            if constexpr (EPV == 4) {
                if (stride == 3) sg_load_phase<T, 3, false>(p, phase, v);
                else if (wide32) sg_load_phase<T, 4, true>(p, phase, v);
                else sg_load_phase<T, 4, false>(p, phase, v);
            } else {
                sg_load_phase<T, 2, false>(p, phase, v); // (not reached: the host admits strides <= EPV)
            }
            break;
    }
}
template<typename T, typename Fn, bool WIDE>
__global__ void __launch_bounds__(256) k_sgather(const T *__restrict__ a, const T *__restrict__ b, T *__restrict__ out,
                                                const __grid_constant__ BcastTable t, int phase_a, int phase_b, int wide32, Fn fn) {
    constexpr int EPV = 16 / (int)sizeof(T);
    const bool wa = wide32 & 1, wb = (wide32 >> 1) & 1;
    const uint64_t nvec = t.count / EPV;
    const int m = t.ndim;
    const int sa = (int)t.sa[m - 1], sb = (int)t.sb[m - 1];
    const uint64_t step = (uint64_t)gridDim.x * kBlock;
    for (uint64_t v = (uint64_t)blockIdx.x * kBlock + threadIdx.x; v < nvec; v += step) {
        uint64_t oa, ob;
        offsets_of<WIDE>(t, t.lin_base + v * EPV, oa, ob);
        T va[EPV], vb[EPV];
        sg_load<T>(a + oa, sa, phase_a, wa, va);
        sg_load<T>(b + ob, sb, phase_b, wb, vb);
        Pack<T, 16> r;
#pragma unroll
        for (int e = 0; e < EPV; ++e) r.e[e] = fn(va[e], vb[e], t.lane_base + v * EPV + e);
        VecIO<16, true>::store(reinterpret_cast<RawVec<16> *>(out) + v, r.raw);
    }
}

// ---------------------------------------------------------------------------
// k_dot: sum_i a[i]*b[i]  (SMArray::operator%, reference math/product.h:8-224) -- the first
// "next" row after the elementwise path (SURVEY.md §8f).  HBM-bound reduction: each thread
// accumulates UNROLL independent vector products per iteration, then warp shuffle -> shared
// memory -> one partial per CTA; the LAST CTA to finish (ticket counter) adds the partials in
// index order, so the result is deterministic for a given grid and needs no float atomics.
// int32 wraps (product.h:26-71: mullo + add_epi32), so any summation order is bit-exact;
// float/double are summed pairwise in their own type -- closer to the exact sum than the
// reference's 8 (4) sequential lane accumulators, so parity there is a tolerance.
template<typename T> struct DotAcc { using type = T; };
template<> struct DotAcc<int32_t> { using type = uint32_t; };

template<typename T>
__device__ __forceinline__ typename DotAcc<T>::type dot_mul(T x, T y) {
    if constexpr (sizeof(T) == 8) return __dmul_rn(x, y);
    else if constexpr (std::is_same<T, float>::value) return __fmul_rn(x, y);
    else return (uint32_t)x * (uint32_t)y;
}
template<typename A> __device__ __forceinline__ A dot_add(A x, A y) {
    if constexpr (std::is_same<A, double>::value) return __dadd_rn(x, y);
    else if constexpr (std::is_same<A, float>::value) return __fadd_rn(x, y);
    else return x + y;
}

// EPV: elements per load -- 16 / sizeof(T) when the two operands share a 16-byte phase (`head`
// leading elements up to the first common vector boundary are then added by block 0, like the
// ragged tail), 1 when they do not (views hand us interior pointers; the reference reads them with
// loadu, product.h:26-71): element-wise coalesced loads.
template<typename T, int UNROLL, int EPV>
__global__ void __launch_bounds__(256, SMB_DOT_MIN_BLOCKS(T)) k_dot(const T *__restrict__ a, const T *__restrict__ b, uint64_t n, uint64_t head,
                                            typename DotAcc<T>::type *__restrict__ partials, unsigned int *__restrict__ ticket,
                                            typename DotAcc<T>::type *__restrict__ result) {
    using A = typename DotAcc<T>::type;
    constexpr int VB = EPV * (int)sizeof(T);
    const uint64_t nvec = (n - head) / EPV;
    const T *av = a + head, *bv = b + head;
    A acc[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) acc[u] = A(0);
    const uint64_t stride = (uint64_t)gridDim.x * kBlock * UNROLL;
    for (uint64_t v0 = (uint64_t)blockIdx.x * kBlock * UNROLL + threadIdx.x; v0 < nvec; v0 += stride) {
        Pack<T, VB> pa[UNROLL], pb[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint64_t v = v0 + (uint64_t)u * kBlock;
            if (v < nvec) {
                if constexpr (EPV == 1) {
                    pa[u].e[0] = __ldg(av + v);
                    pb[u].e[0] = __ldg(bv + v);
                } else {
                    pa[u].raw = VecIO<VB, true>::load(reinterpret_cast<const RawVec<VB> *>(av) + v);
                    pb[u].raw = VecIO<VB, true>::load(reinterpret_cast<const RawVec<VB> *>(bv) + v);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint64_t v = v0 + (uint64_t)u * kBlock;
            if (v < nvec) {
                A s = dot_mul<T>(pa[u].e[0], pb[u].e[0]);
#pragma unroll
                for (int k = 1; k < EPV; ++k) s = dot_add<A>(s, dot_mul<T>(pa[u].e[k], pb[u].e[k]));
                acc[u] = dot_add<A>(acc[u], s);
            }
        }
    }
    A sum = acc[0];
#pragma unroll
    for (int u = 1; u < UNROLL; ++u) sum = dot_add<A>(sum, acc[u]);
    // the peeled head and the ragged tail (each < one vector) by the first threads of block 0
    if (blockIdx.x == 0) {
        if (threadIdx.x < head) sum = dot_add<A>(sum, dot_mul<T>(a[threadIdx.x], b[threadIdx.x]));
        const uint64_t tail0 = head + nvec * EPV;
        if (threadIdx.x < n - tail0) sum = dot_add<A>(sum, dot_mul<T>(a[tail0 + threadIdx.x], b[tail0 + threadIdx.x]));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sum = dot_add<A>(sum, __shfl_down_sync(0xffffffffu, sum, off));
    __shared__ A warp_sums[kBlock / 32];
    __shared__ bool is_last;
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        A s = warp_sums[0];
        for (int w = 1; w < kBlock / 32; ++w) s = dot_add<A>(s, warp_sums[w]);
        partials[blockIdx.x] = s;
        __threadfence();
        is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (is_last) { // fixed-order final reduction of the per-CTA partials
        __threadfence();
        A s = A(0);
        for (unsigned i = threadIdx.x; i < gridDim.x; i += kBlock) s = dot_add<A>(s, ((volatile A *)partials)[i]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s = dot_add<A>(s, __shfl_down_sync(0xffffffffu, s, off));
        if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            A t = warp_sums[0];
            for (int w = 1; w < kBlock / 32; ++w) t = dot_add<A>(t, warp_sums[w]);
            *result = t;
            *ticket = 0; // ready for the next launch on this stream
        }
    }
}

// ---------------------------------------------------------------------------
// k_pow_audit_f32 (test / bench support, smb_pow_audit_f32): the error of EVERY element of a
// sm::pow(x, y) result against |x|^y evaluated in double -- the value of the reference-accuracy
// pipeline before its single final rounding (log2_pos + exp2_d: relative error < 2^-31 after the
// multiplication by y, i.e. < 0.01 f32 ulp) -- in units of the f32 ulp at the correctly rounded
// result: the measure of oracle.ulp_error_f32, whose std::pow-in-double reference pins this one on
// samples (tests/test_gpu_parity.py).  Special pairs (C99 Annex F table) must match exactly.  Counts
// the elements above `bound` and keeps the maximum, so a 2^30-element result is checked
// exhaustively at memory speed instead of through sampled windows.
__global__ void __launch_bounds__(256) k_pow_audit_f32(const float *__restrict__ x, const float *__restrict__ got, uint64_t n,
                                                      PowExpF32 pe, float bound, unsigned long long *__restrict__ count_over,
                                                      unsigned int *__restrict__ max_err_bits) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned int over = 0;
    float worst = 0.0f;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float xv = x[i], g = got[i];
        const uint32_t ux = f2u(xv);
        bool negate = false, special = false;
        float want = 0.0f;
        if (!(pe.y_class == 0 && (ux - 1u) < 0x7f7fffffu)) special = pow_special<float, PowExpF32>(xv, pe, &want, &negate);
        float err;
        if (special) {
            err = (g == want && signbit(g) == signbit(want)) || (g != g && want != want) ? 0.0f : INFINITY;
        } else {
            double t = dmul((double)pe.y, log2_pos((double)u2f(ux & 0x7fffffffu)));
            t = t > 200.0 ? 200.0 : t;
            t = t < -200.0 ? -200.0 : t;
            double rd = exp2_d(t);
            if (negate) rd = -rd;
            const float r32 = (float)rd;
            if (isinf(r32) || isinf(g) || g != g) {
                err = g == r32 ? 0.0f : INFINITY;
            } else {
                const uint32_t e = (f2u(r32) >> 23) & 0xffu;
                const double ulp = e <= 1 ? 0x1p-149 : u2d((uint64_t)(e - 127 - 23 + 1023) << 52);
                err = (float)(fabs((double)g - rd) / ulp);
            }
        }
        if (!(err <= bound)) ++over;
        worst = err > worst ? err : worst;
    }
    // per-warp, then one atomic pair per warp (the kernel is read-bound; atomics are rare)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        over += __shfl_down_sync(0xffffffffu, over, off);
        worst = fmaxf(worst, __shfl_down_sync(0xffffffffu, worst, off));
    }
    if ((threadIdx.x & 31) == 0) {
        if (over) atomicAdd(count_over, (unsigned long long)over);
        atomicMax(max_err_bits, f2u(worst)); // non-negative floats order like their bit patterns
    }
}

// ---------------------------------------------------------------------------
// fill (sm::ones / sm::zeros) and the counter-based uniform generator.
template<typename T>
__global__ void __launch_bounds__(256) k_fill(T *__restrict__ out, uint64_t n, T v) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = v;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// Same arithmetic as oracle/oracle.c:orc_fill_uniform_f32 (two roundings, no FMA).
__global__ void __launch_bounds__(256) k_fill_uniform_f32(float *__restrict__ out, uint64_t first, uint64_t n,
                                                         uint64_t seed, float lo, float hi) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const float span = __fsub_rn(hi, lo);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t h = splitmix64(seed * 0xD1342543DE82EF95ull + first + i);
        const float u = __fmul_rn((float)(uint32_t)(h >> 40), 1.0f / 16777216.0f);
        out[i] = __fadd_rn(lo, __fmul_rn(span, u));
    }
}

} // namespace smb
