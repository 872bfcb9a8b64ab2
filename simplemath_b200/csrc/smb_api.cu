// smb_api.cu -- the C ABI of libsmb200.so (declared in include/smb200.h): ONE translation unit.  This file holds the
// fused-chain launcher and the extern "C" entry points; the runtime underneath is included from the .inl files below
// (runtime, launchers, staging / async mode, device sets).  See DESIGN.md for the data-flow picture.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <cstdlib>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>
#include <utility>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/smb200.h"
#include "smb_alloc.h"
#include "smb_kernels.cuh"
#include "smb_plan.h"
#include "smb_shard.h"

namespace smb {

#include "smb_runtime.inl"
#include "smb_launch.inl"
#include "smb_staging.inl"
#include "smb_devices.inl"

} // namespace smb

using namespace smb;

// =============================================================== C ABI =====
// ---- op-chain fusion (SURVEY.md §8f rank 1) ---------------------------------
// sm::pow by 2, 0.5, -1, 1 has an exact single-operation form that the eager operator uses (SMB_OPT_POW_SPECIALISE, on by
// default); a pow step of a chain takes the same form, so that lazy and eager results agree bit for bit there too:
// CH_SQR, CH_SQRT, 1 / acc (CH_RDIV with the constant 1), and -- exponent 1 -- acc * 1.  -1: an ordinary pow step.
template<typename T>
static int chain_pow_special(const smb_chain_step &st) {
    if constexpr (!std::is_floating_point<T>::value) return -1;
    if (st.op != SMB_OP_POW || !g_opt_pow_specialise.load()) return -1;
    const double y = sizeof(T) == 8 ? st.value.f64 : (double)st.value.f32;
    return y == 2.0 ? CH_SQR : y == 0.5 ? CH_SQRT : y == -1.0 ? CH_RDIV : y == 1.0 ? CH_MUL : -1;
}
template<typename T>
static int chain_launch(DeviceCtx &c, const ChainPlan &p, const smb_chain_step *steps, const void *const *data,
                        uint64_t lin_begin, uint64_t lin_count, uint64_t lane_end, T *out, cudaStream_t s) {
    ChainTable t;
    memset(&t, 0, sizeof t);
    t.ndim = p.ndim;
    t.nsteps = p.nleaf;
    const bool wide = p.n > 0x7fffffffull || g_opt_force_wide.load() != 0;
    for (int k = 0; k < SMB_MAX_NDIM; ++k) {
        t.shape64[k] = p.shape[k];
        if (!wide) {
            const FastDiv32 f = make_fastdiv32((uint32_t)p.shape[k]);
            t.shape[k] = f.d; t.mul[k] = f.mul; t.shr[k] = f.shr;
        }
    }
    constexpr int EPVV = 16 / (int)sizeof(T);
    bool vec = p.inner_unit_or_zero && p.shape[p.ndim - 1] % EPVV == 0 && lin_begin % EPVV == 0 && lin_count % EPVV == 0 &&
               (uintptr_t)out % 16 == 0;
    for (int i = 0; i < p.nleaf; ++i) {
        t.data[i] = data[i];
        // leaf (op) acc: only - and / care which side the leaf is on
        t.op[i] = (uint8_t)(steps[i].swap && steps[i].op == SMB_OP_SUB ? CH_RSUB : steps[i].swap && steps[i].op == SMB_OP_DIV ? CH_RDIV : steps[i].op);
        const int special = i > 0 ? chain_pow_special<T>(steps[i]) : -1;
        if (special >= 0) t.op[i] = (uint8_t)special;
        for (int k = 0; k < SMB_MAX_NDIM; ++k) t.stride[i][k] = p.stride[i][k];
        if (!data[i]) {
            if (sizeof(T) == 8) memcpy(&t.cbits[i], &steps[i].value.f64, 8);
            else { uint32_t w; memcpy(&w, &steps[i].value.f32, 4); t.cbits[i] = w; } // f32 and i32 share the low word
            if (special == CH_RDIV || special == CH_MUL) { // 1 / acc, acc * 1: the constant becomes 1
                if constexpr (sizeof(T) == 8) { const double one = 1.0; memcpy(&t.cbits[i], &one, 8); }
                else t.cbits[i] = 0x3f800000u;
            }
        } else if (p.stride[i][p.ndim - 1] == 1) {
            if ((uintptr_t)data[i] % 16 != 0) vec = false;
            for (int k = 0; k + 1 < p.ndim; ++k) if (p.stride[i][k] % EPVV != 0) vec = false;
        }
    }
    t.lin_base = lin_begin;
    t.count = lin_count;
    t.lane_end = lane_end;
    const uint64_t items = vec ? lin_count / EPVV : lin_count;
    // f32 pow steps with an exponent the table-driven core takes: stage its tables (vector variant)
    bool powfast = false;
    t.pow_consts = pow_consts();
    t.pow_small = 1;
    if constexpr (std::is_same<T, float>::value) {
        for (int i = 1; i < p.nleaf && vec; ++i) {
            if (steps[i].op != SMB_OP_POW || chain_pow_special<T>(steps[i]) >= 0) continue;
            const PowExpF32 pe = classify_exp(steps[i].value.f32);
            if (!pow_f32_fast_ok(pe)) continue;
            t.pow_fast[i] = 1;
            t.pow_abs_mask[i] = pe.y_is_int ? 0x7fffffffu : 0xffffffffu;
            t.pow_sign_or[i] = pe.y_is_odd ? 0x80000000u : 0u;
            if (pow_f32_tier(pe) == POW_TIER_LARGE) t.pow_small = 0;
            powfast = true;
        }
    }
    // sm::pow(a (op) b, y) on dense same-shape arrays -- THE fused pow: the pow kernel itself with the operator applied
    // to the two loaded operands (k_stream<PowF32FnPre>), bit-identical to the operator followed by the pow kernel and at
    // that kernel's speed; the general chain kernel below was instruction-bound at 4.4-4.7 TB/s whatever its shape
    // (profiles/r2_chain_pow_sweep.md).
    if constexpr (std::is_same<T, float>::value) {
        if (p.nleaf == 3 && p.ndim == 1 && data[0] && data[1] && !data[2] && steps[2].op == SMB_OP_POW && chain_pow_special<T>(steps[2]) < 0 &&
            p.stride[0][0] == 1 && p.stride[1][0] == 1 && steps[1].op != SMB_OP_POW && pow_f32_fast_ok(classify_exp(steps[2].value.f32))) {
            // (any length and alignment: launch_stream peels heads and tails exactly as it does for sm::pow itself)
            const float y = steps[2].value.f32;
            const PowExpF32 pe = classify_exp(y);
            const int pre = steps[1].op == SMB_OP_ADD ? PRE_ADD : steps[1].op == SMB_OP_MUL ? PRE_MUL
                            : steps[1].op == SMB_OP_SUB ? (steps[1].swap ? PRE_RSUB : PRE_SUB) : (steps[1].swap ? PRE_RDIV : PRE_DIV);
            const float *pa = (const float *)data[0] + lin_begin, *pb = (const float *)data[1] + lin_begin;
            const bool lt1 = pow_f32_y_lt_1(pe);
            const int tier = pow_f32_tier(pe), sign = pow_f32_sign_mode(pe);
            g_last_kernel = "k_stream<pow,fused-pre>";
#define SMB_POWPRE(S, G, L) launch_stream<float, PowF32FnPre<S, G, L>, true>(c, pa, pb, (float *)out, lin_count, lin_begin, PowF32FnPre<S, G, L>::make(y, 0, pre), s)
#define SMB_POWPRE_BY_SIGN(S) (sign == POW_SIGN_REJECT ? SMB_POWPRE(S, POW_SIGN_REJECT, false) : sign == POW_SIGN_EVEN ? SMB_POWPRE(S, POW_SIGN_EVEN, false) : SMB_POWPRE(S, POW_SIGN_ODD, false))
            int rc;
            if (lt1) rc = SMB_POWPRE(POW_TIER_SMALL, POW_SIGN_REJECT, true);
            else if (tier == POW_TIER_SMALL) rc = SMB_POWPRE_BY_SIGN(POW_TIER_SMALL);
            else if (tier == POW_TIER_MEDIUM) rc = SMB_POWPRE_BY_SIGN(POW_TIER_MEDIUM);
            else rc = SMB_POWPRE_BY_SIGN(POW_TIER_LARGE);
#undef SMB_POWPRE_BY_SIGN
#undef SMB_POWPRE
            if (rc == SMB_OK) g_last_kernel = "k_stream<pow,fused-pre>";
            return rc;
        }
    }
    // sm::pow(a (op) constant, y), op in + - *, on a dense array: the pow kernel with a one-operand pre-operator (PowF32FnPre1).
    if constexpr (std::is_same<T, float>::value) {
        if (p.nleaf == 3 && p.ndim == 1 && data[0] && !data[1] && !data[2] && steps[2].op == SMB_OP_POW && chain_pow_special<T>(steps[2]) < 0 &&
            p.stride[0][0] == 1 && steps[1].op != SMB_OP_POW && steps[1].op != SMB_OP_DIV && pow_f32_fast_ok(classify_exp(steps[2].value.f32))) {
            const float y = steps[2].value.f32, cst = steps[1].value.f32;
            const PowExpF32 pe = classify_exp(y);
            const int pre = steps[1].op == SMB_OP_ADD ? PRE_ADD : steps[1].op == SMB_OP_MUL ? PRE_MUL : (steps[1].swap ? PRE_RSUB : PRE_SUB);
            const float *pa = (const float *)data[0] + lin_begin;
            const bool lt1 = pow_f32_y_lt_1(pe);
            const int tier = pow_f32_tier(pe), sign = pow_f32_sign_mode(pe);
#define SMB_POWPRE1(S, G, L) launch_stream<float, PowF32FnPre1<S, G, L>, false>(c, pa, nullptr, (float *)out, lin_count, lin_begin, PowF32FnPre1<S, G, L>::make(y, 0, pre, cst), s)
#define SMB_POWPRE1_BY_SIGN(S) (sign == POW_SIGN_REJECT ? SMB_POWPRE1(S, POW_SIGN_REJECT, false) : sign == POW_SIGN_EVEN ? SMB_POWPRE1(S, POW_SIGN_EVEN, false) : SMB_POWPRE1(S, POW_SIGN_ODD, false))
            int rc;
            if (lt1) rc = SMB_POWPRE1(POW_TIER_SMALL, POW_SIGN_REJECT, true);
            else if (tier == POW_TIER_SMALL) rc = SMB_POWPRE1_BY_SIGN(POW_TIER_SMALL);
            else if (tier == POW_TIER_MEDIUM) rc = SMB_POWPRE1_BY_SIGN(POW_TIER_MEDIUM);
            else rc = SMB_POWPRE1_BY_SIGN(POW_TIER_LARGE);
#undef SMB_POWPRE1_BY_SIGN
#undef SMB_POWPRE1
            if (rc == SMB_OK) g_last_kernel = "k_stream<pow,fused-pre1>";
            return rc;
        }
    }
    // the same two shapes for double (PowF64FnPre / PowF64FnPre1)
    if constexpr (std::is_same<T, double>::value) {
        const bool shape_ok = p.nleaf == 3 && p.ndim == 1 && data[0] && !data[2] && steps[2].op == SMB_OP_POW &&
                              chain_pow_special<T>(steps[2]) < 0 && p.stride[0][0] == 1 && steps[1].op != SMB_OP_POW;
        const bool two = shape_ok && data[1] && p.stride[1][0] == 1, one = shape_ok && !data[1] && steps[1].op != SMB_OP_DIV;
        if (two || one) {
            const double y = steps[2].value.f64;
            const PowExpF64 pe = classify_exp(y);
            const bool small = pow_f64_small_y(pe), odd = pe.y_is_odd != 0;
            const int pre = steps[1].op == SMB_OP_ADD ? PRE_ADD : steps[1].op == SMB_OP_MUL ? PRE_MUL
                            : steps[1].op == SMB_OP_SUB ? (steps[1].swap ? PRE_RSUB : PRE_SUB) : (steps[1].swap ? PRE_RDIV : PRE_DIV);
            const double *pa = (const double *)data[0] + lin_begin;
            int rc;
            if (two) {
                const double *pb = (const double *)data[1] + lin_begin;
#define SMB_POW64PRE(S, O) launch_stream<double, PowF64FnPre<S, O>, true>(c, pa, pb, (double *)out, lin_count, lin_begin, PowF64FnPre<S, O>::make(y, 0, pre), s)
                rc = small ? (odd ? SMB_POW64PRE(true, true) : SMB_POW64PRE(true, false)) : (odd ? SMB_POW64PRE(false, true) : SMB_POW64PRE(false, false));
#undef SMB_POW64PRE
                if (rc == SMB_OK) g_last_kernel = "k_stream<pow,fused-pre>";
            } else {
                const double cst = steps[1].value.f64;
#define SMB_POW64PRE1(S, O) launch_stream<double, PowF64FnPre1<S, O>, false>(c, pa, nullptr, (double *)out, lin_count, lin_begin, PowF64FnPre1<S, O>::make(y, 0, pre, cst), s)
                rc = small ? (odd ? SMB_POW64PRE1(true, true) : SMB_POW64PRE1(true, false)) : (odd ? SMB_POW64PRE1(false, true) : SMB_POW64PRE1(false, false));
#undef SMB_POW64PRE1
                if (rc == SMB_OK) g_last_kernel = "k_stream<pow,fused-pre1>";
            }
            return rc;
        }
    }
    t.tiles_per_cta = powfast ? 32 : 1; // amortise the 24 KB table copy, stay many waves deep
    // compiled-in chain capacity / vectors per thread: short chains keep more loads in flight
#define SMB_CHAIN_LAUNCH(E, W, NS, U, PF, ND)                                                                     \
    k_chain<T, E, W, NS, U, PF, ND><<<grid_for(items, (uint64_t)kThreads * U * t.tiles_per_cta, c.sm_count, 0), kThreads, 0, s>>>(out, t)
#define SMB_CHAIN_BY_LEN(E, W, PF, ND)                                                            \
    do {                                                                                          \
        if (p.nleaf <= 3 && PF) { /* sm::pow(a (op) b, e) the fused pow kernel does not take: one vector per thread */ \
            if constexpr (PF) SMB_CHAIN_LAUNCH(E, W, 3, 1, true, ND);                             \
        }                                                                                         \
        else if (p.nleaf <= 3) SMB_CHAIN_LAUNCH(E, W, 3, 4, PF, ND);                              \
        else if (p.nleaf <= 5) SMB_CHAIN_LAUNCH(E, W, 5, 2, PF, ND);                              \
        else SMB_CHAIN_LAUNCH(E, W, 8, 1, PF, ND);                                                \
    } while (0)
    // rank 1 needs no division (one 64-bit index); rank 2 and the general case come in 32- / 64-bit index forms
#define SMB_CHAIN_BY_RANK(E, PF)                                                                  \
    do {                                                                                          \
        if (p.ndim == 1) SMB_CHAIN_BY_LEN(E, true, PF, 1);                                        \
        else if (p.ndim == 2 && wide) SMB_CHAIN_BY_LEN(E, true, PF, 2);                           \
        else if (p.ndim == 2) SMB_CHAIN_BY_LEN(E, false, PF, 2);                                  \
        else if (wide) SMB_CHAIN_BY_LEN(E, true, PF, 0);                                          \
        else SMB_CHAIN_BY_LEN(E, false, PF, 0);                                                   \
    } while (0)
    if (vec && powfast) {
        if constexpr (std::is_same<T, float>::value) SMB_CHAIN_BY_RANK(EPVV, true);
        g_last_kernel = wide ? "k_chain<vec16,wide,pow>" : "k_chain<vec16,pow>";
    } else if (vec) {
        SMB_CHAIN_BY_RANK(EPVV, false);
        g_last_kernel = wide ? "k_chain<vec16,wide>" : "k_chain<vec16>";
    } else {
        if (wide) SMB_CHAIN_BY_LEN(1, true, false, 0);
        else SMB_CHAIN_BY_LEN(1, false, false, 0);
        g_last_kernel = wide ? "k_chain<scalar,wide>" : "k_chain<scalar>";
    }
#undef SMB_CHAIN_BY_RANK
#undef SMB_CHAIN_BY_LEN
#undef SMB_CHAIN_LAUNCH
    ++g_launches;
    note_other_op(); // a plain launch: the next stream kernel after it is launched plainly too
    SMB_CK(cudaGetLastError());
    return SMB_OK;
}

static int chain_dispatch(DeviceCtx &c, int dtype, const ChainPlan &p, const smb_chain_step *steps, const void *const *data,
                          uint64_t lin_begin, uint64_t lin_count, uint64_t lane_end, void *po, cudaStream_t s) {
    switch (dtype) {
        case SMB_F32: return chain_launch<float>(c, p, steps, data, lin_begin, lin_count, lane_end, (float *)po, s);
        case SMB_F64: return chain_launch<double>(c, p, steps, data, lin_begin, lin_count, lane_end, (double *)po, s);
        default: return chain_launch<int32_t>(c, p, steps, data, lin_begin, lin_count, lane_end, (int32_t *)po, s);
    }
}

static int chain_entry(int dtype, const smb_chain_step *steps, int nsteps, const uint64_t *shape, int ndim,
                       uint64_t lin_begin, uint64_t lin_count, bool whole, void *out, void *stream) {
    if (dtype < SMB_F32 || dtype > SMB_I32) return fail(SMB_ERR_INVALID, "unknown dtype %d (float, double, int32 only)", dtype);
    if (!steps || nsteps < 1 || nsteps > SMB_CHAIN_MAX) return fail(SMB_ERR_INVALID, "chain of %d steps (1..%d)", nsteps, SMB_CHAIN_MAX);
    if (ndim < 1 || ndim > SMB_MAX_NDIM || !shape) return fail(SMB_ERR_INVALID, "rank %d outside 1..%d", ndim, SMB_MAX_NDIM);
    const uint64_t *strides[SMB_CHAIN_MAX];
    for (int i = 0; i < nsteps; ++i) {
        strides[i] = steps[i].data ? steps[i].stride : nullptr;
        if (i == 0) continue;
        if (steps[i].op < SMB_OP_ADD || steps[i].op > SMB_OP_POW) return fail(SMB_ERR_INVALID, "step %d: unknown op %d", i, steps[i].op);
        if (steps[i].op == SMB_OP_POW && (steps[i].data || steps[i].swap))
            return fail(SMB_ERR_INVALID, "step %d: pow in a chain takes a constant exponent on the right (array ^ scalar)", i);
    }
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    const size_t es = esize(dtype);
    const int dev = c->device;
    // int32 pow has two semantics in the reference (AVX2 lanes wrap, the scalar tail goes through double),
    // applied by POSITION in the array sm::pow sees: array_scalar_op over the DENSE intermediate,
    // lane_end = its size rounded down to 8 (calculate.h:139-140).  The fused kernel derives the position
    // from the result's flat index, which is that array's only when the accumulator already has the
    // result's shape at the pow step.  When leaves AFTER the pow step broadcast the result further
    // (sm::pow(lazy(a{1,N}), e) + B{M,N}), the prefix up to the pow is evaluated first, as its own chain
    // of its own (smaller) shape, and joins the rest as a leaf -- bit-identical to the unfused sequence.
    if (dtype == SMB_I32 && whole) {
        for (int sidx = nsteps - 1; sidx >= 1; --sidx) {
            if (steps[sidx].op != SMB_OP_POW) continue;
            uint64_t pshape[SMB_MAX_NDIM], pn = 1, rn = 1;
            bool any_array = false;
            for (int k = 0; k < ndim; ++k) {
                bool varies = false;
                for (int i = 0; i < sidx; ++i) if (steps[i].data) { any_array = true; if (steps[i].stride[k] != 0) varies = true; }
                pshape[k] = varies || shape[k] == 1 ? shape[k] : 1;
                pn *= pshape[k];
                rn *= shape[k];
            }
            if (!any_array || pn == rn) continue;
            if (stream) return fail(SMB_ERR_INVALID, "smb_chain: an int32 pow step on a broadcast intermediate needs the synchronous form");
            // prefix [0, sidx]: strides of its leaves restricted to the dims it spans
            smb_chain_step prefix[SMB_CHAIN_MAX], rest[SMB_CHAIN_MAX];
            for (int i = 0; i <= sidx; ++i) {
                prefix[i] = steps[i];
                for (int k = 0; k < ndim; ++k) if (pshape[k] == 1) prefix[i].stride[k] = 0;
            }
            Scratch mid;
            if (int rc = mid.get(pn * es, dev)) return rc;
            if (int rc = chain_entry(dtype, prefix, sidx + 1, pshape, ndim, 0, 0, true, mid.p, nullptr)) return rc;
            if (g_opt_async.load()) SMB_CK(cudaStreamSynchronize(c->main)); // `mid` is released when this call returns
            rest[0] = smb_chain_step{};
            rest[0].data = mid.p;
            uint64_t acc = 1;
            for (int k = ndim - 1; k >= 0; --k) { rest[0].stride[k] = pshape[k] == 1 ? 0 : acc; acc *= pshape[k]; }
            int nrest = 1;
            for (int i = sidx + 1; i < nsteps; ++i) rest[nrest++] = steps[i];
            const int rc = chain_entry(dtype, rest, nrest, shape, ndim, 0, 0, true, out, nullptr);
            if (rc == SMB_OK && g_opt_async.load()) SMB_CK(cudaStreamSynchronize(c->main));
            return rc;
        }
    }
    const ChainPlan p = make_chain_plan(strides, nsteps, shape, ndim);
    if (whole) { lin_begin = 0; lin_count = p.n; }
    if (lin_begin > p.n || lin_count > p.n - lin_begin) return fail(SMB_ERR_INVALID, "flat range outside the result");
    if (lin_count == 0) return SMB_OK;
    if (!out) return fail(SMB_ERR_INVALID, "null result pointer");
    const uint64_t lane_end = dtype == SMB_I32 ? scalar_lane_end(dtype, p.n) : 0; // array_scalar_op on the dense intermediate
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    // classify the operands once
    MemType mt[SMB_CHAIN_MAX], to = mem_type(out);
    bool all_managed = to == MT_MANAGED, any_host = on_host(to);
    for (int i = 0; i < nsteps; ++i) {
        if (!steps[i].data) continue;
        mt[i] = mem_type(steps[i].data);
        if (mt[i] != MT_MANAGED) all_managed = false;
        if (on_host(mt[i])) any_host = true;
    }
    if (any_host && stream) return fail(SMB_ERR_INVALID, "smb_chain: host operands / results need the synchronous form (stream == NULL)");
    std::vector<int> devs;
    if (all_managed && want_sharding(devs, lin_count * es, stream, lin_begin == 0 && lin_count == p.n)) {
        const int G = (int)devs.size();
        const uint64_t rows = p.ndim >= 2 ? p.shape[0] : p.n, inner = p.ndim >= 2 ? p.n / p.shape[0] : 1;
        const ShardSplit split = split_flat(p.n, rows, inner, p.ndim, G, es);
        const void *bases[SMB_CHAIN_MAX];
        const uint64_t *cstr[SMB_CHAIN_MAX];
        for (int i = 0; i < nsteps; ++i) { bases[i] = steps[i].data; cstr[i] = p.stride[i]; }
        ShardOperand ops[SMB_CHAIN_MAX], res;
        if (shard_operands(devs, split, p.shape, p.ndim, bases, cstr, nsteps, es, ops)) {
            res = shard_result(devs, split, out);
            return run_sharded(devs, split, ops, nsteps, res, es, async_mode(nullptr),
                               [&](DeviceCtx &cg, int, uint64_t lo, uint64_t cnt, const void *const *use, cudaStream_t sg) {
                                   return chain_dispatch(cg, dtype, p, steps, use, lo, cnt, lane_end, (char *)out + lo * es, sg);
                               });
        }
    }
    if (int rc = begin_call(*c, stream)) return rc;
    // host leaves / result are staged whole through pooled scratch (no overlap: the fused path is
    // meant for resident arrays); managed blocks are prefetched like everywhere else
    Scratch scratch[SMB_CHAIN_MAX], dout;
    DrainGuard drain; // after the scratch blocks: an early return drains the stream before they are released
    if (any_host) drain.add(s);
    const void *data[SMB_CHAIN_MAX];
    for (int i = 0; i < nsteps; ++i) {
        data[i] = steps[i].data;
        if (!data[i]) continue;
        if (on_host(mt[i])) {
            if (int rc = scratch[i].get(p.extent[i] * es, dev)) return rc;
            note_other_op();
            SMB_CK(cudaMemcpyAsync(scratch[i].p, data[i], p.extent[i] * es, cudaMemcpyDefault, s));
            data[i] = scratch[i].p;
        } else if (mt[i] == MT_MANAGED) prefetch_managed(data[i], p.extent[i] * es, dev, s);
    }
    void *po = out;
    if (on_host(to)) {
        if (int rc = dout.get(lin_count * es, dev)) return rc;
        po = dout.p;
    } else if (to == MT_MANAGED) prefetch_managed(out, lin_count * es, dev, s, true);
    if (int rc = chain_dispatch(*c, dtype, p, steps, data, lin_begin, lin_count, lane_end, po, s)) return rc;
    note_other_op();
    if (on_host(to)) SMB_CK(cudaMemcpyAsync(out, po, lin_count * es, cudaMemcpyDefault, s));
    if (any_host) { SMB_CK(cudaStreamSynchronize(s)); return SMB_OK; } // scratch in use: synchronous whatever the mode
    return finish_call(*c, s, stream);
}
extern "C" {

int smb_elementwise(int op, int dtype, const void *a, const uint64_t *stride_a, const void *b, const uint64_t *stride_b,
                    const uint64_t *shape, int ndim, uint64_t n, void *out, void *stream) {
    if (shape && ndim >= 1 && ndim <= SMB_MAX_NDIM) {
        uint64_t prod = 1;
        for (int k = 0; k < ndim; ++k) prod *= shape[k];
        if (prod != n) return fail(SMB_ERR_INVALID, "n (%llu) != prod(shape) (%llu)", (unsigned long long)n, (unsigned long long)prod);
    }
    return elementwise_entry(op, dtype, a, stride_a, b, stride_b, shape, ndim, 0, 0, true, out, stream);
}

int smb_elementwise_range(int op, int dtype, const void *a, const uint64_t *stride_a, const void *b,
                          const uint64_t *stride_b, const uint64_t *shape, int ndim, uint64_t lin_begin,
                          uint64_t lin_count, void *out, void *stream) {
    return elementwise_entry(op, dtype, a, stride_a, b, stride_b, shape, ndim, lin_begin, lin_count, false, out, stream);
}

int smb_contiguous(int op, int dtype, const void *a, const void *b, void *out, uint64_t n, void *stream) {
    const uint64_t one = 1, shape = n;
    return elementwise_entry(op, dtype, a, &one, b, &one, &shape, 1, 0, 0, true, out, stream);
}

int smb_array_scalar(int op, int dtype, const void *a, const void *scalar, uint64_t n, void *out, void *stream) {
    if (int rc = check_args(op, dtype)) return rc;
    if (!scalar) return fail(SMB_ERR_INVALID, "null scalar pointer");
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (n == 0) return SMB_OK;
    if (!a || !out) return fail(SMB_ERR_INVALID, "null operand pointer");
    const uint64_t lane_end = scalar_lane_end(dtype, n);
    const MemType ta = mem_type(a), to = mem_type(out);
    const size_t es = esize(dtype);
    if (on_host(ta) || on_host(to)) { // always synchronous; pending asynchronous work may be producing `a`
        if (!stream && g_pending.load(std::memory_order_acquire)) if (int rc = sync_all()) return rc;
        return scalar_staged(*c, op, dtype, a, ta, scalar, out, to, n, lane_end, (cudaStream_t)stream);
    }
    std::vector<int> devs;
    if (ta == MT_MANAGED && to == MT_MANAGED && want_sharding(devs, n * es, stream, true)) {
        const int G = (int)devs.size();
        const ShardSplit split = split_flat(n, n, 1, 1, G, es);
        const uint64_t shape1[1] = {n}, unit[1] = {1};
        const void *bases[1] = {a};
        const uint64_t *strides[1] = {unit};
        ShardOperand ops[1];
        if (shard_operands(devs, split, shape1, 1, bases, strides, 1, es, ops)) {
            const ShardOperand res = shard_result(devs, split, out);
            return run_sharded(devs, split, ops, 1, res, es, async_mode(nullptr),
                               [&](DeviceCtx &cg, int, uint64_t lo, uint64_t cnt, const void *const *use, cudaStream_t s) {
                                   return scalar_device(cg, op, dtype, (const char *)use[0] + lo * es, scalar, (char *)out + lo * es, cnt, lo, lane_end, s);
                               });
        }
    }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    if (int rc = begin_call(*c, stream)) return rc;
    if (ta == MT_MANAGED) prefetch_managed(a, n * es, c->device, s);
    if (to == MT_MANAGED) prefetch_managed(out, n * es, c->device, s, true);
    if (int rc = scalar_device(*c, op, dtype, a, scalar, out, n, 0, lane_end, s)) return rc;
    return finish_call(*c, s, stream);
}

int smb_dot(int dtype, const void *a, const void *b, uint64_t n, void *result, void *stream) {
    if (dtype < SMB_F32 || dtype > SMB_I32) return fail(SMB_ERR_INVALID, "unknown dtype %d", dtype);
    if (!result) return fail(SMB_ERR_INVALID, "null result pointer");
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    const size_t es = esize(dtype);
    if (n == 0) { memset(result, 0, es); return SMB_OK; }
    if (!a || !b) return fail(SMB_ERR_INVALID, "null operand pointer");
    const MemType ta = mem_type(a), tb = mem_type(b);
    constexpr size_t kSlot = 16; // one partial result per device, in pinned memory
    Scratch pinned;
    if (int rc = pinned.get(kSlot * kMaxShards, -1, SMB_MEM_PINNED)) return rc;
    std::vector<int> devs;
    if (ta == MT_MANAGED && tb == MT_MANAGED && want_sharding(devs, 2 * n * es, stream, true)) {
        // Sharded reduction: device g reduces its flat range, the host adds the G partials in device
        // order (SURVEY.md §8f rank 2: the one place a combine step sits on a path; across PROCESSES
        // bench.py does the same with one NCCL all-reduce of a scalar).
        const int G = (int)devs.size();
        const ShardSplit split = split_flat(n, n, 1, 1, G, es);
        const uint64_t shape1[1] = {n}, unit[1] = {1};
        const void *bases[2] = {a, b};
        const uint64_t *strides[2] = {unit, unit};
        ShardOperand ops[2], none;
        if (shard_operands(devs, split, shape1, 1, bases, strides, 2, es, ops)) {
            std::vector<Scratch> partial_scratch((size_t)G);
            memset(pinned.p, 0, kSlot * (size_t)G); // a device without elements contributes zero; slot g belongs to device g (the launchers run side by side)
            // a scalar result: always synchronous (async = false), every device's stream is drained before the sum
            const int rc = run_sharded(devs, split, ops, 2, none, es, false,
                                       [&](DeviceCtx &cg, int g, uint64_t lo, uint64_t cnt, const void *const *use, cudaStream_t s) {
                                           return dot_enqueue_dtype(cg, dtype, (const char *)use[0] + lo * es, (const char *)use[1] + lo * es, cnt,
                                                                    partial_scratch[(size_t)g], (char *)pinned.p + kSlot * (size_t)g, s);
                                       });
            if (rc) return rc;
            dot_combine(dtype, pinned.p, G, kSlot, result);
            return SMB_OK;
        }
    }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    const int dev = c->device;
    if (int rc = begin_call(*c, stream)) return rc;
    Scratch da, db, work;
    DrainGuard drain;
    drain.add(s);
    note_other_op();
    if (on_host(ta)) { if (int rc = da.get(n * es, dev)) return rc; SMB_CK(cudaMemcpyAsync(da.p, a, n * es, cudaMemcpyDefault, s)); a = da.p; }
    else if (ta == MT_MANAGED) prefetch_managed(a, n * es, dev, s);
    note_other_op();
    if (on_host(tb)) { if (int rc = db.get(n * es, dev)) return rc; SMB_CK(cudaMemcpyAsync(db.p, b, n * es, cudaMemcpyDefault, s)); b = db.p; }
    else if (tb == MT_MANAGED) prefetch_managed(b, n * es, dev, s);
    if (int rc = dot_enqueue_dtype(*c, dtype, a, b, n, work, pinned.p, s)) return rc;
    SMB_CK(cudaStreamSynchronize(s)); // a scalar result: always synchronous
    dot_combine(dtype, pinned.p, 1, kSlot, result);
    return SMB_OK;
}

int smb_chain(int dtype, const smb_chain_step *steps, int nsteps, const uint64_t *shape, int ndim, uint64_t n, void *out,
              void *stream) {
    if (shape && ndim >= 1 && ndim <= SMB_MAX_NDIM) {
        uint64_t prod = 1;
        for (int k = 0; k < ndim; ++k) prod *= shape[k];
        if (prod != n) return fail(SMB_ERR_INVALID, "n = %llu is not the product of the shape (%llu)", (unsigned long long)n, (unsigned long long)prod);
    }
    return chain_entry(dtype, steps, nsteps, shape, ndim, 0, 0, true, out, stream);
}
int smb_chain_range(int dtype, const smb_chain_step *steps, int nsteps, const uint64_t *shape, int ndim, uint64_t lin_begin,
                    uint64_t lin_count, void *out, void *stream) {
    return chain_entry(dtype, steps, nsteps, shape, ndim, lin_begin, lin_count, false, out, stream);
}

void *smb_alloc(size_t bytes, int kind) {
    if (kind < SMB_MEM_DEVICE || kind > SMB_MEM_PINNED) { fail(SMB_ERR_INVALID, "unknown memory kind %d", kind); return nullptr; }
    DeviceCtx *c = nullptr;
    if (current_ctx(&c)) return nullptr;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaError_t e;
    void *p = Pool::instance().alloc(bytes, kind, dev, &e);
    if (!p) fail(e == cudaErrorMemoryAllocation ? SMB_ERR_OOM : SMB_ERR_CUDA, "smb_alloc(%zu, kind %d): %s", bytes, kind, cudaGetErrorString(e));
    return p;
}

int smb_free(void *ptr) {
    if (!ptr) return SMB_OK;
    if (!Pool::instance().free(ptr)) return fail(SMB_ERR_INVALID, "smb_free: %p was not returned by smb_alloc", ptr);
    // high-water mark: beyond it the largest cached blocks go back to the driver (cudaFree waits for
    // the device, so nothing in flight loses its memory)
    uint64_t st[4];
    Pool::instance().stats(st);
    const int64_t cap = g_opt_pool_max_cached.load(std::memory_order_relaxed);
    if (cap >= 0 && st[1] > (uint64_t)cap) Pool::instance().trim_to((uint64_t)cap);
    return SMB_OK;
}

int smb_host_written(const void *ptr) {
    if (ptr) Pool::instance().clear_placement(ptr);
    return SMB_OK;
}

int smb_owns(const void *ptr) { return ptr && Pool::instance().owns(ptr) ? 1 : 0; }

int smb_pool_trim(void) {
    cudaDeviceSynchronize();
    Pool::instance().trim();
    return SMB_OK;
}

int smb_pool_stats(uint64_t stats[4]) {
    if (!stats) return fail(SMB_ERR_INVALID, "null stats");
    Pool::instance().stats(stats);
    return SMB_OK;
}

static int fill_device(DeviceCtx &c, int dtype, void *out, const void *value, uint64_t n, cudaStream_t s) {
    const unsigned grid = grid_for(n, kThreads * 4, c.sm_count, 16);
    if (dtype == SMB_F64) k_fill<double><<<grid, kThreads, 0, s>>>((double *)out, n, *(const double *)value);
    else k_fill<uint32_t><<<grid, kThreads, 0, s>>>((uint32_t *)out, n, *(const uint32_t *)value);
    ++g_launches;
    note_other_op(); // a plain launch: the next stream kernel after it is launched plainly too
    SMB_CK(cudaGetLastError());
    return SMB_OK;
}

int smb_fill(int dtype, void *out, const void *value, uint64_t n, void *stream) {
    if (dtype < SMB_F32 || dtype > SMB_I32) return fail(SMB_ERR_INVALID, "unknown dtype %d", dtype);
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (n == 0) return SMB_OK;
    if (!out || !value) return fail(SMB_ERR_INVALID, "null pointer");
    const MemType to = mem_type(out);
    if (on_host(to)) return fail(SMB_ERR_INVALID, "smb_fill needs device or managed memory");
    const size_t es = esize(dtype);
    std::vector<int> devs;
    if (to == MT_MANAGED && want_sharding(devs, n * es, stream, true)) {
        // sm::ones / sm::zeros over the device set: the block is BORN partitioned the way the operators use it
        const int G = (int)devs.size();
        const ShardSplit split = split_flat(n, n, 1, 1, G, es);
        {
            ShardOperand ops[1];
            const ShardOperand res = shard_result(devs, split, out);
            return run_sharded(devs, split, ops, 0, res, es, async_mode(nullptr),
                               [&](DeviceCtx &cg, int, uint64_t lo, uint64_t cnt, const void *const *, cudaStream_t s) {
                                   return fill_device(cg, dtype, (char *)out + lo * es, value, cnt, s);
                               });
        }
    }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    if (int rc = begin_call(*c, stream)) return rc;
    if (to == MT_MANAGED) prefetch_managed(out, n * es, c->device, s, true);
    if (int rc = fill_device(*c, dtype, out, value, n, s)) return rc;
    return finish_call(*c, s, stream);
}

int smb_prefetch(const void *ptr, size_t bytes, int device, void *stream) {
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (mem_type(ptr) != MT_MANAGED) return SMB_OK; // nothing to migrate
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    note_other_op();
    SMB_CK(cudaMemPrefetchAsync(ptr, bytes, device < 0 ? cudaCpuDeviceId : device, s));
    if (!stream) SMB_CK(cudaStreamSynchronize(s));
    return SMB_OK;
}

int smb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int smb_set_device(int device) {
    SMB_CK(cudaSetDevice(device));
    return SMB_OK;
}
int smb_get_device(void) {
    int d = -1;
    if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return -1; }
    return d;
}
int smb_sync(void) {
    if (int rc = sync_all()) return rc;
    SMB_CK(cudaDeviceSynchronize()); // the caller's own streams on the current device too
    return SMB_OK;
}
int smb_wait_pending(void) {
    if (!g_pending.load(std::memory_order_acquire)) return SMB_OK;
    return sync_all();
}

int smb_set_devices(const int *devices, int count) {
    devices_from_env_once(); // an explicit call wins over SMB_DEVICES from here on
    if (int rc = sync_all()) return rc;
    std::lock_guard<std::mutex> lk(g_set_mu);
    return set_devices_locked(devices, count);
}
int smb_get_devices(int *devices, int capacity) {
    const std::vector<int> d = active_devices();
    if (d.empty()) {
        const int cur = smb_get_device();
        if (cur < 0) return 0;
        if (devices && capacity > 0) devices[0] = cur;
        return 1;
    }
    for (int i = 0; i < (int)d.size() && i < capacity; ++i) if (devices) devices[i] = d[i];
    return (int)d.size();
}

int smb_set_option(int key, int64_t value) {
    switch (key) {
        case SMB_OPT_POW_SPECIALISE: g_opt_pow_specialise = value ? 1 : 0; return SMB_OK;
        case SMB_OPT_STAGE_CHUNK_BYTES: g_opt_chunk_bytes = value; return SMB_OK;
        case SMB_OPT_FORCE_WIDE_INDEX: g_opt_force_wide = value ? 1 : 0; return SMB_OK;
        case SMB_OPT_ASYNC:
            if (!value && g_opt_async.load()) { g_opt_async = 0; return sync_all(); } // leaving async mode: everything lands
            g_opt_async = value ? 1 : 0;
            return SMB_OK;
        case SMB_OPT_PDL: g_opt_pdl = value < 0 ? 0 : value > 2 ? 2 : value; return SMB_OK;
        case SMB_OPT_SHARD_MIN_BYTES: g_opt_shard_min_bytes = value; return SMB_OK;
        case SMB_OPT_REPLICATE_MAX_BYTES: g_opt_replicate_max_bytes = value; return SMB_OK;
        case SMB_OPT_POOL_MAX_CACHED_BYTES: g_opt_pool_max_cached = value; return SMB_OK;
    }
    return fail(SMB_ERR_INVALID, "unknown option %d", key);
}
int64_t smb_get_option(int key) {
    switch (key) {
        case SMB_OPT_POW_SPECIALISE: return g_opt_pow_specialise;
        case SMB_OPT_STAGE_CHUNK_BYTES: return g_opt_chunk_bytes;
        case SMB_OPT_FORCE_WIDE_INDEX: return g_opt_force_wide;
        case SMB_OPT_ASYNC: return g_opt_async;
        case SMB_OPT_PDL: return g_opt_pdl;
        case SMB_OPT_SHARD_MIN_BYTES: return g_opt_shard_min_bytes;
        case SMB_OPT_REPLICATE_MAX_BYTES: return g_opt_replicate_max_bytes;
        case SMB_OPT_POOL_MAX_CACHED_BYTES: return g_opt_pool_max_cached;
    }
    return -1;
}

uint64_t smb_launch_count(void) { return g_launches.load(); }
const char *smb_last_kernel(void) { return g_last_kernel; }
const char *smb_last_error(void) { return g_err.c_str(); }
const char *smb_version(void) { return "smb200 0.1 (sm_100a)"; }

int smb_plan_chain(const smb_chain_step *steps, int nsteps, const uint64_t *shape, int ndim, int *out_ndim,
                   uint64_t *out_shape, uint64_t *out_strides) {
    if (!steps || nsteps < 1 || nsteps > SMB_CHAIN_MAX || ndim < 1 || ndim > SMB_MAX_NDIM || !shape) return -SMB_ERR_INVALID;
    const uint64_t *strides[SMB_CHAIN_MAX];
    for (int i = 0; i < nsteps; ++i) strides[i] = steps[i].data ? steps[i].stride : nullptr;
    const ChainPlan p = make_chain_plan(strides, nsteps, shape, ndim);
    if (out_ndim) *out_ndim = p.ndim;
    for (int k = 0; k < p.ndim; ++k)
        if (out_shape) out_shape[k] = p.shape[k];
    if (out_strides)
        for (int i = 0; i < nsteps; ++i)
            for (int k = 0; k < SMB_MAX_NDIM; ++k) out_strides[i * SMB_MAX_NDIM + k] = p.stride[i][k];
    return p.inner_unit_or_zero ? 1 : 0;
}

int smb_plan_elementwise(const uint64_t *stride_a, const uint64_t *stride_b, const uint64_t *shape, int ndim, int elem_size,
                         int *out_ndim, uint64_t *out_shape, uint64_t *out_stride_a, uint64_t *out_stride_b) {
    (void)elem_size;
    if (ndim < 1 || ndim > SMB_MAX_NDIM || !stride_a || !stride_b || !shape) return -SMB_ERR_INVALID;
    const ElementwisePlan p = make_plan(stride_a, stride_b, shape, ndim);
    if (out_ndim) *out_ndim = p.ndim;
    for (int k = 0; k < p.ndim; ++k) {
        if (out_shape) out_shape[k] = p.shape[k];
        if (out_stride_a) out_stride_a[k] = p.sa[k];
        if (out_stride_b) out_stride_b[k] = p.sb[k];
    }
    return p.kind;
}

int smb_plan_shards(const uint64_t *stride_a, const uint64_t *stride_b, const uint64_t *shape, int ndim, int elem_size,
                    int ndev, uint64_t *out_bounds, uint64_t *out_range_a, uint64_t *out_range_b, int *out_modes) {
    if (ndim < 1 || ndim > SMB_MAX_NDIM || !stride_a || !stride_b || !shape || ndev < 1 || ndev > kMaxShards ||
        (elem_size != 4 && elem_size != 8))
        return -SMB_ERR_INVALID;
    const ElementwisePlan p = make_plan(stride_a, stride_b, shape, ndim);
    const uint64_t rows = p.ndim >= 2 ? p.shape[0] : p.n, inner = p.ndim >= 2 && p.shape[0] ? p.n / p.shape[0] : 1;
    const ShardSplit split = split_flat(p.n, rows, inner, p.ndim, ndev, (size_t)elem_size);
    const uint64_t rmax = (uint64_t)std::max<int64_t>(0, g_opt_replicate_max_bytes.load());
    const OperandShards oa = plan_operand(p.shape, p.sa, p.ndim, split, (size_t)elem_size, rmax);
    const OperandShards ob = plan_operand(p.shape, p.sb, p.ndim, split, (size_t)elem_size, rmax);
    for (int g = 0; g <= ndev; ++g) if (out_bounds) out_bounds[g] = split.bounds[g];
    for (int g = 0; g < ndev; ++g) {
        if (out_range_a) { out_range_a[2 * g] = oa.r[g].lo; out_range_a[2 * g + 1] = oa.r[g].hi; }
        if (out_range_b) { out_range_b[2 * g] = ob.r[g].lo; out_range_b[2 * g + 1] = ob.r[g].hi; }
    }
    if (out_modes) { out_modes[0] = oa.mode; out_modes[1] = ob.mode; }
    return oa.mode == SHARD_REFUSE || ob.mode == SHARD_REFUSE ? 0 : 1;
}

int smb_register_op(const char *name, int dtype, const smb_user_op *launchers) {
    if (!name || !*name || !launchers || dtype < SMB_F32 || dtype > SMB_I32 || !launchers->contiguous || !launchers->scalar || !launchers->strided) {
        fail(SMB_ERR_INVALID, "smb_register_op: name, dtype and all three launchers are required");
        return -SMB_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lk(g_user_mu);
    int idx = -1;
    for (size_t i = 0; i < g_user_ops.size(); ++i) if (g_user_ops[i].name == name) idx = (int)i;
    if (idx < 0) { g_user_ops.emplace_back(); idx = (int)g_user_ops.size() - 1; g_user_ops[idx].name = name; }
    g_user_ops[idx].fn[dtype] = *launchers;
    g_user_ops[idx].have[dtype] = true;
    return kUserOpBase + idx;
}
int smb_find_op(const char *name) {
    if (!name) return -SMB_ERR_INVALID;
    std::lock_guard<std::mutex> lk(g_user_mu);
    for (size_t i = 0; i < g_user_ops.size(); ++i) if (g_user_ops[i].name == name) return kUserOpBase + (int)i;
    return -SMB_ERR_INVALID;
}

int smb_pow_audit_f32(const void *x, float y, const void *got, uint64_t n, float bound_ulp, uint64_t *count_over, float *max_ulp) {
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (!count_over || !max_ulp) return fail(SMB_ERR_INVALID, "null result pointer");
    *count_over = 0;
    *max_ulp = 0.0f;
    if (n == 0) return SMB_OK;
    if (!x || !got || on_host(mem_type(x)) || on_host(mem_type(got))) return fail(SMB_ERR_INVALID, "smb_pow_audit_f32 needs device or managed memory");
    if (int rc = sync_all()) return rc;
    Scratch acc;
    if (int rc = acc.get(16, c->device)) return rc;
    cudaStream_t s = c->main;
    DrainGuard drain;
    drain.add(s);
    note_other_op();
    SMB_CK(cudaMemsetAsync(acc.p, 0, 16, s));
    const unsigned grid = grid_for(n, kThreads * 8, c->sm_count, 16);
    k_pow_audit_f32<<<grid, kThreads, 0, s>>>((const float *)x, (const float *)got, n, classify_exp(y), bound_ulp,
                                             (unsigned long long *)acc.p, (unsigned int *)((char *)acc.p + 8));
    ++g_launches;
    note_other_op(); // a plain launch: the next stream kernel after it is launched plainly too
    SMB_CK(cudaGetLastError());
    unsigned long long host[2] = {0, 0};
    note_other_op();
    SMB_CK(cudaMemcpyAsync(host, acc.p, 16, cudaMemcpyDeviceToHost, s));
    SMB_CK(cudaStreamSynchronize(s));
    *count_over = host[0];
    const uint32_t bits = (uint32_t)host[1];
    memcpy(max_ulp, &bits, 4);
    return SMB_OK;
}

int smb_fill_uniform_f32(void *out, uint64_t first, uint64_t n, uint64_t seed, float lo, float hi, void *stream) {
    DeviceCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (n == 0) return SMB_OK;
    const MemType to = out ? mem_type(out) : MT_HOST;
    if (!out || on_host(to)) return fail(SMB_ERR_INVALID, "smb_fill_uniform_f32 needs device or managed memory");
    auto fill = [&](DeviceCtx &cg, float *dst, uint64_t at, uint64_t cnt, cudaStream_t s) {
        const unsigned grid = grid_for(cnt, kThreads * 4, cg.sm_count, 16);
        k_fill_uniform_f32<<<grid, kThreads, 0, s>>>(dst, first + at, cnt, seed, lo, hi);
        ++g_launches;
        note_other_op(); // a plain launch: the next stream kernel after it is launched plainly too
        SMB_CK(cudaGetLastError());
        return (int)SMB_OK;
    };
    std::vector<int> devs;
    if (to == MT_MANAGED && want_sharding(devs, n * 4, stream, true)) { // a function of the flat index: shards trivially
        const int G = (int)devs.size();
        const ShardSplit split = split_flat(n, n, 1, 1, G, 4);
        {
            ShardOperand ops[1];
            const ShardOperand res = shard_result(devs, split, out);
            return run_sharded(devs, split, ops, 0, res, 4, async_mode(nullptr),
                               [&](DeviceCtx &cg, int, uint64_t at, uint64_t cnt, const void *const *, cudaStream_t s) {
                                   return fill(cg, (float *)out + at, at, cnt, s);
                               });
        }
    }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->main;
    if (int rc = begin_call(*c, stream)) return rc;
    if (to == MT_MANAGED) prefetch_managed(out, n * 4, c->device, s, true);
    if (int rc = fill(*c, (float *)out, 0, n, s)) return rc;
    return finish_call(*c, s, stream);
}

} // extern "C"
