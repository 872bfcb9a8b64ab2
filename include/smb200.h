/*
 * smb200.h -- C ABI of libsmb200.so: the B200 (sm_100a) engine behind
 * simpleMath's elementwise hot path.
 *
 * This is the drop-in boundary.  The reference has no ABI of its own (it is a
 * header-only C++20 template library); these entry points are exactly what its
 * three hot-path function templates and its array storage would bind to.  Each
 * declaration cites the reference interface it replaces (paths relative to the
 * reference repo root).  The C++ headers under include/sm/ keep the reference's
 * names and signatures and forward to this ABI; INTEGRATION.md shows the same
 * bindings as a patch a reference maintainer would apply.
 *
 * Conventions
 *   - Plain pointers and sizes only.  No torch / CUDA types in any signature
 *     (`stream` is a cudaStream_t passed as void*).
 *   - Strides and shapes are in ELEMENTS, uint64_t, never negative
 *     (include/SMArray.h:357-364), rank <= SMB_MAX_NDIM (include/math/helpers.h:4).
 *   - Operand / result pointers may be device, managed, pinned-host or plain
 *     host memory, and may be interior pointers of a larger block (views,
 *     include/SMArray.h:397-437).  Host operands are staged through HBM by the
 *     library (chunked, copy/compute overlapped).
 *   - stream == NULL: the call is synchronous -- the result is complete when it
 *     returns, like the reference (SURVEY.md App. B.10) -- unless SMB_OPT_ASYNC is
 *     set.  stream != NULL: the work is enqueued on that stream (device / managed
 *     memory) and the caller synchronises.  A call with HOST operands (pinned
 *     included) is always synchronous: its copies start after the work already
 *     enqueued on `stream`, and the result is in host memory on return.
 *   - smb_free requires that no work the CALLER enqueued on its own streams still
 *     uses the block (work on the library's private stream is ordered by the pool).
 *   - Return value 0 on success, non-zero on error; smb_last_error() then
 *     returns a thread-local message.  The C++ wrappers rethrow it as
 *     std::runtime_error, the reference's error convention (include/SMUtils.h:77).
 *   - There is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with SMB_ERR_NO_DEVICE.
 */
#ifndef SMB200_H
#define SMB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMB_MAX_NDIM 6 /* include/math/helpers.h:4 (MAX_NDIM) */

/* Op tags: one per reference Op struct. */
enum {
    SMB_OP_ADD = 0, /* AddOp<T>       include/math/add.h:5-14        */
    SMB_OP_SUB = 1, /* SubtractOp<T>  include/math/subtract.h:5-14   */
    SMB_OP_MUL = 2, /* MultiplyOp<T>  include/math/multiply.h:7-16   */
    SMB_OP_DIV = 3, /* DivideOp<T>    include/math/division.h:8-17,67-70 */
    SMB_OP_POW = 4, /* PowOp<T>       include/math/pow.h:6-14, math/simd/crafted_pow.h:54-103 */
    SMB_OP_USER = 16 /* first id smb_register_op hands out (user-defined Op structs, README.md:86-133) */
};

/* Element types: exactly the SimdTraits<T> specialisations of the reference
 * (include/math/helpers.h:23-119). */
enum { SMB_F32 = 0, SMB_F64 = 1, SMB_I32 = 2 };

/* Memory kinds for smb_alloc. */
enum {
    SMB_MEM_DEVICE = 0,  /* HBM only (cudaMalloc), pooled                          */
    SMB_MEM_MANAGED = 1, /* host-dereferenceable, HBM-preferred (cudaMallocManaged) */
    SMB_MEM_PINNED = 2   /* page-locked host memory (cudaHostAlloc)                 */
};

/* Error codes. */
enum {
    SMB_OK = 0,
    SMB_ERR_INVALID = 1,   /* bad op / dtype / rank / null pointer */
    SMB_ERR_NO_DEVICE = 2, /* no CUDA device: there is no CPU fallback */
    SMB_ERR_CUDA = 3,      /* a CUDA runtime call failed            */
    SMB_ERR_OOM = 4
};

/* Options for smb_set_option. */
enum {
    /* 1 (default): sm::pow(arr, y) with y in {0, 1, 2, 0.5, -1} uses the exact
     * single-instruction form (x*x, sqrt, 1/x ...); 0: always run the general
     * exp2(y*log2 x) kernel (what bench.py reports as the headline). */
    SMB_OPT_POW_SPECIALISE = 0,
    /* Bytes per staging chunk of the host-operand pipeline (default 64 MiB). */
    SMB_OPT_STAGE_CHUNK_BYTES = 1,
    /* Test hook: 1 = take the 64-bit index path (results beyond 2^31 elements) for every
     * broadcast launch, so it can be exercised on small shapes. */
    SMB_OPT_FORCE_WIDE_INDEX = 4,
    /* 1: calls with stream == NULL enqueue on the library's private stream and return without waiting
     * (the asynchronous result hand-off of SURVEY.md §8f rank 4); results are complete after
     * smb_sync() / smb_wait_pending().  0 (default): the reference's contract, complete on return.
     * Calls with host (non-pinned or pinned) operands and smb_dot stay synchronous in either mode.
     * Setting it back to 0 waits for everything pending. */
    SMB_OPT_ASYNC = 5,
    /* 1 (default): back-to-back kernels on the library's PRIVATE stream (stream == NULL calls) use programmatic
     * dependent launch -- the next grid's CTAs become resident while the previous grid drains, and overlap it
     * outright when the host sees no data hazard; a kernel that follows a copy / prefetch is launched plainly.
     * 2: also on the streams callers pass in (always waiting first) -- the caller vouches that only this
     * library's kernels, events and ordinary copies precede them there (bench.py does).  0: plain stream order. */
    SMB_OPT_PDL = 6,
    /* Device set (smb_set_devices): results smaller than this many bytes stay on one device
     * (default 32 MiB). */
    SMB_OPT_SHARD_MIN_BYTES = 7,
    /* Device set: an operand several devices read (a broadcast row, an outer-product factor) is
     * kept as a read-mostly duplicate on each device when it is at most this large (default 64 MiB): the
     * driver keeps a read-only copy per device and invalidates them on any write, raw host writes
     * included.  A larger shared operand makes the operator run on one device. */
    SMB_OPT_REPLICATE_MAX_BYTES = 8,
    /* Pool high-water mark: when more than this many freed bytes sit cached, smb_free returns the
     * largest blocks to the driver (default 64 GiB; negative: never). */
    SMB_OPT_POOL_MAX_CACHED_BYTES = 9
    /* 2, 3 and 10..13 are retired: setting one fails like any unknown option, and they are not reused. */
};

/* ---- the hot path ------------------------------------------------------- */

/* Replaces element_wise_op<T, Operation>(a, stride_a, b, stride_b, n, result,
 * shape) -- include/math/calculate.h:5-99.  `stride_a` / `stride_b` are the
 * broadcast stride tables sm::broadcast() returns (0 on broadcast dims),
 * `shape` the result shape, n == prod(shape); `out` receives the dense
 * row-major result.  The fast-path dispatch (calculate.h:10-13), dimension
 * coalescing and the N-d index -> offset math all happen inside. */
int smb_elementwise(int op, int dtype,
                    const void *a, const uint64_t *stride_a,
                    const void *b, const uint64_t *stride_b,
                    const uint64_t *shape, int ndim, uint64_t n,
                    void *out, void *stream);

/* Same computation restricted to the flat output range
 * [lin_begin, lin_begin + lin_count) of the broadcast result -- the unit of
 * multi-GPU sharding (SURVEY.md §8e).  `a` and `b` address the FULL operands;
 * `out` addresses the shard: out[0] is flat element lin_begin. */
int smb_elementwise_range(int op, int dtype,
                          const void *a, const uint64_t *stride_a,
                          const void *b, const uint64_t *stride_b,
                          const uint64_t *shape, int ndim,
                          uint64_t lin_begin, uint64_t lin_count,
                          void *out, void *stream);

/* Replaces handle_contiguous_arrays<T, Operation>(a, b, result, n) --
 * include/math/calculate.h:101-134: three dense streams. */
int smb_contiguous(int op, int dtype, const void *a, const void *b, void *out,
                   uint64_t n, void *stream);

/* Replaces array_scalar_op<T, Operation>(a, value, n, result) --
 * include/math/calculate.h:137-169.  `scalar` points at one host T; it is the
 * RIGHT operand (calculate.h:159,167).  sm::pow(arr, e) is op == SMB_OP_POW
 * (include/UserFunctions.h:42-48). */
int smb_array_scalar(int op, int dtype, const void *a, const void *scalar,
                     uint64_t n, void *out, void *stream);

/* ---- next row after the elementwise path (SURVEY.md §8f) -------------------- */
/* Replaces dot_product<T>(a, b, n) behind SMArray::operator% -- include/math/product.h:8-224,
 * include/SMArray.h:213-215.  Dense operands at ANY element-aligned address (views pass interior
 * pointers; the reference reads them with loadu), `result` points at one host T.
 * int32 wraps like the reference's mullo/add_epi32 (bit-exact); float/double are summed
 * pairwise in their own type (deterministic; more accurate than the reference's sequential
 * lane accumulators, so parity is a tolerance). */
int smb_dot(int dtype, const void *a, const void *b, uint64_t n, void *result, void *stream);

/* Op-chain fusion (SURVEY.md §8f rank 1): a left-deep chain of the same Op structs evaluated in
 * ONE pass,
 *     acc = leaf_0;  acc = acc (op_i) leaf_i   [or leaf_i (op_i) acc when swap_i]   i = 1 .. nsteps-1
 * instead of one full temporary per operator (the reference materialises a fresh result in every
 * SMArray operator, include/SMArray.h:217-305, and in sm::pow, include/UserFunctions.h:42-48).
 * Each leaf is an array broadcast against the result shape (its stride table as sm::broadcast()
 * returns it, 0 on broadcast dims) or a scalar constant.  Every intermediate is rounded to T
 * exactly as the separate operators would round it (no contraction), so + - * / chains are
 * bit-identical to the unfused sequence; SMB_OP_POW needs a constant leaf as exponent (array ^
 * scalar, the only pow the reference exposes) and uses the reference-accuracy path (int32: the
 * lane / scalar-tail split of array_scalar_op on the dense intermediate).
 * Leaves must be device-accessible (device, managed or pinned memory).  At most SMB_CHAIN_MAX
 * steps. */
#define SMB_CHAIN_MAX 8
typedef struct smb_chain_step {
    int32_t op;                    /* SMB_OP_*; ignored for step 0                           */
    int32_t swap;                  /* 1: acc = leaf (op) acc                                  */
    const void *data;              /* array leaf, or NULL for the constant `value`           */
    uint64_t stride[SMB_MAX_NDIM]; /* element strides against the result shape (array leaf)  */
    union { float f32; double f64; int32_t i32; } value;
} smb_chain_step;
int smb_chain(int dtype, const smb_chain_step *steps, int nsteps,
              const uint64_t *shape, int ndim, uint64_t n, void *out, void *stream);
/* The flat output range [lin_begin, lin_begin + lin_count) only (multi-GPU shards); out[0] is
 * flat element lin_begin. */
int smb_chain_range(int dtype, const smb_chain_step *steps, int nsteps,
                    const uint64_t *shape, int ndim, uint64_t lin_begin, uint64_t lin_count,
                    void *out, void *stream);

/* ---- user-defined device Ops ------------------------------------------------------------------
 * The reference's "Extending with Custom Operations" recipe (README.md:86-133: an Op struct with
 * apply / apply_simd, used through element_wise_op<T, MyOp<T>>) without patching this library.  The
 * user's .cu file includes include/smb200_plugin.cuh, which instantiates this library's kernel
 * templates over MyOp<T>::apply_device and fills an smb_user_op; smb_register_op files it under a
 * name and returns the op id (>= SMB_OP_USER) that smb_elementwise / smb_elementwise_range /
 * smb_contiguous / smb_array_scalar then accept like a built-in one (host operands, views, device
 * sets and async mode included; smb_chain takes built-in ops only).  Registering the same name for
 * another dtype returns the same id.  The launchers return a cudaError_t value (0 = success). */
typedef struct smb_launch_env { void *stream; int sm_count; int device; } smb_launch_env;
typedef struct smb_user_op {
    /* out[i] = op(a[i], b[i]), i < n: dense streams at any element-aligned addresses */
    int (*contiguous)(const smb_launch_env *env, const void *a, const void *b, void *out, uint64_t n);
    /* out[i] = op(a[i], *scalar) */
    int (*scalar)(const smb_launch_env *env, const void *a, const void *scalar, void *out, uint64_t n);
    /* the broadcast / strided loop over a prepared stride table (smb::BcastTable of table_bytes bytes):
     * generic != 0: arbitrary element strides; else inner strides in {0,1} and `vector_bytes` (16, or the
     * element size) is the widest access the addresses and strides allow; wide != 0: 64-bit index math */
    int (*strided)(const smb_launch_env *env, const void *a, const void *b, void *out, const void *table, int table_bytes,
                   int generic, int wide, int vector_bytes, int a_reused, int b_reused);
} smb_user_op;
int smb_register_op(const char *name, int dtype, const smb_user_op *launchers);
/* The id a name was registered under, or a negative value. */
int smb_find_op(const char *name);

/* ---- storage: replaces `new T[n]` / `delete[]` of SMArray<T>::data ------- */
/* include/SMArray.h:33-34,70-76,219,342-346; include/UserFunctions.h:8-40.
 * Pooled (size-class caching) so a fresh result block per operator call costs
 * no cudaMalloc.  smb_free accepts only pointers smb_alloc returned;
 * smb_owns accepts any address, including interior ones. */
void *smb_alloc(size_t bytes, int kind);
int smb_free(void *ptr);
int smb_owns(const void *ptr);
/* Hint: the host has (re)written a managed block wholesale (constructor memcpy, a fill loop
 * through SMArray::data).  The next launch that reads it prefetches it to the GPU instead of
 * demand-paging.  Never needed for correctness. */
int smb_host_written(const void *ptr);
int smb_pool_trim(void);
/* stats[0]=bytes in use, [1]=bytes cached, [2]=cudaMalloc-class calls, [3]=pool hits */
int smb_pool_stats(uint64_t stats[4]);

/* Replaces std::fill_n in sm::ones / sm::zeros (include/UserFunctions.h:18-40):
 * fills n elements with *value on the device that owns `out`. */
int smb_fill(int dtype, void *out, const void *value, uint64_t n, void *stream);

/* Migrate a managed block to `device` (>= 0) or to the host (-1). */
int smb_prefetch(const void *ptr, size_t bytes, int device, void *stream);

/* ---- device / runtime ----------------------------------------------------- */
int smb_device_count(void);
int smb_set_device(int device);
int smb_get_device(void);
/* Waits for everything the library has enqueued on every device (and for the current device). */
int smb_sync(void);
/* SMB_OPT_ASYNC: waits only if asynchronous work is pending (one atomic load otherwise) -- what the
 * C++ headers call before the host dereferences SMArray<T>::data. */
int smb_wait_pending(void);
/* Multi-GPU behind the operator API (SURVEY.md §8e; BASELINE north_star: "large arrays are partitioned
 * across the 8 GPUs of one box by splitting the broadcast output's flat index range; broadcast
 * operands are replicated").  After smb_set_devices({d0..dG-1}) every stream == NULL operator whose
 * operands and result are MANAGED blocks (the drop-in SMArray storage) and whose result is at least
 * SMB_OPT_SHARD_MIN_BYTES is spread over those devices from the calling thread: device g computes
 * flat range g of the result on its own stream, reading its ranges of the contiguous operands in
 * place (pages prefetched to it once, then remembered) and a read-mostly duplicate of shared operands.  The
 * caller still writes `a + b` and nothing else (reference include/SMArray.h:217-225).  count <= 1
 * restores single-device behaviour; a device listed k times owns k ranges.  The environment variable SMB_DEVICES ("all", "0-7", "0,2")
 * presets the set for unmodified programs.  Device blocks (SMB_MEM_DEVICE) are computed where they
 * live; host operands go through the staging pipeline of the current device. */
int smb_set_devices(const int *devices, int count);
/* Writes up to `capacity` device indices of the active set; returns its size (1 = single device). */
int smb_get_devices(int *devices, int capacity);
int smb_set_option(int key, int64_t value);
int64_t smb_get_option(int key);
/* Kernels launched by this library in this process so far. */
uint64_t smb_launch_count(void);
/* Name of the kernel variant the last compute call on this thread launched. */
const char *smb_last_kernel(void);
const char *smb_last_error(void);
const char *smb_version(void);

/* ---- planning, exposed for host-side tests (no GPU needed) ---------------- */
/* Runs the host planner only: dimension coalescing + kernel choice for an
 * smb_elementwise call.  Writes the coalesced rank / shape / strides and
 * returns the kernel kind (>= 0: 0 contiguous, 1 row-broadcast, 2 generic
 * strided) or a negative error. */
int smb_plan_elementwise(const uint64_t *stride_a, const uint64_t *stride_b,
                         const uint64_t *shape, int ndim, int elem_size,
                         int *out_ndim, uint64_t *out_shape,
                         uint64_t *out_stride_a, uint64_t *out_stride_b);

/* The same for an smb_chain call: coalesces the result shape across all leaves (data == NULL marks a
 * constant).  Writes the coalesced rank / shape and, leaf after leaf, SMB_MAX_NDIM strides each
 * into out_strides[nsteps * SMB_MAX_NDIM].  Returns 1 when every leaf has inner stride 0 or 1 (the
 * vector kernels), 0 otherwise, or a negative error. */
int smb_plan_chain(const smb_chain_step *steps, int nsteps, const uint64_t *shape, int ndim,
                   int *out_ndim, uint64_t *out_shape, uint64_t *out_strides);

/* The multi-GPU planner alone (smb_set_devices acts on it): where the flat result range of an
 * smb_elementwise call is cut for `ndev` devices (out_bounds[ndev + 1]), which element range
 * [lo, hi) of each operand device g reads (out_range_x[2 g], [2 g + 1]) and how each operand reaches
 * the devices (out_modes: 0 in place -- the ranges are disjoint --, 1 read-mostly duplicate per device, 2 shared
 * and larger than SMB_OPT_REPLICATE_MAX_BYTES).  Returns 1 when the call would be sharded, 0 when it
 * would run on one device, or a negative error. */
int smb_plan_shards(const uint64_t *stride_a, const uint64_t *stride_b, const uint64_t *shape, int ndim,
                    int elem_size, int ndev, uint64_t *out_bounds, uint64_t *out_range_a,
                    uint64_t *out_range_b, int *out_modes);

/* ---- bench / test support -------------------------------------------------- */
/* Counter-based generator: out[i] = lo + (hi-lo) * U(seed, first+i), the same
 * arithmetic as oracle/oracle.c:orc_fill_uniform_f32, so inputs larger than
 * PCIe can comfortably carry are produced in HBM and re-derived on the CPU. */
int smb_fill_uniform_f32(void *out, uint64_t first, uint64_t n, uint64_t seed,
                         float lo, float hi, void *stream);

/* Exhaustive accuracy audit of a float sm::pow result (device or managed memory, synchronous):
 * the error of every got[i] against |x[i]|^y evaluated in double, in f32 ulps at the correctly
 * rounded result; special pairs (C99 Annex F) must match exactly (they count as infinite error
 * otherwise).  *count_over = elements whose error exceeds bound_ulp, *max_ulp = the largest error. */
int smb_pow_audit_f32(const void *x, float y, const void *got, uint64_t n, float bound_ulp,
                      uint64_t *count_over, float *max_ulp);

#ifdef __cplusplus
}
#endif
#endif /* SMB200_H */
