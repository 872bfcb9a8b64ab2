// tools/sweep.cu -- kernel-variant microbenchmark for the dense-stream and
// row-broadcast kernels (same kernels header as libsmb200.so).  Run on a B200:
//     tools/sweep [n_log2=28] [reps=20] > gpurun_out/sweep.jsonl
// Prints one JSON object per variant: {"name", params..., "ms", "gbs"}.
// The library defaults (SMB_STREAM_VB / SMB_STREAM_UNROLL / grid caps in
// smb_api.cu) are chosen from this output; summaries live under profiles/.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include <string>

#include "../simplemath_b200/csrc/smb_kernels.cuh"

using namespace smb;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); exit(1); } } while (0)

static int g_sms = 148;
static int g_reps = 20;

template<typename F>
static float time_ms(F &&launch) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) launch();
    CK(cudaDeviceSynchronize());
    std::vector<float> t;
    // median of per-launch timings AND the back-to-back average
    CK(cudaEventRecord(e0));
    for (int i = 0; i < g_reps; ++i) launch();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return ms / g_reps;
}

static void report(const char *name, const char *params, double bytes, float ms) {
    printf("{\"name\": \"%s\", \"params\": \"%s\", \"ms\": %.5f, \"gbs\": %.1f}\n", name, params, ms, bytes / (ms * 1e-3) / 1e9);
    fflush(stdout);
}

// ---------------------------------------------------------------- plain copy
template<int VB, int UNROLL>
__global__ void __launch_bounds__(256) k_copy(const float *__restrict__ a, float *__restrict__ out, uint64_t n) {
    struct Id { uint64_t lane_end; __device__ __forceinline__ float operator()(float x, float, uint64_t) const { return x; } };
    constexpr int EPV = VB / 4;
    const uint64_t nvec = n / EPV, tile_vecs = (uint64_t)blockDim.x * UNROLL, full = nvec / tile_vecs;
#pragma unroll 1
    for (uint64_t tile = blockIdx.x; tile < full; tile += gridDim.x)
        stream_tile<float, Id, false, VB, UNROLL, false>(a, nullptr, out, tile * tile_vecs + threadIdx.x, nvec, 0, Id{0});
}

// ------------------------------------------------- TMA bulk-copy pipeline add
// Persistent CTAs; a STAGES-deep ring of {a tile, b tile, out tile} in shared
// memory.  One thread issues cp.async.bulk global->shared for the operands
// (completion on an mbarrier) and cp.async.bulk shared->global for results;
// all threads do LDS.128 / FADD / STS.128 in between.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return smem_addr(p); }
__device__ __forceinline__ void bulk_s2g(void *gmem, const void *smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gmem), "r"(smem_u32(smem)), "r"(bytes) : "memory");
}

template<int TILE_BYTES, int STAGES, bool HAS_B>
__global__ void __launch_bounds__(256) k_add_tma(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ out,
                                                uint64_t n) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int TILE_ELEMS = TILE_BYTES / 4;
    constexpr int NARR = HAS_B ? 3 : 2;
    float *sa = reinterpret_cast<float *>(smem);
    float *sb = sa + (size_t)STAGES * TILE_ELEMS;
    float *so = HAS_B ? sb + (size_t)STAGES * TILE_ELEMS : sb;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)NARR * STAGES * TILE_BYTES);
    const uint64_t ntiles = n / TILE_ELEMS; // sweep sizes are multiples of the tile
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint64_t first = blockIdx.x, step = gridDim.x;
    if (threadIdx.x == 0) { // prologue: fill the ring
        for (int s = 0; s < STAGES; ++s) {
            const uint64_t t = first + (uint64_t)s * step;
            if (t < ntiles) {
                mbar_expect_tx(&full[s], HAS_B ? 2 * TILE_BYTES : TILE_BYTES);
                bulk_g2s(sa + (size_t)s * TILE_ELEMS, a + t * TILE_ELEMS, TILE_BYTES, &full[s]);
                if (HAS_B) bulk_g2s(sb + (size_t)s * TILE_ELEMS, b + t * TILE_ELEMS, TILE_BYTES, &full[s]);
            }
        }
    }
    uint32_t it = 0;
    for (uint64_t t = first; t < ntiles; t += step, ++it) {
        const int s = it % STAGES;
        const uint32_t parity = (it / STAGES) & 1;
        mbar_wait(&full[s], parity);
        // out stage s was last read by the bulk store of iteration it-STAGES; thread 0 waited for it below
        const float4 *va = reinterpret_cast<const float4 *>(sa + (size_t)s * TILE_ELEMS);
        const float4 *vb = reinterpret_cast<const float4 *>(sb + (size_t)s * TILE_ELEMS);
        float4 *vo = reinterpret_cast<float4 *>(so + (size_t)s * TILE_ELEMS);
        float4 r[TILE_BYTES / 16 / 256];
#pragma unroll
        for (int k = 0; k < TILE_BYTES / 16 / 256; ++k) {
            const float4 x = va[threadIdx.x + k * 256];
            if (HAS_B) {
                const float4 y = vb[threadIdx.x + k * 256];
                r[k] = make_float4(__fadd_rn(x.x, y.x), __fadd_rn(x.y, y.y), __fadd_rn(x.z, y.z), __fadd_rn(x.w, y.w));
            } else r[k] = x;
        }
        __syncthreads(); // everyone has read stage s inputs; thread 0 has drained out stage s
#pragma unroll
        for (int k = 0; k < TILE_BYTES / 16 / 256; ++k) vo[threadIdx.x + k * 256] = r[k];
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            bulk_s2g(out + t * TILE_ELEMS, vo, TILE_BYTES);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            const uint64_t tn = t + (uint64_t)STAGES * step;
            if (tn < ntiles) { // refill input stage s (everyone finished reading it before the first barrier)
                mbar_expect_tx(&full[s], HAS_B ? 2 * TILE_BYTES : TILE_BYTES);
                bulk_g2s(sa + (size_t)s * TILE_ELEMS, a + tn * TILE_ELEMS, TILE_BYTES, &full[s]);
                if (HAS_B) bulk_g2s(sb + (size_t)s * TILE_ELEMS, b + tn * TILE_ELEMS, TILE_BYTES, &full[s]);
            }
            // allow STAGES-1 stores in flight: the out stage the NEXT iteration writes is drained
            asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(STAGES - 1) : "memory");
        }
        // note: with STAGES >= 2 the next iteration touches a different stage, and thread 0's
        // wait_group above is ordered before everyone's writes by the first __syncthreads of that iteration
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------- drivers
template<int VB, int UNROLL>
static void run_add(const float *a, const float *b, float *out, uint64_t n) {
    const int caps[] = {0, 2, 4, 8, 16, 32};
    for (int cap : caps) {
        constexpr uint64_t per_block = 256ull * UNROLL * (VB / 4);
        uint64_t blocks = (n + per_block - 1) / per_block;
        if (cap) blocks = std::min<uint64_t>(blocks, (uint64_t)g_sms * cap);
        using Fn = BinaryFn<OP_ADD, float>;
        float ms = time_ms([&] { k_stream<float, Fn, true, VB, UNROLL><<<(unsigned)blocks, 256>>>(a, b, out, n, 0, Fn{0}, smb::kPdlWaitFirst); });
        char p[128];
        snprintf(p, sizeof p, "vb=%d unroll=%d ctas_per_sm=%d", VB, UNROLL, cap);
        report("add_f32_ldg", p, 12.0 * n, ms);
    }
}

// The pow kernel's loop (persistent grid, register double buffer, pinned prefetch) with the
// arithmetic removed: what its memory access pattern alone sustains.
struct PowLoopOnlyFn {
    static constexpr bool PAIRWISE = true;
    static constexpr bool POW_TABLES = true;
    uint64_t lane_end;
    __device__ __forceinline__ float operator()(float a, float, uint64_t) const { return a; }
    __device__ __forceinline__ float slow(float a) const { return a; }
    __device__ __forceinline__ float slow_call(float a) const { return a; }
    __device__ __forceinline__ bool pair(float a0, float a1, float &r0, float &r1) const { r0 = a0 + 1.0f; r1 = a1 + 1.0f; return true; }
    __device__ __forceinline__ void block_init() {}
    __device__ __forceinline__ void block_wait() {}
};
template<int VB, int UNROLL>
static void run_pow_loop_only(const float *a, float *out, uint64_t n) {
    const int caps[] = {1, 2, 4, 8, 16, 32, 64, 128};
    for (int cap : caps) { // cap = consecutive tiles per CTA, as the library's pow launch sizes them
        constexpr uint64_t per_block = 256ull * UNROLL * (VB / 4);
        uint64_t blocks = (n + per_block - 1) / per_block;
        blocks = (blocks + cap - 1) / cap;
        float ms = time_ms([&] { k_stream<float, PowLoopOnlyFn, false, VB, UNROLL><<<(unsigned)blocks, 256>>>(a, nullptr, out, n, 0, PowLoopOnlyFn{0}, smb::kPdlWaitFirst); });
        char p[128];
        snprintf(p, sizeof p, "vb=%d unroll=%d tiles_per_cta=%d", VB, UNROLL, cap);
        report("pow_loop_only", p, 8.0 * n, ms);
    }
}

template<int VB, int UNROLL, bool SMALL>
static void run_pow(const float *a, float *out, uint64_t n, float y) {
    const int caps[] = {1, 2, 4, 8, 16, 32, 64, 128};
    for (int cap : caps) { // cap = consecutive tiles per CTA, as the library's pow launch sizes them
        constexpr uint64_t per_block = 256ull * UNROLL * (VB / 4);
        uint64_t blocks = (n + per_block - 1) / per_block;
        blocks = (blocks + cap - 1) / cap;
        using Fn = PowF32Fn<SMALL ? POW_TIER_SMALL : POW_TIER_LARGE, POW_SIGN_REJECT, false>;
        Fn fn = Fn::make(y, 0);
        float ms = time_ms([&] { k_stream<float, Fn, false, VB, UNROLL><<<(unsigned)blocks, 256>>>(a, nullptr, out, n, 0, fn, smb::kPdlWaitFirst); });
        char p[128];
        snprintf(p, sizeof p, "y=%.2f small_y=%d vb=%d unroll=%d tiles_per_cta=%d", y, (int)SMALL, VB, UNROLL, cap);
        report("pow_f32_general", p, 8.0 * n, ms);
    }
}

template<int VB, int UNROLL>
static void run_copy(const float *a, float *out, uint64_t n) {
    const int caps[] = {0, 8, 16};
    for (int cap : caps) {
        constexpr uint64_t per_block = 256ull * UNROLL * (VB / 4);
        uint64_t blocks = (n + per_block - 1) / per_block;
        if (cap) blocks = std::min<uint64_t>(blocks, (uint64_t)g_sms * cap);
        float ms = time_ms([&] { k_copy<VB, UNROLL><<<(unsigned)blocks, 256>>>(a, out, n); });
        char p[128];
        snprintf(p, sizeof p, "vb=%d unroll=%d ctas_per_sm=%d", VB, UNROLL, cap);
        report("copy_f32_ldg", p, 8.0 * n, ms);
    }
}

template<int TILE_BYTES, int STAGES, bool HAS_B>
static void run_tma(const float *a, const float *b, float *out, uint64_t n) {
    const size_t smem = (size_t)(HAS_B ? 3 : 2) * STAGES * TILE_BYTES + 8 * STAGES;
    if (smem > 227 * 1024) return;
    CK(cudaFuncSetAttribute(k_add_tma<TILE_BYTES, STAGES, HAS_B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_add_tma<TILE_BYTES, STAGES, HAS_B>, 256, smem));
    for (int use = 1; use <= per_sm; use *= 2) {
        const unsigned grid = g_sms * use;
        float ms = time_ms([&] { k_add_tma<TILE_BYTES, STAGES, HAS_B><<<grid, 256, smem>>>(a, b, out, n); });
        char p[128];
        snprintf(p, sizeof p, "tile=%dKiB stages=%d ctas_per_sm=%d(max %d)", TILE_BYTES / 1024, STAGES, use, per_sm);
        report(HAS_B ? "add_f32_tma" : "copy_f32_tma", p, (HAS_B ? 12.0 : 8.0) * n, ms);
    }
}

template<typename T, int OP, int UNROLL>
static void run_row_variant(const char *name, const T *a, const T *b, T *out, const ElementwisePlan &p, const BcastTable &t,
                            double bytes) {
    using Fn = BinaryFn<OP, T>;
    auto reused = [&](const uint64_t *s) { for (int k = 0; k < p.ndim; ++k) if (s[k] == 0 && p.shape[k] > 1) return 1; return 0; };
    const int ar = reused(p.sa), br = reused(p.sb);
    const int caps[] = {0, 4, 8, 16, 32};
    for (int cap : caps) {
        uint64_t nvec = p.n / (16 / sizeof(T));
        uint64_t blocks = (nvec + 256 * UNROLL - 1) / (256 * UNROLL);
        if (cap) blocks = std::min<uint64_t>(blocks, (uint64_t)g_sms * cap);
        float ms = time_ms([&] { k_row<T, Fn, 16, false, UNROLL><<<(unsigned)blocks, 256>>>(a, b, out, t, ar, br, Fn{0}); });
        char pr[128];
        snprintf(pr, sizeof pr, "vec16 unroll=%d ctas_per_sm=%d", UNROLL, cap);
        report(name, pr, bytes, ms);
    }
}

template<typename T, int OP>
static void run_row(const char *name, const T *a, const T *b, T *out, const uint64_t *shape, const uint64_t *sa, const uint64_t *sb,
                    int ndim, double bytes) {
    ElementwisePlan p = make_plan(sa, sb, shape, ndim);
    BcastTable t;
    memset(&t, 0, sizeof t);
    t.ndim = p.ndim;
    for (int k = 0; k < SMB_MAX_NDIM; ++k) {
        const uint64_t d = k < p.ndim ? p.shape[k] : 1;
        t.shape64[k] = d;
        t.sa[k] = k < p.ndim ? p.sa[k] : 0;
        t.sb[k] = k < p.ndim ? p.sb[k] : 0;
        FastDiv32 f = make_fastdiv32((uint32_t)d);
        t.shape[k] = f.d; t.mul[k] = f.mul; t.shr[k] = f.shr;
    }
    t.lin_base = 0; t.count = p.n; t.lane_base = 0;
    run_row_variant<T, OP, 1>(name, a, b, out, p, t, bytes);
    run_row_variant<T, OP, 2>(name, a, b, out, p, t, bytes);
    run_row_variant<T, OP, 4>(name, a, b, out, p, t, bytes);
}

int main(int argc, char **argv) {
    const int lg = argc > 1 ? atoi(argv[1]) : 28;
    g_reps = argc > 2 ? atoi(argv[2]) : 20;
    const char *only = argc > 3 ? argv[3] : "";
    auto want = [&](const char *s) { return !*only || std::string(only).find(s) != std::string::npos; };
    const uint64_t n = 1ull << lg;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    g_sms = prop.multiProcessorCount;
    fprintf(stderr, "device %s, %d SMs, n = 2^%d\n", prop.name, g_sms, lg);
    float *a, *b, *out;
    CK(cudaMalloc(&a, n * 4));
    CK(cudaMalloc(&b, n * 4));
    CK(cudaMalloc(&out, n * 4));
    k_fill_uniform_f32<<<g_sms * 8, 256>>>(a, 0, n, 1, 0.01f, 100.f);
    k_fill_uniform_f32<<<g_sms * 8, 256>>>(b, 0, n, 2, -1.f, 1.f);
    CK(cudaDeviceSynchronize());

    if (want("memcpy")) {
        float ms = time_ms([&] { cudaMemcpyAsync(out, a, n * 4, cudaMemcpyDeviceToDevice); });
        report("cudaMemcpyD2D", "", 8.0 * n, ms);
    }
    if (want("copy")) {
        run_copy<16, 4>(a, out, n);
        run_copy<32, 2>(a, out, n);
        run_copy<32, 4>(a, out, n);
        run_tma<16384, 4, false>(a, b, out, n);
        run_tma<8192, 4, false>(a, b, out, n);
        run_tma<32768, 3, false>(a, b, out, n);
    }
    if (want("add")) {
        run_add<16, 1>(a, b, out, n);
        run_add<16, 2>(a, b, out, n);
        run_add<16, 4>(a, b, out, n);
        run_add<16, 8>(a, b, out, n);
        run_add<32, 1>(a, b, out, n);
        run_add<32, 2>(a, b, out, n);
        run_add<32, 4>(a, b, out, n);
        run_tma<16384, 4, true>(a, b, out, n);
        run_tma<16384, 3, true>(a, b, out, n);
        run_tma<8192, 4, true>(a, b, out, n);
        run_tma<8192, 8, true>(a, b, out, n);
        run_tma<4096, 4, true>(a, b, out, n);
        run_tma<4096, 8, true>(a, b, out, n);
    }
    if (want("loop")) {
        run_pow_loop_only<16, 4>(a, out, n);
        run_pow_loop_only<16, 2>(a, out, n);
        run_pow_loop_only<16, 8>(a, out, n);
    }
    if (want("pow")) {
        k_pow_image_init<<<8, 256>>>();
        CK(cudaDeviceSynchronize());
        run_pow<16, 2, true>(a, out, n, 2.5f);
        run_pow<16, 4, true>(a, out, n, 2.5f);
        run_pow<32, 2, true>(a, out, n, 2.5f);
        run_pow<16, 4, false>(a, out, n, 9.25f);
    }
    if (want("fill")) { // write-only roofline (C4 is write-dominated)
        const int caps[] = {0, 8, 16, 32};
        for (int cap : caps) {
            uint64_t blocks = (n + 1023) / 1024;
            if (cap) blocks = std::min<uint64_t>(blocks, (uint64_t)g_sms * cap);
            float ms = time_ms([&] { k_fill<uint32_t><<<(unsigned)blocks, 256>>>((uint32_t *)out, n, 5u); });
            char p[64];
            snprintf(p, sizeof p, "scalar stores ctas_per_sm=%d", cap);
            report("fill_u32", p, 4.0 * n, ms);
        }
        float ms = time_ms([&] { cudaMemsetAsync(out, 0, n * 4); });
        report("cudaMemset", "", 4.0 * n, ms);
    }
    if (want("row")) {
        { // C2: f32 {4096,4096} + {1,4096}
            const uint64_t shape[2] = {4096, 4096}, sa[2] = {4096, 1}, sb[2] = {0, 1};
            run_row<float, OP_ADD>("c2_row_add_f32", a, b, out, shape, sa, sb, 2, 4.0 * (2 * 16777216.0 + 4096));
        }
        { // C2 scaled up to 1 GiB so it is not L2-resident: {65536,4096} + {1,4096}
            const uint64_t shape[2] = {65536, 4096}, sa[2] = {4096, 1}, sb[2] = {0, 1};
            if (n >= (1ull << 28)) run_row<float, OP_ADD>("c2x16_row_add_f32", a, b, out, shape, sa, sb, 2, 4.0 * (2 * 268435456.0 + 4096));
        }
        { // C4: i32 {512,1,1024} * {1,512,1024}
            const uint64_t shape[3] = {512, 512, 1024}, sa[3] = {1024, 0, 1}, sb[3] = {0, 1024, 1};
            if (n >= (1ull << 28)) {
                run_row<int32_t, OP_MUL>("c4_row_mul_i32", (const int32_t *)a, (const int32_t *)b, (int32_t *)out, shape, sa, sb, 3, 4.0 * (268435456.0 + 2 * 524288));
                k_fill<uint32_t><<<g_sms * 8, 256>>>((uint32_t *)b, 524288, 7u);
                CK(cudaDeviceSynchronize());
                run_row<int32_t, OP_DIV>("c4_row_div_i32", (const int32_t *)a, (const int32_t *)b, (int32_t *)out, shape, sa, sb, 3, 4.0 * (268435456.0 + 2 * 524288));
            }
        }
    }
    return 0;
}
