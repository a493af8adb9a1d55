// Design-space probe (not product code): how fast can ONE stream-ordered launch move a 65,536-env Tron batch
// (13 x 16 B per env, SoA [13][B]; the 2-D variant also at 10 of the 13 rows) HBM -> SM -> HBM, for different data-movement strategies and tile sizes?
// Same harness as bench.py: G replicas (> 4 x L2), in-place, K launches captured in one CUDA graph.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/tron_move_probe tools/tron_move_probe.cu
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstdio>
#include <cstring>
#include <cstdint>
#include <vector>
#include <algorithm>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int WORK>
__device__ __forceinline__ uint32_t busy(uint32_t x) {   // WORK dependent ALU instructions
#pragma unroll 16
    for (int i = 0; i < WORK; i++) x = x * 1664525u + 1013904223u;
    return x;
}

// V0: per-thread 128-bit loads/stores
template <int BLOCK, int WORK>
__global__ void __launch_bounds__(BLOCK) k_ldg(uint4 *st, long long B) {
    long long e = (long long)blockIdx.x * BLOCK + threadIdx.x;
    if (e >= B) return;
    uint4 v[13];
#pragma unroll
    for (int i = 0; i < 13; i++) v[i] = st[(long long)i * B + e];
    v[12].x = busy<WORK>(v[12].x ^ v[0].x);
#pragma unroll
    for (int i = 0; i < 13; i++) st[(long long)i * B + e] = v[i];
}

// V1: TMA bulk tile in / out, one tile per CTA
template <int TILE, int WORK, bool PDL>
__global__ void __launch_bounds__(TILE) k_tma(uint4 *st, long long B) {
    __shared__ __align__(128) uint4 tile[13][TILE];
    __shared__ __align__(8) uint64_t bar;
    if (PDL) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const long long e0 = (long long)blockIdx.x * TILE;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (PDL) asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&bar)), "r"(13 * TILE * 16) : "memory");
#pragma unroll
        for (int v = 0; v < 13; v++)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(&tile[v][0])), "l"(st + (long long)v * B + e0), "r"(TILE * 16), "r"(smem_u32(&bar)) : "memory");
    }
    __syncthreads();
    asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t@p bra D_%=;\n\tbra W_%=;\n\tD_%=:\n\t}" :: "r"(smem_u32(&bar)) : "memory");
    uint4 h = tile[12][threadIdx.x];
    h.x = busy<WORK>(h.x ^ tile[threadIdx.x % 12][threadIdx.x].y);
    tile[12][threadIdx.x] = h;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int v = 0; v < 13; v++)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(st + (long long)v * B + e0), "r"(smem_u32(&tile[v][0])), "r"(TILE * 16) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// V2: persistent CTAs, STAGES-deep ring of tiles: loads of the next tiles are in flight while one is processed
template <int TILE, int STAGES, int WORK>
__global__ void __launch_bounds__(TILE) k_tma_persist(uint4 *st, long long B, int ntiles) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint4 (*tile)[13][TILE] = reinterpret_cast<uint4 (*)[13][TILE]>(smem_raw);
    __shared__ __align__(8) uint64_t bar[STAGES];
    const int first = blockIdx.x, stride = gridDim.x;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&bar[s])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int it) {
        const int tl = first + it * stride, s = it % STAGES;
        if (tl < ntiles && threadIdx.x == 0) {
            const long long e0 = (long long)tl * TILE;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&bar[s])), "r"(13 * TILE * 16) : "memory");
#pragma unroll
            for (int v = 0; v < 13; v++)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(smem_u32(&tile[s][v][0])), "l"(st + (long long)v * B + e0), "r"(TILE * 16), "r"(smem_u32(&bar[s])) : "memory");
        }
    };
    for (int it = 0; it < STAGES - 1; it++) issue(it);
    for (int it = 0; first + it * stride < ntiles; it++) {
        const int s = it % STAGES;
        const uint32_t phase = (it / STAGES) & 1;
        // the slot the next load goes to was stored from at iteration it-1: wait until that store has read it
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();
        issue(it + STAGES - 1);
        asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra D_%=;\n\tbra W_%=;\n\tD_%=:\n\t}" :: "r"(smem_u32(&bar[s])), "r"(phase) : "memory");
        uint4 h = tile[s][12][threadIdx.x];
        h.x = busy<WORK>(h.x ^ tile[s][threadIdx.x % 12][threadIdx.x].y);
        tile[s][12][threadIdx.x] = h;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const long long e0 = (long long)(first + it * stride) * TILE;
#pragma unroll
            for (int v = 0; v < 13; v++)
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             :: "l"(st + (long long)v * B + e0), "r"(smem_u32(&tile[s][v][0])), "r"(TILE * 16) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// V3: ONE 2-D tensor-map TMA load and ONE store per CTA (box = TILE*4 uint32 x ROWS rows of the [13][B*4] tensor).
// HDR: like the step kernel, the box covers ROWS - 1 plane rows and the header row 12 travels as one extra 1-D bulk copy
// each way.  ROWS = 13 is the four-plane layout, ROWS = 10 the three-plane (owner code) layout.
template <int TILE, int ROWS, bool HDR>
__global__ void __launch_bounds__(TILE) k_tma2d(const __grid_constant__ CUtensorMap tm, uint4 *st, long long B) {
    __shared__ __align__(128) uint4 tile[ROWS][TILE];
    __shared__ __align__(8) uint64_t bar;
    const int x0 = (int)(blockIdx.x * TILE * 4);
    const long long e0 = (long long)blockIdx.x * TILE;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&bar)), "r"(ROWS * TILE * 16) : "memory");
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                     :: "r"(smem_u32(&tile[0][0])), "l"(&tm), "r"(x0), "r"(0), "r"(smem_u32(&bar)) : "memory");
        if (HDR)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(&tile[ROWS - 1][0])), "l"(st + 12ll * B + e0), "r"(TILE * 16), "r"(smem_u32(&bar)) : "memory");
    }
    __syncthreads();
    asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t@p bra D_%=;\n\tbra W_%=;\n\tD_%=:\n\t}" :: "r"(smem_u32(&bar)) : "memory");
    uint4 h = tile[ROWS - 1][threadIdx.x];
    h.x ^= tile[threadIdx.x % (ROWS - 1)][threadIdx.x].y;
    tile[ROWS - 1][threadIdx.x] = h;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                     :: "l"(&tm), "r"(x0), "r"(0), "r"(smem_u32(&tile[0][0])) : "memory");
        if (HDR)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(st + 12ll * B + e0), "r"(smem_u32(&tile[ROWS - 1][0])), "r"(TILE * 16) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// V4: like V1 but the 13 bulk copies are issued by 13 different warps' ... (TILE threads = TILE/32 warps): warp w issues v = w, w+W, ...
template <int TILE>
__global__ void __launch_bounds__(TILE) k_tma_split(uint4 *st, long long B) {
    __shared__ __align__(128) uint4 tile[13][TILE];
    __shared__ __align__(8) uint64_t bar;
    constexpr int W = TILE / 32;
    const long long e0 = (long long)blockIdx.x * TILE;
    const int w = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(&bar)), "r"(W));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        int nv = 0;
        for (int v = w; v < 13; v += W) nv++;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&bar)), "r"(nv * TILE * 16) : "memory");
        for (int v = w; v < 13; v += W)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(&tile[v][0])), "l"(st + (long long)v * B + e0), "r"(TILE * 16), "r"(smem_u32(&bar)) : "memory");
    }
    asm volatile("{\n\t.reg .pred p;\n\tW_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t@p bra D_%=;\n\tbra W_%=;\n\tD_%=:\n\t}" :: "r"(smem_u32(&bar)) : "memory");
    uint4 h = tile[12][threadIdx.x];
    h.x ^= tile[threadIdx.x % 12][threadIdx.x].y;
    tile[12][threadIdx.x] = h;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        for (int v = w; v < 13; v += W)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(st + (long long)v * B + e0), "r"(smem_u32(&tile[v][0])), "r"(TILE * 16) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                              const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_fn get_encode() {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    return (encode_fn)fn;
}
static CUtensorMap make_map(uint4 *p, long long B, int tile, int rows) {
    CUtensorMap tm;
    cuuint64_t dims[2] = {(cuuint64_t)B * 4, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)B * 16};
    cuuint32_t box[2] = {(cuuint32_t)tile * 4, (cuuint32_t)rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode()(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, p, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { printf("cuTensorMapEncodeTiled failed %d\n", (int)r); exit(1); }
    return tm;
}

struct Harness {
    long long B; int G, K;
    std::vector<uint4 *> rep;
    cudaStream_t s;
    Harness(long long B_, int K_) : B(B_), K(K_) {
        size_t bytes = (size_t)B * 13 * 16;
        G = (int)std::max<size_t>(2, (4ull * (126ull << 20) + bytes - 1) / bytes);
        for (int g = 0; g < G; g++) { uint4 *p; CK(cudaMalloc(&p, bytes)); CK(cudaMemset(p, g + 1, bytes)); rep.push_back(p); }
        CK(cudaStreamCreate(&s));
    }
    template <class F> double run(const char *name, F launch, int moved = 208) {
        for (int k = 0; k < G + 3; k++) launch(rep[k % G], s);
        CK(cudaStreamSynchronize(s));
        cudaGraph_t g; cudaGraphExec_t ge;
        CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeGlobal));
        for (int k = 0; k < K; k++) launch(rep[k % G], s);
        CK(cudaStreamEndCapture(s, &g));
        CK(cudaGraphInstantiate(&ge, g, 0));
        cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        double best = 1e30;
        for (int r = 0; r < 3; r++) {
            CK(cudaEventRecord(e0, s)); CK(cudaGraphLaunch(ge, s)); CK(cudaEventRecord(e1, s)); CK(cudaStreamSynchronize(s));
            float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
            best = std::min(best, (double)ms * 1e3 / K);
        }
        CK(cudaGetLastError());
        printf("%-52s %8.2f us/step  %7.1f GB/s (2 x %d B/env)\n", name, best, 2.0 * moved * B / (best * 1e-6) / 1e9, moved);
        CK(cudaGraphExecDestroy(ge)); CK(cudaGraphDestroy(g));
        return best;
    }
};

template <int TILE, int WORK, bool PDL>
void launch_tma(uint4 *p, long long B, cudaStream_t s) {
    if (!PDL) { k_tma<TILE, WORK, false><<<(unsigned)((B + TILE - 1) / TILE), TILE, 0, s>>>(p, B); return; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((B + TILE - 1) / TILE)); cfg.blockDim = dim3(TILE); cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CK(cudaLaunchKernelEx(&cfg, k_tma<TILE, WORK, true>, p, B));
}

template <int TILE, int STAGES, int WORK>
void launch_persist(uint4 *p, long long B, cudaStream_t s, int ctas_per_sm) {
    int smem = STAGES * 13 * TILE * 16;
    static bool once = false;
    if (!once) { CK(cudaFuncSetAttribute(k_tma_persist<TILE, STAGES, WORK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); once = true; }
    int ntiles = (int)(B / TILE);
    k_tma_persist<TILE, STAGES, WORK><<<148 * ctas_per_sm, TILE, smem, s>>>(p, B, ntiles);
}

// 2-D tensor-map variant at ROWS rows per environment (one map per replica)
template <int TILE, int ROWS, bool HDR>
static double run_2d(Harness &h, long long B, const char *name) {
    std::vector<CUtensorMap> maps;
    for (auto p : h.rep) maps.push_back(make_map(p, B, TILE, HDR ? ROWS - 1 : ROWS));
    auto idx = [&](uint4 *p) { return (int)(std::find(h.rep.begin(), h.rep.end(), p) - h.rep.begin()); };
    return h.run(name, [&](uint4 *p, cudaStream_t s) {
        k_tma2d<TILE, ROWS, HDR><<<(unsigned)(B / TILE), TILE, 0, s>>>(maps[idx(p)], p, B);
    }, ROWS * 16);
}

//   tron_move_probe [B] [K] [rows]: "rows" runs only the 2-D variant at 13 and 10 rows per environment
int main(int argc, char **argv) {
    long long B = argc > 1 ? atoll(argv[1]) : 65536;
    int K = argc > 2 ? atoi(argv[2]) : 400;
    const bool rows_only = argc > 3 && !strcmp(argv[3], "rows");
    Harness h(B, K);
    printf("B = %lld envs, %d replicas, %d launches per graph\n", B, h.G, K);
    if (rows_only) {
        for (int rep = 0; rep < 3; rep++) {
            const double a = run_2d<64, 13, false>(h, B, "2-D map, tile 64, 13-row box");
            const double b = run_2d<64, 10, false>(h, B, "2-D map, tile 64, 10-row box");
            const double c = run_2d<64, 13, true>(h, B, "2-D map, tile 64, 12 plane rows + header copy");
            const double d = run_2d<64, 10, true>(h, B, "2-D map, tile 64, 9 plane rows + header copy");
            printf("ratio 10/13 rows: box %.3f, planes + header %.3f  (bytes: %.3f)\n", b / a, d / c, 10.0 / 13.0);
        }
        return 0;
    }
    h.run("tma tile 32, no work", [&](uint4 *p, cudaStream_t s) { launch_tma<32, 0, false>(p, B, s); });
    h.run("tma tile 64, no work", [&](uint4 *p, cudaStream_t s) { launch_tma<64, 0, false>(p, B, s); });
    h.run("tma tile 128, no work", [&](uint4 *p, cudaStream_t s) { launch_tma<128, 0, false>(p, B, s); });
    h.run("tma tile 64, no work, PDL", [&](uint4 *p, cudaStream_t s) { launch_tma<64, 0, true>(p, B, s); });
    h.run("tma tile 128, no work, PDL", [&](uint4 *p, cudaStream_t s) { launch_tma<128, 0, true>(p, B, s); });
    run_2d<64, 13, false>(h, B, "tma 2-D tensor map, tile 64 (1 load + 1 store)");
    run_2d<32, 13, false>(h, B, "tma 2-D tensor map, tile 32 (1 load + 1 store)");
    h.run("tma tile 64, copies issued by 2 warps", [&](uint4 *p, cudaStream_t s) { k_tma_split<64><<<(unsigned)(B / 64), 64, 0, s>>>(p, B); });
    h.run("tma tile 128, copies issued by 4 warps", [&](uint4 *p, cudaStream_t s) { k_tma_split<128><<<(unsigned)(B / 128), 128, 0, s>>>(p, B); });
    h.run("persistent 148x1, tile 64, 4 stages", [&](uint4 *p, cudaStream_t s) { launch_persist<64, 4, 0>(p, B, s, 1); });
    h.run("persistent 148x2, tile 64, 3 stages", [&](uint4 *p, cudaStream_t s) { launch_persist<64, 3, 0>(p, B, s, 2); });
    h.run("persistent 148x4, tile 32, 2 stages", [&](uint4 *p, cudaStream_t s) { launch_persist<32, 2, 0>(p, B, s, 4); });
    return 0;
}
