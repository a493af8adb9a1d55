// C ABI of libcolosseum_b200.so (see include/colosseum_b200.h).  Thin launchers only: argument checks,
// grid sizing, kernel launch on the caller's stream, error capture.  No allocation, no synchronisation.
// Static helpers first, then the entry points in header order.
#ifdef CRL_HOSTSIM
#include "cuda_shim.h"
#endif
#include "crl_common.cuh"
#include "philox.cuh"
#include "tron.cuh"
#include "tron_wide.cuh"
#include "ttt.cuh"
#include "blokus.cuh"
#include "../../include/colosseum_b200.h"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <type_traits>
#include <vector>

static thread_local char g_err[512] = "";

__attribute__((format(printf, 2, 3))) static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static int check_launch(const char *what) {
#ifndef CRL_HOSTSIM
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(CRL_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
#endif
    return CRL_OK;
}

static inline unsigned blocks_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

// Launch shape of one kernel: grid, block, dynamic shared memory, and whether it is a programmatic dependent launch.
struct Launch {
    unsigned grid;
    int block, smem = 0;
    bool pdl = false;
};

// kernel<<<l.grid, l.block, l.smem, stream>>>(args...), then the launch error (if any) under `name`.  With l.pdl the
// launch carries the programmatic-stream-serialization attribute (crl_use_pdl): the kernel prefetches, waits
// (griddepcontrol.wait) for its predecessor's completion before it reads anything, and lets its successor's CTAs become
// resident right after.  Only launches carrying the attribute may start early, so ordering against any other kernel is
// unchanged.  The emulator build runs the kernel on hostsim::launch.
template <class... Params, class... Args>
static int launch(const char *name, void (*kernel)(Params...), Launch l, crl_stream_t stream, const Args &...args) {
#ifndef CRL_HOSTSIM
    if (l.pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(l.grid); cfg.blockDim = dim3(l.block); cfg.dynamicSmemBytes = l.smem;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = crl_use_pdl() ? 1 : 0;
        cudaLaunchKernelEx(&cfg, kernel, args...);
    } else {
        kernel<<<l.grid, l.block, l.smem, (cudaStream_t)stream>>>(args...);
    }
#else
    hostsim::launch(dim3(l.grid), dim3(l.block), [&] { kernel(args...); });
#endif
    return check_launch(name);
}

// f(std::integral_constant<.., v>()) for the first v of V, Vs... equal to `value`, or for the last one if none is:
// picks a kernel's template instantiation from a run-time value.
template <auto V, auto... Vs, class T, class F>
static int dispatch(T value, F &&f) {
    if constexpr (sizeof...(Vs) == 0) return f(std::integral_constant<decltype(V), V>());
    else return value == V ? f(std::integral_constant<decltype(V), V>()) : dispatch<Vs...>(value, f);
}

/* ------------------------------------------------------------------------------------------- Tron helpers */

// generate_start_positions (TronGridEnvironment.py:183-226); new_state's defaults are ring_offset = 1 and the
// deterministic spawn_offset = 2 (:228, :222-224: randint(o, o + 1) == o).  The ring `ring_offset` cells in from the
// wall is listed row-major, cut into four sides by the reference's slices, walked clockwise, split into P arcs
// (np.array_split) and the element `len//2 + spawn_offset` (clamped to the arc) of each arc is the spawn.
static int tron_starts(int N, int P, int ring_offset, const int *spawn_offsets, int32_t *heads, int32_t *dirs) {
    const int half = N / 2, odd = N % 2;
    const double center = -0.5 * (odd - 1);
    const int r_in = half - ring_offset - 1, r_out = half - ring_offset, side = 2 * (r_in + 1);
    if (ring_offset < 0 || r_in < 0 || side <= 0) return CRL_ERR_ARG;
    std::vector<int> ring_rm;
    for (int iy = 0; iy < N; iy++)
        for (int ix = 0; ix < N; ix++) {
            double y = iy - half + center, x = ix - half + center;
            bool inner = (x <= r_in && x >= -r_in && y <= r_in && y >= -r_in);
            bool outer = (x <= r_out && x >= -r_out && y <= r_out && y >= -r_out);
            if (inner != outer) ring_rm.push_back(iy * N + ix);
        }
    auto slice = [&](int start, int stop, int step) {
        std::vector<int> r;
        int L = (int)ring_rm.size();
        for (int i = start < L ? start : L; i < (stop < L ? stop : L); i += step) r.push_back(ring_rm[i]);
        return r;
    };
    std::vector<int> top = slice(0, side, 1), right = slice(side, 3 * side, 2);
    std::vector<int> bottom = slice(3 * side, 1 << 30, 1), left = slice(side + 1, 3 * side + 1, 2);
    std::vector<int> loop(top);
    loop.insert(loop.end(), right.begin(), right.end());
    loop.insert(loop.end(), bottom.rbegin(), bottom.rend());
    loop.insert(loop.end(), left.rbegin(), left.rend());
    auto arc = [&](int len, int p, int &begin, int &size) {  // np.array_split bounds
        int q = len / P, r = len % P;
        size = q + (p < r ? 1 : 0);
        begin = p * q + (p < r ? p : r);
    };
    for (int p = 0; p < P; p++) {
        int b, s;
        arc((int)loop.size(), p, b, s);
        if (s <= 0) return CRL_ERR_ARG;
        auto clamp = [](int i, int size) { return i < 0 ? 0 : (i > size - 1 ? size - 1 : i); };   // get_centers :216-220
        const int spawn_offset = spawn_offsets[p];               // one offset per player (:222-224)
        heads[p] = loop[b + clamp(s / 2 + spawn_offset, s)];
        arc(4 * side, p, b, s);
        if (s <= 0) return CRL_ERR_ARG;
        dirs[p] = ((b + clamp(s / 2 + spawn_offset, s)) / side + 2) % 4;
    }
    for (int p = 0; p < P; p++)
        for (int q = 0; q < p; q++)
            if (heads[p] == heads[q]) return CRL_ERR_ARG;    // two players on one cell (degenerate ring)
    return CRL_OK;
}

static const int TRON_DEFAULT_SPAWNS[TRONW_MAXP] = {2, 2, 2, 2, 2, 2, 2, 2};           // new_state's default spawn_offset = 2 (:228)

// per-player spawn offsets -> the fixed-size array the helpers take (absent players: 0)
static int tron_spawn_array(int P, const int32_t *spawn_offsets, int *so) {
    if (!spawn_offsets) return fail(CRL_ERR_ARG, "tron: null spawn_offsets");
    for (int p = 0; p < TRONW_MAXP; p++) so[p] = p < P ? (int)spawn_offsets[p] : 0;
    return CRL_OK;
}

// A Tron shape resolved in two steps, so that a launcher can check its pointers in between: tron_shape checks the
// ranges and picks the layout, tron_place puts the spawns into that layout's kernel parameters.  N <= 19 and P <= 4
// (BASELINE.json's shape and everything near it) run the tuned kernels of tron.cuh on the 208-byte layout (prm); every
// other shape the reference accepts runs the plain kernels of tron_wide.cuh on the word-major layout (wp).
struct TronShape {
    bool wide;
    TronParams prm;
    TronWideParams wp;
};

static int tron_shape(int N, int P, int64_t B, TronShape &s) {
    if (N < 5 || N > 64) return fail(CRL_ERR_UNSUPPORTED, "tron: board size must satisfy 5 <= N <= 64");
    if (P < 2 || P > TRONW_MAXP) return fail(CRL_ERR_UNSUPPORTED, "tron: player count must satisfy 2 <= P <= 8");
    if (B < 0) return fail(CRL_ERR_ARG, "tron: negative batch");
    s.wide = N * N > 64 * TRON_WORDS || P > 4;
    s.prm.N = s.wp.N = N;
    s.prm.P = s.wp.P = P;
    s.wp.WPP = (N * N + 31) / 32;
    s.wp.W = P * s.wp.WPP + 2 * P + 1;
    return CRL_OK;
}

// The parameters of (shape, ring_offset, spawn offsets) are cached per thread for the last few keys: every launch
// needs them and tron_starts walks the whole ring.
static int tron_place(TronShape &s, int ring_offset = 1, const int *spawn_offsets = TRON_DEFAULT_SPAWNS) {
    const int N = s.wp.N, P = s.wp.P;
    struct Entry { int key[3 + TRONW_MAXP]; TronShape s; };       // N, P, ring_offset, offsets (0 for absent players)
    static thread_local Entry cache[4];                           // (an unused entry has N = 0: never a hit)
    static thread_local int next = 0;
    int key[3 + TRONW_MAXP] = {N, P, ring_offset};
    for (int p = 0; p < P; p++) key[3 + p] = spawn_offsets[p];
    for (const Entry &e : cache)
        if (!memcmp(e.key, key, sizeof(key))) { s = e.s; return CRL_OK; }
    int32_t heads[TRONW_MAXP] = {0}, dirs[TRONW_MAXP] = {0};
    if (tron_starts(N, P, ring_offset, spawn_offsets, heads, dirs) != CRL_OK)
        return fail(CRL_ERR_ARG, "tron: cannot place spawns for this N / P / ring_offset / spawn_offset");
    for (int p = 0; p < TRONW_MAXP; p++) { s.wp.start_head[p] = heads[p]; s.wp.start_dir[p] = dirs[p]; }
    TronParams &prm = s.prm;
    prm.pmask = 0; prm.rkmask = (1u << (2 * P)) - 1u;
    TronHdr h;
    for (int p = 0; p < 4; p++) {
        if (p < P) prm.pmask |= 1u << (8 * p);
        h.hx[p] = p < P ? heads[p] % N : 0; h.hy[p] = p < P ? heads[p] / N : 0;
        h.dir[p] = p < P ? dirs[p] : 0; h.death[p] = 0; h.cells[p] = p < P ? 1 : 0;
        prm.spawn_word[p] = p < P ? (uint32_t)(heads[p] >> 5) : 0u;
        prm.spawn_bit[p] = p < P ? 1u << (heads[p] & 31) : 0u;
    }
    h.terminal = 0; h.ep_len = 0;
    uint4 e = tron_hdr_encode(h);
    prm.start_hdr[0] = e.x; prm.start_hdr[1] = e.y; prm.start_hdr[2] = e.z; prm.start_hdr[3] = e.w;
    Entry &slot = cache[next];
    memcpy(slot.key, key, sizeof(key));
    slot.s = s;
    next = (next + 1) & 3;
    return CRL_OK;
}

// Tensor map of the plane part of a Tron state buffer: [rows][B*4 uint32] (rows = TRON_PVEC), row pitch B*16 bytes,
// box = rows x tile*4 words.  The driver's encoder is fetched through the runtime (no link-time dependency on libcuda); the last
// few maps are cached per thread because an actor steps the same buffers over and over.
#ifndef CRL_HOSTSIM
typedef CUresult (*crl_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int tron_plane_map(const void *state, int64_t B, int tile, int rows, CUtensorMap *out) {
    struct Entry { const void *p; int64_t B; int tile, rows; CUtensorMap tm; };
    static thread_local Entry cache[8];
    static thread_local int next = 0;
    for (int i = 0; i < 8; i++)
        if (cache[i].p == state && cache[i].B == B && cache[i].tile == tile && cache[i].rows == rows) { *out = cache[i].tm; return CRL_OK; }
    static thread_local crl_encode_fn encode = nullptr;
    if (!encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn)
            return fail(CRL_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
        encode = (crl_encode_fn)fn;
    }
    cuuint64_t dims[2] = {(cuuint64_t)B * 4, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)B * 16};
    cuuint32_t box[2] = {(cuuint32_t)tile * 4, (cuuint32_t)rows};
    cuuint32_t estr[2] = {1, 1};
    Entry &e = cache[next];
    CUresult r = encode(&e.tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void *>(state), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { e.p = nullptr; return fail(CRL_ERR_CUDA, "cuTensorMapEncodeTiled failed"); }
    e.p = state; e.B = B; e.tile = tile; e.rows = rows;
    *out = e.tm;
    next = (next + 1) & 7;
    return CRL_OK;
}
#endif

// environments (= threads) per CTA of the step / rollout kernels: 64 (10 KB of shared memory, ~7 CTAs per SM at
// B = 65,536); CRL_TRON_TILE=32 for exploration
static int tron_tile() {
    static const int tile = [] {
        const int t = getenv("CRL_TRON_TILE") ? atoi(getenv("CRL_TRON_TILE")) : 64;
        return t == 32 ? 32 : 64;
    }();
    return tile;
}

// The fused rollout of a placed shape: the random-policy kernels when avoid_mask == 0, else their avoid instantiations.
static int tron_rollout_launch(const TronShape &s, void *state, uint8_t *result, int64_t *stats, uint64_t seed,
                               uint64_t first_env, uint32_t step0, int K, int64_t B, int avoid_mask, int noise_q16,
                               crl_stream_t stream) {
    return dispatch<false, true>(avoid_mask != 0, [&](auto AVOID) {
        if (s.wide)
            return launch("tronw_rollout_kernel", tronw_rollout_kernel<AVOID>, {blocks_for(B, 128), 128}, stream,
                          (uint32_t *)state, (uint4 *)result, (crl_u64 *)stats, B, s.wp, (crl_u64)seed, (crl_u64)first_env,
                          step0, K, (uint32_t)avoid_mask, (uint32_t)noise_q16);
        return dispatch<32, 64>(tron_tile(), [&](auto T) {
            return launch("tron_rollout_kernel", tron_rollout_kernel<T, AVOID>, {blocks_for(B, T), T}, stream,
                          (uint4 *)state, (uint2 *)result, (crl_u64 *)stats, B, s.prm, (crl_u64)seed, (crl_u64)first_env,
                          step0, K, (uint32_t)avoid_mask, (uint32_t)noise_q16);
        });
    });
}

// The checks the two avoid-policy entry points share, after the shape and pointer checks: the seat mask, the noise
// level, then the spawns (NULL = new_state's defaults) placed into the shape's parameters.
static int tron_avoid_args(const char *fn, TronShape &s, int seat_mask, int noise_q16, int ring_offset,
                           const int32_t *spawn_offsets) {
    if (seat_mask < 0 || (seat_mask >> s.wp.P) != 0) return fail(CRL_ERR_ARG, "%s: seat mask bits must be below P", fn);
    if (noise_q16 < 0 || noise_q16 > 65536) return fail(CRL_ERR_ARG, "%s: noise_q16 must satisfy 0 <= noise_q16 <= 65536", fn);
    int so[TRONW_MAXP];
    if (!spawn_offsets) return tron_place(s, ring_offset);
    tron_spawn_array(s.wp.P, spawn_offsets, so);
    return tron_place(s, ring_offset, so);
}

/* ------------------------------------------------------------------------------------------- Tic Tac Toe helpers */

// Line directions and start masks from the board dimensions (2p 3x3, 3p 3x5, 4p 3x3x3).
static int ttt_params(int n, TTTParams &prm) {
    int D[3];
    if (n == 2) { D[0] = 1; D[1] = 3; D[2] = 3; }
    else if (n == 3) { D[0] = 1; D[1] = 3; D[2] = 5; }
    else if (n == 4) { D[0] = 3; D[1] = 3; D[2] = 3; }
    else return fail(CRL_ERR_UNSUPPORTED, "tictactoe: players must be 2, 3 or 4");
    prm.n = n; prm.cells = D[0] * D[1] * D[2]; prm.cellmask = (1u << prm.cells) - 1u; prm.ndirs = 0;
    for (int d = 0; d < TTT_MAX_DIRS; d++) { prm.stride[d] = 1; prm.start[d] = 0; }
    for (int da = 0; da <= 1; da++)
        for (int db = -1; db <= 1; db++)
            for (int dc = -1; dc <= 1; dc++) {
                // canonical sign: first non-zero component positive
                if (da == 0 && (db < 0 || (db == 0 && dc <= 0))) continue;
                uint32_t start = 0;
                for (int a = 0; a < D[0]; a++)
                    for (int b = 0; b < D[1]; b++)
                        for (int c = 0; c < D[2]; c++) {
                            int a2 = a + 2 * da, b2 = b + 2 * db, c2 = c + 2 * dc;
                            if (a2 < 0 || a2 >= D[0] || b2 < 0 || b2 >= D[1] || c2 < 0 || c2 >= D[2]) continue;
                            start |= 1u << ((a * D[1] + b) * D[2] + c);
                        }
                if (!start) continue;
                prm.stride[prm.ndirs] = (uint32_t)((da * D[1] + db) * D[2] + dc);
                prm.start[prm.ndirs] = start;
                prm.ndirs++;
            }
    return CRL_OK;
}

// TTT step / rollout grids: 256 threads, a thread steps up to TTT_ACC_MAX environments (grid-stride) so that the
// fused statistics are reduced once per thread block pass; small batches keep one environment per thread.
static unsigned ttt_blocks(int64_t B) {
    const int64_t one_wave = 148 * 8 * 256;              // B200: 148 SMs x 2048 resident threads
    int64_t per_thread = (B + one_wave - 1) / one_wave;
    if (per_thread < 1) per_thread = 1;
    if (per_thread > TTT_ACC_MAX) per_thread = TTT_ACC_MAX;
    return blocks_for(B, 256 * per_thread);
}

extern "C" {

int crl_version(void) { return 100; }
const char *crl_last_error(void) { return g_err; }

int crl_init(int device) {
#ifndef CRL_HOSTSIM
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(CRL_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(CRL_ERR_ARG, "bad device index");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(CRL_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10) return fail(CRL_ERR_UNSUPPORTED, "libcolosseum_b200 is built for sm_100a only (device is %s)", prop.name);
    // (the caller's current device is left alone: launches go to the device that owns `stream`, and the host layer
    // brackets every call with a device guard -- two environments on two GPUs in one process work)
#endif
    return CRL_OK;
}

int crl_philox_words(uint32_t *out, uint64_t seed, uint64_t first_env, uint32_t step, uint32_t tag, int64_t B,
                     crl_stream_t stream) {
    if (!out || B < 0) return fail(CRL_ERR_ARG, "crl_philox_words: bad argument");
    if (B == 0) return CRL_OK;
    return launch("philox_words_kernel", philox_words_kernel, {blocks_for(B, 256), 256}, stream, (uint4 *)out,
                  (crl_u64)seed, (crl_u64)first_env, step, tag, B);
}

int crl_stats_reduce(const int64_t *stats_rows, int64_t *out, int accumulate, crl_stream_t stream) {
    if (!stats_rows || !out) return fail(CRL_ERR_ARG, "crl_stats_reduce: null pointer");
    return launch("stats_reduce_kernel", stats_reduce_kernel, {1, 256}, stream, (const crl_u64 *)stats_rows,
                  (crl_u64 *)out, accumulate);
}

/* Host-side helpers of the host-policy step loop (colosseumrl_b200/base.py::HostStepper): ONE foreign call per
 * launch (graph launch + completion-event record) and one per wait.  The loop is bound by the host's per-step cost, and a
 * ctypes call costs as much as the runtime call it wraps. */
int crl_host_graph_launch(void *graph_exec, crl_stream_t stream, void *done_event) {
#ifndef CRL_HOSTSIM
    cudaError_t e = cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream);
    if (e == cudaSuccess && done_event) e = cudaEventRecord((cudaEvent_t)done_event, (cudaStream_t)stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorInvalidResourceHandle ? CRL_ERR_ARG : CRL_ERR_CUDA, "crl_host_graph_launch: %s",
                    cudaGetErrorString(e));
    }
    return CRL_OK;
#else
    return fail(CRL_ERR_UNSUPPORTED, "crl_host_graph_launch: no CUDA runtime in the emulator build");
#endif
}

int crl_host_graph_launch_wait(void *graph_exec, crl_stream_t stream, void *done_event, void *wait_event) {
#ifndef CRL_HOSTSIM
    int rc = crl_host_graph_launch(graph_exec, stream, done_event);
    if (rc || !wait_event) return rc;
    cudaError_t e = cudaEventSynchronize((cudaEvent_t)wait_event);
    if (e != cudaSuccess) return fail(CRL_ERR_CUDA, "crl_host_graph_launch_wait: %s", cudaGetErrorString(e));
    return CRL_OK;
#else
    return fail(CRL_ERR_UNSUPPORTED, "crl_host_graph_launch_wait: no CUDA runtime in the emulator build");
#endif
}

int crl_host_event_wait(void *event) {
#ifndef CRL_HOSTSIM
    cudaError_t e = cudaEventSynchronize((cudaEvent_t)event);
    if (e != cudaSuccess) return fail(CRL_ERR_CUDA, "crl_host_event_wait: %s", cudaGetErrorString(e));
    return CRL_OK;
#else
    return fail(CRL_ERR_UNSUPPORTED, "crl_host_event_wait: no CUDA runtime in the emulator build");
#endif
}

/* ------------------------------------------------------------------------------------------- Tron */

int64_t crl_tron_state_bytes(int N, int P, int64_t B) {
    TronShape s;
    if (tron_shape(N, P, B, s)) return -1;
    return s.wide ? (int64_t)s.wp.W * 4 * B : (int64_t)TRON_VEC * 16 * B;
}

int crl_tron_action_stride(int N, int P) {
    TronShape s;
    if (tron_shape(N, P, 0, s)) return -1;
    return s.wide ? TRONW_MAXP : 4;
}

int crl_tron_result_bytes(int N, int P) {
    TronShape s;
    if (tron_shape(N, P, 0, s)) return -1;
    return s.wide ? 16 : 8;
}

int crl_tron_start_positions(int N, int P, int32_t *heads, int32_t *directions) {
    return crl_tron_start_positions_at(N, P, 1, 2, heads, directions);
}

int crl_tron_reset(void *state, const uint8_t *mask, int64_t B, int N, int P, crl_stream_t stream) {
    return crl_tron_reset_at(state, mask, B, N, P, 1, 2, stream);
}

int crl_tron_start_positions_at(int N, int P, int ring_offset, int spawn_offset, int32_t *heads, int32_t *directions) {
    int32_t so[TRONW_MAXP];
    for (int p = 0; p < TRONW_MAXP; p++) so[p] = spawn_offset;
    return crl_tron_start_positions_spawns(N, P, ring_offset, so, heads, directions);
}

int crl_tron_reset_at(void *state, const uint8_t *mask, int64_t B, int N, int P, int ring_offset, int spawn_offset,
                      crl_stream_t stream) {
    int32_t so[TRONW_MAXP];
    for (int p = 0; p < TRONW_MAXP; p++) so[p] = spawn_offset;
    return crl_tron_reset_spawns(state, mask, B, N, P, ring_offset, so, stream);
}

int crl_tron_start_positions_spawns(int N, int P, int ring_offset, const int32_t *spawn_offsets, int32_t *heads,
                                    int32_t *directions) {
    TronShape s;
    int rc = tron_shape(N, P, 0, s), so[TRONW_MAXP];
    if (rc) return rc;
    if (!heads || !directions) return fail(CRL_ERR_ARG, "crl_tron_start_positions: null pointer");
    if ((rc = tron_spawn_array(P, spawn_offsets, so))) return rc;
    if (tron_starts(N, P, ring_offset, so, heads, directions))
        return fail(CRL_ERR_ARG, "tron: cannot place spawns for this N / P / ring_offset / spawn_offset");
    return CRL_OK;
}

int crl_tron_reset_spawns(void *state, const uint8_t *mask, int64_t B, int N, int P, int ring_offset,
                          const int32_t *spawn_offsets, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s), so[TRONW_MAXP];
    if (rc) return rc;
    if (!state) return fail(CRL_ERR_ARG, "crl_tron_reset: null state");
    if ((rc = tron_spawn_array(P, spawn_offsets, so)) || (rc = tron_place(s, ring_offset, so))) return rc;
    if (B == 0) return CRL_OK;
    if (s.wide)
        return launch("tronw_reset_kernel", tronw_reset_kernel, {blocks_for(B * s.wp.W, 256), 256}, stream,
                      (uint32_t *)state, mask, B, s.wp);
    return launch("tron_reset_kernel", tron_reset_kernel, {blocks_for(B * TRON_VEC, 256), 256}, stream, (uint4 *)state,
                  mask, B, s.prm);
}

int crl_tron_step_spawns(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result, int64_t *stats,
                         int64_t B, int N, int P, int flags, int ring_offset, const int32_t *spawn_offsets,
                         crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s), so[TRONW_MAXP];
    if (rc || (rc = tron_spawn_array(P, spawn_offsets, so))) return rc;
    if (!state_in || !state_out || !actions || !result) return fail(CRL_ERR_ARG, "crl_tron_step: null pointer");
    if (s.wide && (flags & (CRL_FLAG_COMPACT_RESULT | CRL_FLAG_COMPACT2_RESULT | CRL_FLAG_PACKED_ACTIONS)))
        return fail(CRL_ERR_UNSUPPORTED, "crl_tron_step: compact records / packed actions exist for N <= 19, P <= 4 only");
    if ((rc = tron_place(s, ring_offset, so))) return rc;
    if (B == 0) return CRL_OK;
    if (s.wide) {
        if (((uintptr_t)actions & 7) || ((uintptr_t)result & 15))
            return fail(CRL_ERR_ARG, "crl_tron_step: actions must be 8-byte, result 16-byte aligned");
        return launch("tronw_step_kernel", tronw_step_kernel, {blocks_for(B, 128), 128}, stream, (const uint32_t *)state_in,
                      (uint32_t *)state_out, actions, (uint4 *)result, (crl_u64 *)stats, B, s.wp, flags);
    }
    if (((uintptr_t)state_in | (uintptr_t)state_out) & 15) return fail(CRL_ERR_ARG, "crl_tron_step: state buffers must be 16-byte aligned");
    if (B > (INT32_MAX >> 2)) return fail(CRL_ERR_UNSUPPORTED, "crl_tron_step: batch too large for one launch");
    TronMaps maps;
    const int tile = tron_tile();
#ifndef CRL_HOSTSIM
    if ((rc = tron_plane_map(state_in, B, tile, TRON_PVEC, &maps.in)) ||
        (rc = tron_plane_map(state_out, B, tile, TRON_PVEC, &maps.out)))
        return rc;
#else
    maps.in_ptr = (const uint4 *)state_in; maps.out_ptr = (uint4 *)state_out;
#endif
    return dispatch<32, 64>(tile, [&](auto T) {
        return launch("tron_step_kernel", tron_step_kernel<T>, {blocks_for(B, T), T, 0, true}, stream, maps,
                      (const uint4 *)state_in, (uint4 *)state_out, (const uint32_t *)actions, (uint2 *)result,
                      (crl_u64 *)stats, B, s.prm, flags);
    });
}

int crl_tron_step(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result, int64_t *stats,
                  int64_t B, int N, int P, int flags, crl_stream_t stream) {
    return crl_tron_step_spawns(state_in, state_out, actions, result, stats, B, N, P, flags, 1, TRON_DEFAULT_SPAWNS, stream);
}

int crl_tron_policy_random(int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step, int64_t B,
                           crl_stream_t stream) {
    if (!actions || B < 0) return fail(CRL_ERR_ARG, "crl_tron_policy_random: bad argument");
    if (B == 0) return CRL_OK;
    return launch("tron_policy_random_kernel", tron_policy_random_kernel, {blocks_for(B, 256), 256}, stream,
                  (uint32_t *)actions, B, (crl_u64)seed, (crl_u64)first_env, step);
}

int crl_tron_policy_random_wide(int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step, int64_t B,
                                crl_stream_t stream) {
    if (!actions || B < 0 || ((uintptr_t)actions & 7)) return fail(CRL_ERR_ARG, "crl_tron_policy_random_wide: bad argument");
    if (B == 0) return CRL_OK;
    return launch("tronw_policy_random_kernel", tronw_policy_random_kernel, {blocks_for(B, 256), 256}, stream, actions, B,
                  (crl_u64)seed, (crl_u64)first_env, step);
}

int crl_tron_rollout(void *state, uint8_t *result, int64_t *stats, uint64_t seed, uint64_t first_env,
                     uint32_t step0, int K, int64_t B, int N, int P, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state || K < 0) return fail(CRL_ERR_ARG, "crl_tron_rollout: bad argument");
    if ((rc = tron_place(s))) return rc;
    if (B == 0 || K == 0) return CRL_OK;
    return tron_rollout_launch(s, state, result, stats, seed, first_env, step0, K, B, 0, 0, stream);
}

int crl_tron_observe(const void *state, int player, int8_t *board, int32_t *heads, int32_t *directions,
                     int32_t *deaths, uint8_t *terminal, int64_t B, int N, int P, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state || !board || player >= P || player < -3 || player == -2) return fail(CRL_ERR_ARG, "crl_tron_observe: bad argument");
    if ((rc = tron_place(s))) return rc;
    if (B == 0) return CRL_OK;
    const int nview = player == -3 ? P : 1;
    if (s.wide)
        return launch("tronw_observe_kernel", tronw_observe_kernel, {blocks_for(B * nview * N * N, 256), 256}, stream,
                      (const uint32_t *)state, B, s.wp, player, board, heads, directions, deaths, terminal);
    const int img_bytes = (TRON_OBS_TILE * nview * N * N + 15) & ~15;
    return dispatch<true, false>(player == -3, [&](auto ALL) {
        return launch("tron_observe_kernel", tron_observe_kernel<ALL>, {blocks_for(B, TRON_OBS_TILE), 128, img_bytes},
                      stream, (const uint4 *)state, B, s.prm, player, board, heads, directions, deaths, terminal);
    });
}

int crl_tron_ranking(const void *state, uint8_t *ranking, int64_t B, int N, int P, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state || !ranking) return fail(CRL_ERR_ARG, "crl_tron_ranking: null pointer");
    if ((rc = tron_place(s))) return rc;
    if (B == 0) return CRL_OK;
    if (s.wide) {                                            // uint32 per environment, 3 bits per player
        if ((uintptr_t)ranking & 3) return fail(CRL_ERR_ARG, "crl_tron_ranking: ranking must be 4-byte aligned for wide shapes");
        return launch("tronw_ranking_kernel", tronw_ranking_kernel, {blocks_for(B, 256), 256}, stream,
                      (const uint32_t *)state, B, s.wp, (uint32_t *)ranking);
    }
    return launch("tron_ranking_kernel", tron_ranking_kernel, {blocks_for(B, 256), 256}, stream, (const uint4 *)state, B,
                  s.prm, ranking);
}

int crl_tron_pack(void *state, const int8_t *board, const int32_t *heads, const int32_t *directions,
                  const int32_t *deaths, int64_t B, int N, int P, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state || !board || !heads || !directions || !deaths) return fail(CRL_ERR_ARG, "crl_tron_pack: null pointer");
    if ((rc = tron_place(s))) return rc;
    if (B == 0) return CRL_OK;
    if (s.wide)
        return launch("tronw_pack_kernel", tronw_pack_kernel, {blocks_for(B * s.wp.W, 256), 256}, stream, (uint32_t *)state,
                      B, s.wp, board, heads, directions, deaths);
    return launch("tron_pack_kernel", tron_pack_kernel, {blocks_for(B, 128), 128}, stream, (uint4 *)state, B, s.prm,
                  board, heads, directions, deaths);
}

/* ------------------------------------------------------------------------------------------- Tic Tac Toe */

int crl_ttt_cells(int n) {
    TTTParams prm;
    return ttt_params(n, prm) ? -1 : prm.cells;
}

int crl_ttt_lines(int n, uint32_t *line_masks, int capacity) {
    TTTParams prm;
    if (ttt_params(n, prm)) return -1;
    int cnt = 0;
    for (int d = 0; d < prm.ndirs; d++)
        for (int c = 0; c < prm.cells; c++)
            if (prm.start[d] >> c & 1) {
                if (line_masks && cnt < capacity)
                    line_masks[cnt] = 1u << c | 1u << (c + prm.stride[d]) | 1u << (c + 2 * prm.stride[d]);
                cnt++;
            }
    return cnt;
}

int crl_ttt_reset(void *state, const uint8_t *mask, int64_t B, int n, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || B < 0) return fail(CRL_ERR_ARG, "crl_ttt_reset: bad argument");
    if (B == 0) return CRL_OK;
    return launch("ttt_reset_kernel", ttt_reset_kernel, {blocks_for(B, 256), 256}, stream, (uint4 *)state, mask, B);
}

int crl_ttt_step(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result, uint32_t *valid_after,
                 int64_t *stats, int64_t B, int n, int flags, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state_in || !state_out || !actions || !result || B < 0) return fail(CRL_ERR_ARG, "crl_ttt_step: bad argument");
    if (B == 0) return CRL_OK;
    return dispatch<2, 3, 4>(n, [&](auto NP) {
        return launch("ttt_step_kernel", ttt_step_kernel<NP>, {ttt_blocks(B), 256, 0, true}, stream,
                      (const uint4 *)state_in, (uint4 *)state_out, actions, (uint32_t *)result, valid_after,
                      (crl_u64 *)stats, B, flags);
    });
}

int crl_ttt_valid_actions(const void *state, uint32_t *mask, int64_t B, int n, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || !mask || B < 0) return fail(CRL_ERR_ARG, "crl_ttt_valid_actions: bad argument");
    if (B == 0) return CRL_OK;
    return launch("ttt_valid_kernel", ttt_valid_kernel, {blocks_for(B, 256), 256}, stream, (const uint4 *)state, mask, B,
                  prm);
}

int crl_ttt_policy_random(const void *state, int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step,
                          int64_t B, int n, int flags, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || !actions || B < 0) return fail(CRL_ERR_ARG, "crl_ttt_policy_random: bad argument");
    if (B == 0) return CRL_OK;
    return dispatch<2, 3, 4>(n, [&](auto NP) {
        return launch("ttt_policy_random_kernel", ttt_policy_random_kernel<NP>, {blocks_for(B, 256), 256}, stream,
                      (const uint4 *)state, actions, B, flags, (crl_u64)seed, (crl_u64)first_env, step);
    });
}

int crl_ttt_rollout(void *state, uint8_t *result, int64_t *stats, uint64_t seed, uint64_t first_env, uint32_t step0,
                    int K, int64_t B, int n, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || B < 0 || K < 0) return fail(CRL_ERR_ARG, "crl_ttt_rollout: bad argument");
    if (B == 0 || K == 0) return CRL_OK;
    if (B >= (int64_t)1 << 31) return fail(CRL_ERR_UNSUPPORTED, "crl_ttt_rollout: batch too large for one launch");
    const PhiloxKeys keys = philox_expand_keys((crl_u64)seed);
    // resident CTAs per SM the register allocation aims at (CRL_TTT_MINB=8: 32 registers, the round-1 setting)
    static const int minb = getenv("CRL_TTT_MINB") ? atoi(getenv("CRL_TTT_MINB")) : TTT_ROLLOUT_MINB;
    return dispatch<2, 3, 4>(n, [&](auto NP) {
        return dispatch<true, false>(stats != nullptr, [&](auto STATS) {
            return dispatch<8, 6>(minb, [&](auto MINB) {
                return launch("ttt_rollout_kernel", ttt_rollout_kernel<NP, STATS, MINB>, {ttt_blocks(B), 256, 0, true},
                              stream, (uint4 *)state, (uint32_t *)result, (crl_u64 *)stats, (int)B, keys,
                              (crl_u64)first_env, step0, K);
            });
        });
    });
}

int crl_ttt_observe(const void *state, int player, int8_t *board, int8_t *winner, int8_t *mover, int64_t B, int n,
                    crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || !board || B < 0 || player >= n || player < -2) return fail(CRL_ERR_ARG, "crl_ttt_observe: bad argument");
    if (B == 0) return CRL_OK;
    return dispatch<2, 3, 4>(n, [&](auto NP) {
        return launch("ttt_observe_kernel", ttt_observe_kernel<NP>, {blocks_for(B, 256), 256}, stream,
                      (const uint4 *)state, B, player, board, winner, mover);
    });
}

int crl_ttt_pack(void *state, const int8_t *board, const int8_t *winner, const int8_t *mover, int64_t B, int n,
                 crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || !board || !winner || !mover || B < 0) return fail(CRL_ERR_ARG, "crl_ttt_pack: bad argument");
    if (B == 0) return CRL_OK;
    return launch("ttt_pack_kernel", ttt_pack_kernel, {blocks_for(B, 256), 256}, stream, (uint4 *)state, B, prm, board,
                  winner, mover);
}

/* ------------------------------------------------------------------------------------------- Blokus */

int64_t crl_blokus_state_bytes(int64_t B) { return B < 0 ? -1 : (int64_t)BLK_WORDS * 4 * B; }

int crl_blokus_reset(void *state, const uint8_t *mask, int64_t B, crl_stream_t stream) {
    if (!state || B < 0) return fail(CRL_ERR_ARG, "crl_blokus_reset: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_reset_kernel", blokus_reset_kernel, {blocks_for(B * BLK_VEC, 256), 256}, stream, (uint4 *)state,
                  mask, B);
}

int crl_blokus_legal(const void *state, int player, int32_t *counts, int32_t *action_ids, int32_t capacity,
                     int64_t *stats, int64_t B, int flags, crl_stream_t stream) {
    if (!state || !counts || !action_ids || capacity <= 0 || B < 0 || player > 3)
        return fail(CRL_ERR_ARG, "crl_blokus_legal: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_legal_kernel", blokus_legal_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream,
                  (const uint4 *)state, counts, action_ids, (int)capacity, (crl_u64 *)stats, B, player, flags);
}

int crl_blokus_is_valid(const void *state, int player, const int32_t *actions, uint8_t *valid, int64_t B, int flags,
                        crl_stream_t stream) {
    if (!state || !actions || !valid || B < 0 || player > 3) return fail(CRL_ERR_ARG, "crl_blokus_is_valid: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_is_valid_kernel", blokus_is_valid_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream,
                  (const uint4 *)state, actions, valid, B, player, flags);
}

int crl_blokus_step(const void *state_in, void *state_out, const int32_t *actions, uint8_t *result, int64_t *stats,
                    int64_t B, int flags, crl_stream_t stream) {
    if (!state_in || !state_out || !actions || !result || B < 0) return fail(CRL_ERR_ARG, "crl_blokus_step: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_step_kernel", blokus_step_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream,
                  (const uint4 *)state_in, (uint4 *)state_out, actions, (uint2 *)result, (crl_u64 *)stats, B, flags);
}

int crl_blokus_policy_random(const int32_t *counts, const int32_t *action_ids, int32_t capacity, int32_t *actions,
                             uint64_t seed, uint64_t first_env, uint32_t step, int64_t B, crl_stream_t stream) {
    if (!counts || !action_ids || !actions || capacity <= 0 || B < 0) return fail(CRL_ERR_ARG, "crl_blokus_policy_random: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_policy_random_kernel", blokus_policy_random_kernel, {blocks_for(B, 256), 256}, stream, counts,
                  action_ids, (int)capacity, actions, B, (crl_u64)seed, (crl_u64)first_env, step);
}

int crl_blokus_rollout(void *state, uint8_t *result, int64_t *stats, uint64_t seed, uint64_t first_env, uint32_t step0,
                       int K, int64_t B, crl_stream_t stream) {
    if (!state) return fail(CRL_ERR_ARG, "crl_blokus_rollout: null state");
    if (B < 0) return fail(CRL_ERR_ARG, "crl_blokus_rollout: negative batch");
    if (K < 0) return fail(CRL_ERR_ARG, "crl_blokus_rollout: negative step count K");
    if (B == 0 || K == 0) return CRL_OK;
    return launch("blokus_rollout_kernel", blokus_rollout_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream,
                  (uint4 *)state, (uint2 *)result, (crl_u64 *)stats, B, (crl_u64)seed, (crl_u64)first_env, step0, K);
}

int crl_blokus_pick(const int32_t *counts, const int32_t *action_ids, int32_t capacity, const int32_t *choice,
                    int32_t *actions, int64_t B, crl_stream_t stream) {
    if (!counts || !action_ids || !choice || !actions || capacity <= 0 || B < 0) return fail(CRL_ERR_ARG, "crl_blokus_pick: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_pick_kernel", blokus_pick_kernel, {blocks_for(B, 256), 256}, stream, counts, action_ids,
                  (int)capacity, choice, actions, B);
}

int crl_blokus_observe(const void *state, int player, int8_t *board, uint8_t *pieces, int32_t *score, int32_t *meta,
                       int64_t B, crl_stream_t stream) {
    if (!state || !board || !pieces || !score || B < 0 || player > 3 || player < -2) return fail(CRL_ERR_ARG, "crl_blokus_observe: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_observe_kernel", blokus_observe_kernel, {blocks_for(B, BLK_OBS_WARPS), 32 * BLK_OBS_WARPS},
                  stream, (const uint4 *)state, B, player, board, pieces, score, meta);
}

int crl_blokus_pack(void *state, const int8_t *board, const uint8_t *pieces, const int32_t *score, const int32_t *meta,
                    int64_t B, crl_stream_t stream) {
    if (!state || !board || !pieces || !score || !meta || B < 0) return fail(CRL_ERR_ARG, "crl_blokus_pack: bad argument");
    if (B == 0) return CRL_OK;
    return launch("blokus_pack_kernel", blokus_pack_kernel, {blocks_for(B * BLK_WORDS, 256), 256}, stream, (uint4 *)state,
                  B, board, pieces, score, meta);
}

/* ------------------------------------------------------------------------------------------- Tron opponents */

int crl_tron_policy_avoid(const void *state, int8_t *actions, int seat_mask, int noise_q16, uint64_t seed,
                          uint64_t first_env, uint32_t step, int64_t B, int N, int P, int flags, int ring_offset,
                          const int32_t *spawn_offsets, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state || !actions) return fail(CRL_ERR_ARG, "crl_tron_policy_avoid: null pointer");
    if ((rc = tron_avoid_args("crl_tron_policy_avoid", s, seat_mask, noise_q16, ring_offset, spawn_offsets))) return rc;
    if (B == 0) return CRL_OK;
    if (s.wide) {
        if ((uintptr_t)actions & 7) return fail(CRL_ERR_ARG, "crl_tron_policy_avoid: actions must be 8-byte aligned for wide shapes");
        return launch("tronw_policy_avoid_kernel", tronw_policy_avoid_kernel, {blocks_for(B, 128), 128}, stream,
                      (const uint32_t *)state, actions, B, s.wp, (uint32_t)seat_mask, (uint32_t)noise_q16, (crl_u64)seed,
                      (crl_u64)first_env, step, flags);
    }
    if ((uintptr_t)state & 15) return fail(CRL_ERR_ARG, "crl_tron_policy_avoid: state must be 16-byte aligned");
    if ((uintptr_t)actions & 3) return fail(CRL_ERR_ARG, "crl_tron_policy_avoid: actions must be 4-byte aligned");
    return launch("tron_policy_avoid_kernel", tron_policy_avoid_kernel<64>, {blocks_for(B, 64), 64}, stream,
                  (const uint4 *)state, (uint32_t *)actions, B, s.prm, (uint32_t)seat_mask, (uint32_t)noise_q16,
                  (crl_u64)seed, (crl_u64)first_env, step, flags);
}

int crl_tron_rollout_avoid(void *state, uint8_t *result, int64_t *stats, uint64_t seed, uint64_t first_env,
                           uint32_t step0, int K, int64_t B, int N, int P, int avoid_mask, int noise_q16, int ring_offset,
                           const int32_t *spawn_offsets, crl_stream_t stream) {
    TronShape s;
    int rc = tron_shape(N, P, B, s);
    if (rc) return rc;
    if (!state) return fail(CRL_ERR_ARG, "crl_tron_rollout_avoid: null state");
    if (K < 0) return fail(CRL_ERR_ARG, "crl_tron_rollout_avoid: negative step count K");
    if ((rc = tron_avoid_args("crl_tron_rollout_avoid", s, avoid_mask, noise_q16, ring_offset, spawn_offsets))) return rc;
    if (B == 0 || K == 0) return CRL_OK;
    if (!s.wide && ((uintptr_t)state & 15)) return fail(CRL_ERR_ARG, "crl_tron_rollout_avoid: state must be 16-byte aligned");
    return tron_rollout_launch(s, state, result, stats, seed, first_env, step0, K, B, avoid_mask, noise_q16, stream);
}

/* ------------------------------------------------------------------------------------------- one learner */

int crl_ttt_advance(void *state, const int8_t *actions, int seat, uint8_t *result, uint32_t *valid_after, int64_t *stats,
                    uint64_t seed, uint64_t first_env, uint32_t step, int64_t B, int n, crl_stream_t stream) {
    TTTParams prm;
    int rc = ttt_params(n, prm);
    if (rc) return rc;
    if (!state || !result) return fail(CRL_ERR_ARG, "crl_ttt_advance: null state or result");
    if (B < 0) return fail(CRL_ERR_ARG, "crl_ttt_advance: negative batch");
    if (seat < 0 || seat >= n) return fail(CRL_ERR_ARG, "crl_ttt_advance: seat must satisfy 0 <= seat < n");
    if (B == 0) return CRL_OK;
    if (B >= (int64_t)1 << 31) return fail(CRL_ERR_UNSUPPORTED, "crl_ttt_advance: batch too large for one launch");
    if ((uintptr_t)state & 15) return fail(CRL_ERR_ARG, "crl_ttt_advance: state must be 16-byte aligned");
    if (((uintptr_t)result | (uintptr_t)valid_after) & 3)
        return fail(CRL_ERR_ARG, "crl_ttt_advance: result and valid_after must be 4-byte aligned");
    return dispatch<2, 3, 4>(n, [&](auto NP) {
        return dispatch<true, false>(stats != nullptr, [&](auto STATS) {
            return launch("ttt_advance_kernel", ttt_advance_kernel<NP, STATS>, {ttt_blocks(B), 256}, stream,
                          (uint4 *)state, actions, seat, (uint32_t *)result, valid_after, (crl_u64 *)stats, (int)B,
                          (crl_u64)seed, (crl_u64)first_env, step);
        });
    });
}

int crl_blokus_advance(void *state, const int32_t *actions, int seat, uint8_t *result, int64_t *stats, uint64_t seed,
                       uint64_t first_env, uint32_t step, int64_t B, crl_stream_t stream) {
    if (!state || !result) return fail(CRL_ERR_ARG, "crl_blokus_advance: null state or result");
    if (B < 0) return fail(CRL_ERR_ARG, "crl_blokus_advance: negative batch");
    if (seat < 0 || seat > 3) return fail(CRL_ERR_ARG, "crl_blokus_advance: seat must satisfy 0 <= seat < 4");
    if (B == 0) return CRL_OK;
    if ((uintptr_t)state & 15) return fail(CRL_ERR_ARG, "crl_blokus_advance: state must be 16-byte aligned");
    if ((uintptr_t)result & 7) return fail(CRL_ERR_ARG, "crl_blokus_advance: result must be 8-byte aligned");
    if ((uintptr_t)actions & 3) return fail(CRL_ERR_ARG, "crl_blokus_advance: actions must be 4-byte aligned");
    return launch("blokus_advance_kernel", blokus_advance_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream,
                  (uint4 *)state, actions, seat, (uint2 *)result, (crl_u64 *)stats, B, (crl_u64)seed, (crl_u64)first_env,
                  step);
}

}  // extern "C"

/* ------------------------------------------------------------------------------------------- Blokus placements */

extern "C" {

int crl_blokus_placement_mask(const void *state, int player, int frame, uint32_t *mask, int32_t *counts, int64_t B,
                              int flags, crl_stream_t stream) {
    if (!state || !mask || B < 0 || player > 3) return fail(CRL_ERR_ARG, "crl_blokus_placement_mask: bad argument");
    if (frame != 0 && frame != 1) return fail(CRL_ERR_ARG, "crl_blokus_placement_mask: frame must be 0 or 1");
    if (B == 0) return CRL_OK;
    if (((uintptr_t)state | (uintptr_t)mask) & 15)
        return fail(CRL_ERR_ARG, "crl_blokus_placement_mask: state and mask must be 16-byte aligned");
    if ((uintptr_t)counts & 3) return fail(CRL_ERR_ARG, "crl_blokus_placement_mask: counts must be 4-byte aligned");
    return launch("blokus_placement_mask_kernel", blokus_placement_mask_kernel, {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS},
                  stream, (const uint4 *)state, (uint4 *)mask, counts, B, player, frame, flags);
}

int crl_blokus_placement_to_action(const void *state, int player, int frame, const int32_t *placements, int32_t *actions,
                                   int64_t B, int flags, crl_stream_t stream) {
    if (!state || !placements || !actions || B < 0 || player > 3)
        return fail(CRL_ERR_ARG, "crl_blokus_placement_to_action: bad argument");
    if (frame != 0 && frame != 1) return fail(CRL_ERR_ARG, "crl_blokus_placement_to_action: frame must be 0 or 1");
    if (B == 0) return CRL_OK;
    if ((uintptr_t)state & 15) return fail(CRL_ERR_ARG, "crl_blokus_placement_to_action: state must be 16-byte aligned");
    if (((uintptr_t)placements | (uintptr_t)actions) & 3)
        return fail(CRL_ERR_ARG, "crl_blokus_placement_to_action: placements and actions must be 4-byte aligned");
    static const BlkRotTab rot = [] {
        BlkRotTab t = {};
        for (int q = 0; q < 4; q++)
            for (int s = 0; s < BLK_NSHAPE; s++) t.img[q][s] = (uint8_t)BLK_HOST_SHAPE_ROT[s][q];
        return t;
    }();
    return launch("blokus_placement_to_action_kernel", blokus_placement_to_action_kernel,
                  {blocks_for(B, BLK_WARPS), 32 * BLK_WARPS}, stream, (const uint4 *)state, placements, actions, B, player,
                  frame, flags, rot);
}

int crl_blokus_shape_table(int32_t *shape_piece, int32_t *shape_cells, int32_t *shape_rotation, int32_t *action_shape) {
    for (int s = 0; s < BLK_NSHAPE; s++) {
        if (shape_piece) shape_piece[s] = BLK_HOST_SHAPE_PIECE[s];
        for (int i = 0; i < 10; i++)
            if (shape_cells) shape_cells[10 * s + i] = BLK_HOST_SHAPE_CELLS[s][i >> 1][i & 1];
        for (int q = 0; q < 4; q++)
            if (shape_rotation) shape_rotation[4 * s + q] = BLK_HOST_SHAPE_ROT[s][q];
    }
    for (int i = 0; i < BLK_NPIECE * 40 * 3; i++)
        if (action_shape) action_shape[i] = (&BLK_HOST_ACTION_SHAPE[0][0][0])[i];
    return BLK_NSHAPE;
}

}  // extern "C"
