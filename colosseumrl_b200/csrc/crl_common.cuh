// Common device helpers for the colosseum B200 engine (sm_100a).
#pragma once
#include <stdint.h>

#ifndef CRL_HOSTSIM
#include <cuda_runtime.h>
#include <cuda.h>            // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, no -lcuda)
// dynamic shared memory (sized at launch); the emulator gives it its maximum size statically
#define CRL_DYN_SMEM(name, maxbytes) extern __shared__ __align__(128) uint8_t name[]
// launch with the programmatic-stream-serialization attribute (PDL); the kernel must call pdl_wait() before it
// touches memory written by its predecessor in the stream.  CRL_PDL=0 in the environment launches plainly (A/B runs).
#include <stdlib.h>
static inline bool crl_use_pdl() {
    static const bool on = !(getenv("CRL_PDL") && atoi(getenv("CRL_PDL")) == 0);
    return on;
}
#else
// tests/hostsim/cuda_shim.h was included first: kernels run on the SIMT emulator (CPU unit tests only)
#define CRL_DYN_SMEM(name, maxbytes) static __attribute__((aligned(128))) uint8_t name[maxbytes]
#endif

#define CRL_NSTAT 32
#define CRL_STAT_ROWS 256  // the device statistics buffer is int64[CRL_STAT_ROWS][CRL_NSTAT]; CTAs spread their
                           // partial sums over the rows (row = blockIdx % 256) so same-address L2 atomics do not
                           // serialise; the reader sums the rows
// statistics slots (int64 each); identical to oracle/oracle_rollout.c
enum {
    ST_STEPS = 0, ST_EPISODES = 1, ST_EPLEN = 2, ST_WINS = 3 /*..6*/, ST_NOWIN = 7, ST_SCORE = 8 /*..11*/,
    ST_ERRORS = 12, ST_NVALID = 13, ST_RANK = 14 /*..17*/, ST_REWARD = 18
};

// step flags
#define CRL_FLAG_AUTO_RESET 1
#define CRL_FLAG_COMPACT_RESULT 2
#define CRL_FLAG_COMPACT2_RESULT 8
#define CRL_FLAG_PACKED_ACTIONS 4

typedef unsigned long long crl_u64;

// 128-bit streaming accesses: state is touched exactly once per step, keep it out of L1
__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
#ifndef CRL_HOSTSIM
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
#else
    return *p;
#endif
}
__device__ __forceinline__ void st_stream(uint4 *p, uint4 v) {
#ifndef CRL_HOSTSIM
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#else
    *p = v;
#endif
}

// plain 32-bit global store through a pointer whose address space the compiler can no longer infer
__device__ __forceinline__ void st_global_u32(int32_t *p, int32_t v) {
#ifndef CRL_HOSTSIM
    asm volatile("st.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
#else
    *p = v;
#endif
}

// One step of a warp-wide inclusive scan: x += (value of lane - d) if that lane exists.  shfl.sync.up returns the
// "source lane in range" predicate itself, so a step is SHFL + one predicated add (the C form `if (lane >= d)`
// compiles to SHFL + ISETP + SEL + IADD).  All 32 lanes must call.
__device__ __forceinline__ uint32_t warp_scan_step(uint32_t x, int d) {
#ifndef CRL_HOSTSIM
    asm volatile("{ .reg .pred p; .reg .u32 t;\n\t"
                 "shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n\t"
                 "@p add.u32 %0, %0, t; }" : "+r"(x) : "r"(d));
    return x;
#else
    const uint32_t t = __shfl_up_sync(0xffffffffu, x, (unsigned)d);
    return ((int)(threadIdx.x & 31) >= d) ? x + t : x;
#endif
}

// ---- bulk asynchronous copies (TMA 1-D, SASS UBLKCP) between global memory and a shared-memory tile ----------
// The SoA state layout makes every 16-byte vector of a CTA's environments one contiguous global segment, so a
// tile is moved by a handful of bulk copies issued by ONE thread; the other threads never touch the data they
// do not need.  On the SIMT emulator the same helpers are plain cooperative loops.
#ifndef CRL_HOSTSIM
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" :: "r"(smem_u32(bar)), "r"(phase) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
// 2-D tiled TMA through a tensor map (SASS UTMALDG / UTMASTG): ONE instruction moves a whole [rows][TILE*16 B] box,
// out-of-range columns are zero-filled on loads and clipped on stores
__device__ __forceinline__ void tma_load_2d(void *dst_smem, const CUtensorMap *tm, int x, int y, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(dst_smem)), "l"(tm), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *tm, int x, int y, const void *src_smem) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                 :: "l"(tm), "r"(x), "r"(y), "r"(smem_u32(src_smem)) : "memory");
}
__device__ __forceinline__ void tensormap_prefetch(const CUtensorMap *tm) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(tm) : "memory");
}
// L2 prefetch hints (no architectural effect): a 1-D range (multiple of 16 bytes, 16-byte aligned) / a 2-D tensor box
__device__ __forceinline__ void l2_prefetch_bulk(const void *src_gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void l2_prefetch_tensor_2d(const CUtensorMap *tm, int x, int y) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" :: "l"(tm), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_commit_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#endif

// per-thread L2 prefetch hint of the 128-byte line that holds *p
__device__ __forceinline__ void l2_prefetch_line(const void *p) {
#ifndef CRL_HOSTSIM
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
#endif
}

// ---- programmatic dependent launch (PDL): overlap a kernel's launch + prologue with its predecessor's tail ----
__device__ __forceinline__ void pdl_launch_dependents() {
#ifndef CRL_HOSTSIM
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
__device__ __forceinline__ void pdl_wait() {   // blocks until the predecessor grid has completed and flushed
#ifndef CRL_HOSTSIM
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}

// Episode statistics: per-thread contribution -> warp reduce (redux.sync) -> shared-memory partial per CTA
// -> one global atomic per CTA and non-zero slot.  Values are small ints; reduce in 32-bit, accumulate in 64.
// one global atomic per CTA and non-zero slot, into row (blockIdx % CRL_STAT_ROWS); call after a __syncthreads()
__device__ __forceinline__ void stats_flush_row(const int *sm, crl_u64 *g) {
    if (threadIdx.x < CRL_NSTAT && sm[threadIdx.x] != 0)
        atomicAdd(g + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT + threadIdx.x, (crl_u64)(long long)sm[threadIdx.x]);
}

// reader side: out[s] (+)= sum over the CRL_STAT_ROWS rows of rows[r][s]; one CTA of 256 threads (8 x 32 rows each)
__global__ void __launch_bounds__(256) stats_reduce_kernel(const crl_u64 *__restrict__ rows, crl_u64 *__restrict__ out,
                                                           int accumulate) {
    __shared__ crl_u64 part[8][CRL_NSTAT];
    const int slot = threadIdx.x & (CRL_NSTAT - 1), grp = threadIdx.x >> 5;
    crl_u64 s = 0;
#pragma unroll 8
    for (int r = grp * (CRL_STAT_ROWS / 8); r < (grp + 1) * (CRL_STAT_ROWS / 8); r++) s += rows[r * CRL_NSTAT + slot];
    part[grp][slot] = s;
    __syncthreads();
    if (grp == 0) {
#pragma unroll
        for (int g = 1; g < 8; g++) s += part[g][slot];
        out[slot] = accumulate ? out[slot] + s : s;
    }
}

struct BlockStats {
    int *sm;  // __shared__ int[CRL_NSTAT]
    __device__ __forceinline__ void init() const {
        if (threadIdx.x < CRL_NSTAT) sm[threadIdx.x] = 0;
        __syncthreads();
    }
    __device__ __forceinline__ void add(int slot, int v) const {
        int s = __reduce_add_sync(0xffffffffu, v);
        if ((threadIdx.x & 31) == 0 && s != 0) atomicAdd(&sm[slot], s);
    }
    __device__ __forceinline__ void flush(crl_u64 *g) const {
        __syncthreads();
        stats_flush_row(sm, g);
    }
};
