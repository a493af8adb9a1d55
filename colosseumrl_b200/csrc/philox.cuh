// Philox4x32-10 (Random123), counter = (env_lo, env_hi, step, tag), key = (seed_lo, seed_hi).
// Bit-identical to colosseumrl_b200/philox.py (host) -- see SURVEY.md section 8d for the known answers.
#pragma once
#include "crl_common.cuh"

#define CRL_TAG_TRON 1u
#define CRL_TAG_BLOKUS 2u
#define CRL_TAG_TTT 3u
#define CRL_TAG_TRON_AVOID 4u       // Tron avoid policy: seats 0..3 use tag 4, seats 4..7 tag 5
#define CRL_TAG_OPPONENT 6u         // TTT / Blokus random opponents of crl_*_advance: moves 0..3 use tag 6, 4..7 tag 7

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1;
        c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// The ten round keys (k + r * Weyl), expanded once on the host and passed to a kernel BY VALUE: they then sit in the
// constant bank and feed the round's XOR as a constant operand.  (With the seed as a plain argument the compiler
// recomputes the 18 key increments per thread and per call on the ALU pipe.)
struct PhiloxKeys {
    uint32_t k0[10], k1[10];
};
static inline PhiloxKeys philox_expand_keys(crl_u64 seed) {
    PhiloxKeys k;
    uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; r++) { k.k0[r] = a; k.k1[r] = b; a += 0x9E3779B9u; b += 0xBB67AE85u; }
    return k;
}
// word 0 only of philox4x32_10 (the policies use r.x): the last round needs just hi(M1 * c2)
__device__ __forceinline__ uint32_t philox4x32_10_x(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys &k) {
#pragma unroll
    for (int r = 0; r < 9; r++) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k.k0[r]; c1 = l1;
        c2 = h0 ^ c3 ^ k.k1[r]; c3 = l0;
    }
    return __umulhi(0xCD9E8D57u, c2) ^ c1 ^ k.k0[9];
}

__device__ __forceinline__ uint4 env_words(crl_u64 seed, crl_u64 env, uint32_t step, uint32_t tag) {
    return philox4x32_10((uint32_t)env, (uint32_t)(env >> 32), step, tag, (uint32_t)seed, (uint32_t)(seed >> 32));
}

__global__ void philox_words_kernel(uint4 *out, crl_u64 seed, crl_u64 first_env, uint32_t step, uint32_t tag, long long B) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < B) out[e] = env_words(seed, first_env + (crl_u64)e, step, tag);
}
