// Shared device/host helpers for libdvae_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dvae_b200.h"

namespace dvae {

// ----------------------------------------------------------------------------- packed FP32 pairs (sm_100: FFMA2 / FMUL2 / FADD2)
// Two FP32 lanes per issue slot; a pair lives in an aligned 64-bit register pair, so packing adjacent registers is free.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 bf16x2_to_f32x2(uint32_t x) { return pk2(__uint_as_float(x << 16), __uint_as_float(x & 0xffff0000u)); }

// ----------------------------------------------------------------------------- "VsT word": two variances in 32 bits
// The sampler's emission (vst.cu) stores the variances of bins 2j, 2j+1 as one word w: the low half is bf16(v_2j) (round to
// nearest) and the WHOLE word, read as FP32, is the number nearest to v_2j+1 among those with that low half (the same 2^-9
// relative precision as a BF16 rounding).  Reading costs one shift for the even bin and nothing for the odd one.
__device__ __forceinline__ float vst_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float vst_hi(uint32_t w) { return __uint_as_float(w); }
__device__ __forceinline__ uint32_t vst_word(float lo, float hi) {      // positive finite inputs; integer pipe only (4 instructions)
    const uint32_t t = __float_as_uint(lo) + 0x8000u;                    // bf16(lo), round half up, in the upper half
    const uint32_t u = __float_as_uint(hi) + 0x8000u - (t >> 16);
    return __byte_perm(t, u, 0x7632);                                    // {t[31:16] -> low half, u[31:16] -> high half}
}


// ----------------------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
int  check_launch(const char* what);          // returns 0 or the cudaError_t of the launch

#define DVAE_REQUIRE(cond, ...)                                  \
    do {                                                         \
        if (!(cond)) {                                           \
            dvae::set_error(__VA_ARGS__);                        \
            return DVAE_ERR_ARG;                                 \
        }                                                        \
    } while (0)

// ----------------------------------------------------------------------------- small device utilities
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum `v` over the whole block; result valid in every thread. `scratch` holds >= 32 floats.
__device__ __forceinline__ float block_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    float r = 0.f;
    for (int i = 0; i < nw; ++i) r += scratch[i];   // fixed order: deterministic
    return r;
}

// ----------------------------------------------------------------------------- Philox-4x32-10
// Counter-based generator (Salmon et al., SC'11). One call yields four 32-bit words. Draws are addressed as
//   key     = (seed_lo, seed_hi)
//   counter = (utterance id, frame | chain << 20, global Metropolis-Hastings iteration, block)
// so a draw does not depend on how utterances are sharded over GPUs or tiled over CTAs (SURVEY §7.3 item 8).
struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                           uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    return Philox4{c0, c1, c2, c3};
}

// Uniform in (0, 1] from 24 random bits k: (k + 0.5) 2^-24 rounded to FP32.  Never 0.  For k >= 2^23 the sum k + 0.5 is a tie
// between two FP32 neighbours and rounds to the even one, so the upper half sits on the 2^-23 grid and k = 2^24 - 1 gives
// exactly 1.0 (one word in 2^24).  In box_muller, u1 = 1 gives a radius near 0 and u2 = 1 the angle fl(pi).
__device__ __forceinline__ float u01(uint32_t r) { return ((float)(r >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// Box-Muller on two words -> two standard normals. Uses the MUFU approximations on purpose: the FP32 and the
// tensor-core Metropolis-Hastings kernels share this function, so both consume bit-identical draws.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
    const float u1 = u01(a), u2 = u01(b);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    __sincosf(6.283185307179586f * u2 - 3.141592653589793f, &s, &c);   // argument in [-pi, pi): best MUFU accuracy
    n0 = -r * c;                                                       // cos(t) = -cos(t - pi)
    n1 = -r * s;
}

// The accept uniform of an iteration: 24 bits collected from the LOW bytes of the first three words of Philox block 0.  The
// normals of that block are built from the upper 24 bits of the same words (u01 / box_muller), so the uniform is independent of
// them and costs no Philox evaluation of its own (inside the tensor-core sampler a block is ~150 instructions per chain).  Same
// rounding as u01: in (0, 1], and exactly 1.0 when the 24 bits are all ones.
__device__ __forceinline__ float u01_low_bytes(const Philox4& r) {
    const uint32_t v = (r.x & 255u) | ((r.y & 255u) << 8) | ((r.z & 255u) << 16);
    return ((float)v + 0.5f) * (1.0f / 16777216.0f);
}

// Draws for one (frame, chain, iteration): L normals (L <= DVAE_MAX_L) and one uniform.
// Block b of the counter yields normals 4b..4b+3; the uniform comes from the low bytes of block 0 (u01_low_bytes).
__device__ __forceinline__ void mh_draws(uint32_t seed_lo, uint32_t seed_hi, uint32_t utt, uint32_t frame_chain,
                                         uint32_t iter, int L, float* eps, float& u) {
    const int nb = (L + 3) >> 2;
    for (int b = 0; b < nb; ++b) {
        const Philox4 r = philox4x32_10(utt, frame_chain, iter, (uint32_t)b, seed_lo, seed_hi);
        if (b == 0) u = u01_low_bytes(r);
        float n0, n1, n2, n3;
        box_muller(r.x, r.y, n0, n1);
        box_muller(r.z, r.w, n2, n3);
        const int j = 4 * b;
        if (j + 0 < L) eps[j + 0] = n0;
        if (j + 1 < L) eps[j + 1] = n1;
        if (j + 2 < L) eps[j + 2] = n2;
        if (j + 3 < L) eps[j + 3] = n3;
    }
}

// Philox-4x32-10 with the ten round keys precomputed on the host (rk[2r], rk[2r+1]): inside a kernel they are read straight
// from the parameter bank, so the key schedule costs no instructions.  Same function as philox4x32_10(.., rk[0], rk[1]).
struct PhiloxKeys { uint32_t rk[20]; };
inline PhiloxKeys philox_keys(uint32_t k0, uint32_t k1) {
    PhiloxKeys k;
    for (int r = 0; r < 10; ++r) { k.rk[2 * r] = k0 + 0x9E3779B9u * (uint32_t)r; k.rk[2 * r + 1] = k1 + 0xBB67AE85u * (uint32_t)r; }
    return k;
}
__device__ __forceinline__ Philox4 philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys& k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k.rk[2 * r], n1 = lo1, n2 = hi0 ^ c3 ^ k.rk[2 * r + 1], n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    }
    return Philox4{c0, c1, c2, c3};
}

}  // namespace dvae
