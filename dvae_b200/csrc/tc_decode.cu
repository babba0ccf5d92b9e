// tcgen05 (5th-gen tensor core) decoder support: operand packing and the generic kept-sample decode.
//
// Replaces packages/models/mcem.py:280-290 (compute_Vs) on top of packages/models/models.py:119-122 (Decoder.forward),
// in BF16 x BF16 -> FP32 on the tensor cores, for arbitrary row counts (the E-step itself uses the sampler's own
// emission, mh_tc2.cu, and the final filter the pipelined decode of decode_stats_tc.cu).
//
// One CTA owns a tile of 128 rows: all decoder weights sit in shared memory as UMMA operands (K-major, 128-byte
// swizzle), the activations of the tile go registers -> shared memory (A operand) -> tcgen05.mma -> TMEM -> registers.
//
//   layer 1   [128 x K1] x [K1 x 128]   K1 = 64*nkb1: columns = [bf16 hi(z) | bf16 lo(z) | y hi,lo ... | 1 | 0..];
//                                        the hi/lo split keeps the random-walk step (0.1 sigma) resolved, the
//                                        constant-one column carries the bias.
//   layer 2   [128 x 128] x [128 x 128] (absent for single-hidden-layer decoders)
//   layer 3   [128 x 128] x [128 x 528] issued as 4 chunks of N=128 + one of N=16 (bin 512), double-buffered in
//                                        TMEM so the epilogue of chunk j overlaps the MMA of chunk j+1.
//   W3, b3 are pre-scaled by log2(e): Vs = 2^(acc + b3').
//
// Threads: 8 epilogue warps (warp w reads TMEM lanes 32*(w%4).., columns half w/4) + 1 control warp whose lane 0
// issues every tcgen05.mma and whose 32 lanes allocate / free the 512 TMEM columns.
#include "tc_common.cuh"

namespace dvae {
namespace tc {

// ----------------------------------------------------------------------------- packing kernels
__global__ void pack_decoder_kernel(Dims d, const float* __restrict__ wt0, const float* __restrict__ b0,
                                    const float* __restrict__ wt1, const float* __restrict__ b1,
                                    const float* __restrict__ wt2, const float* __restrict__ b2,
                                    unsigned char* __restrict__ image) {
    // wt0: [L+y][128], wt1: [128][128] (two hidden layers only), wt2 = reconstruction: [128][F]
    const int K1 = 64 * d.nkb1;
    const int n1 = HID * K1, n2 = (d.n_hidden == 2) ? HID * HID : 0, n3 = NPAD * HID;
    const int nb = (d.n_hidden == 2 ? HID : 0) + NPAD;
    const int total = n1 + n2 + n3 + nb;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        if (i < n1) {
            const int n = i / K1, k = i % K1;
            float v = 0.f;
            if (k < d.L) v = wt0[k * HID + n];
            else if (k < 2 * d.L) v = wt0[(k - d.L) * HID + n];
            else if (k < 2 * d.L + 2 * d.y_dim) v = wt0[(d.L + (k - 2 * d.L) / 2) * HID + n];
            else if (k == 2 * d.L + 2 * d.y_dim) v = b0[n];
            *reinterpret_cast<__nv_bfloat16*>(image + sw128_offset(HID, n, k)) = __float2bfloat16_rn(v);
        } else if (i < n1 + n2) {
            const int j = i - n1, n = j / HID, k = j % HID;
            *reinterpret_cast<__nv_bfloat16*>(image + d.off_w2 + sw128_offset(HID, n, k)) = __float2bfloat16_rn(wt1[k * HID + n]);
        } else if (i < n1 + n2 + n3) {
            const int j = i - n1 - n2, n = j / HID, k = j % HID;
            const float v = (n < d.F) ? wt2[k * d.F + n] * kLog2e : 0.f;
            *reinterpret_cast<__nv_bfloat16*>(image + d.off_w3 + sw128_offset(NPAD, n, k)) = __float2bfloat16_rn(v);
        } else {
            const int j = i - n1 - n2 - n3;
            float* bias = reinterpret_cast<float*>(image + d.off_bias);
            if (d.n_hidden == 2 && j < HID) bias[j] = b1[j];
            else {
                const int n = j - (d.n_hidden == 2 ? HID : 0);
                bias[j] = (n < d.F) ? b2[n] * kLog2e : 0.f;
            }
        }
    }
}

// P, Vb [NT][ld] (frame-major FP32) -> dst [tile][quad][128 rows] of uint4 {w0, w1, w2, w3}, one 32-bit word per bin:
//
//   low  half of w_j : bf16(Vb'_j)                     (round to nearest even)
//   whole word   w_j : the FP32 number nearest to P'_j among those with that low half (same 2^-9 relative precision
//                      as a bf16 rounding, but the sampler reads P' with NO unpack instruction and Vb' with one shift)
//
// with the layer-3 bias folded into the stream, P'_j = P_j 2^-c_j and Vb'_j = Vb_j 2^-c_j (c = bias in the log2
// domain): Vx = 2^c (g 2^v + Vb'), so P / Vx = P' / (g 2^v + Vb') and log Vx differs from log(g 2^v + Vb') by a
// per-bin constant that cancels in l(z) - l(z').  Bins 0,1 of a quad additionally carry the quad scale k = 2^15 on
// Vb' and bins 2,3 carry 1/k on P' (see loglik16_pv), which saves the explicit scaling multiply.
__device__ __forceinline__ uint32_t bf16_bits_rn(float x) {
    const uint32_t b = __float_as_uint(x);
    return (b + 0x7fffu + ((b >> 16) & 1u)) >> 16;
}
__device__ __forceinline__ uint32_t word_with_low_half(float p, uint32_t low16) {
    long long d = (long long)__float_as_uint(p) - (long long)low16 + 0x8000ll;       // positive floats order like their bits
    if (d < 0) d = 0;
    uint32_t w = ((uint32_t)(d >> 16) << 16) | low16;
    if ((w & 0x7f800000u) == 0x7f800000u) w -= 0x10000u;                               // never Inf / NaN
    return w;
}
// Range of the quad trick (loglik16_pv): the product k^2 X0 X1 X2 X3 of a quad must stay inside FP32.  k = 2^(-2c) centres it on
// the frame's level 2^c, which leaves +-31 octaves per factor.  Two things would still leave that range and are handled HERE, in
// the stream, so that the sampler's inner loop carries no check:
//  * a bin whose noise variance the NMF has driven far below the frame's level while the speech term g 2^v is tiny as well
//    (spectral nulls; noise-only frames where the gain g collapses): Vb' is floored 30 octaves (90 dB) below the frame's level.
//    Both l(z) and l(z') see the same floor, the bin carries no energy, the accept decision is unaffected;
//  * the padding bins 513 .. 543 (no observation, P' = 0): X would be g alone, and g^3 or g^4 underflows once the gain of a frame
//    has collapsed (the first version did exactly that after ~100 EM iterations on noise-only frames: l(z') = NaN).  They carry
//    Vb' = 1 in the quad's own scale (pv_pad_word), i.e. the constant factor 1 + g 2^0.
__device__ __forceinline__ uint32_t pv_word(float p, float vb, float bias_log2, int j, float k) {
    const float sc = exp2f(-bias_log2);
    const float level = rsqrtf(k);                                   // 2^c
    const float pj = p * sc * (j < 2 ? 1.0f : 1.0f / k);
    const float vf = fmaxf(vb * sc, level * 9.313225746e-10f);       // 2^-30 below the frame's level
    const float vj = vf * (j < 2 ? k : 1.0f);
    return word_with_low_half(pj, bf16_bits_rn(vj));
}
// a padding bin of quad position j: k Vb' = level^-1 (j < 2) or Vb' = level (j >= 2), so that the quad's product sees a factor
// of the same size as its real bins; P' = 0
__device__ __forceinline__ uint32_t pv_pad_word(int j, float k) {
    const float level = rsqrtf(k);
    return word_with_low_half(0.f, bf16_bits_rn(j < 2 ? k * level : level));
}

// generic version: one thread per (tile, quad, row), rows fastest (coalesced stores, strided loads)
__global__ void pack_pv_kernel(const float* __restrict__ P, const float* __restrict__ Vb, const float* __restrict__ bias_log2,
                               const float* __restrict__ kscale, int64_t chains, int C, int F, int ld, uint4* __restrict__ dst) {
    const int64_t n_tiles = (chains + TM - 1) / TM;
    const int64_t total = n_tiles * NQ * TM;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i % TM);
        const int q = (int)((i / TM) % NQ);
        const int64_t tile = i / ((int64_t)TM * NQ);
        const int64_t m = tile * TM + r;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (m < chains) {
            const int64_t fr = m / C;
            const int f = 4 * q;
            const float k = kscale ? kscale[fr] : kDefaultQuadScale;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                w[j] = (f + j < F) ? pv_word(P[fr * ld + f + j], Vb[fr * ld + f + j], bias_log2[f + j], j, k) : pv_pad_word(j, k);
        }
        dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// ld % 4 == 0: a CTA packs 8 quads x 128 rows of one tile through shared memory, so that both sides are coalesced: the
// loads run along the bins of a frame (8 quads = 128 contiguous bytes of P and of Vb), the stores along the rows of a quad
// (2 KB contiguous).  The padded row stride (129) keeps both shared-memory passes conflict-free.
constexpr int PPV_Q = 8;
__global__ void __launch_bounds__(256) pack_pv_tiled_kernel(const float* __restrict__ P, const float* __restrict__ Vb,
                                                            const float* __restrict__ bias_log2, const float* __restrict__ kscale,
                                                            int64_t chains, int C, int F, int ld, uint4* __restrict__ dst) {
    __shared__ uint4 sm[PPV_Q * (TM + 1)];
    const int64_t tile = blockIdx.y;
    const int q0 = blockIdx.x * PPV_Q;
#pragma unroll
    for (int k = 0; k < PPV_Q * TM / 256; ++k) {
        const int e = threadIdx.x + 256 * k;
        const int row = e / PPV_Q, ql = e % PPV_Q, q = q0 + ql;
        const int64_t m = tile * TM + row;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (m < chains && q < NQ) {
            const int64_t fr = m / C;
            const int f = 4 * q;
            const float k = kscale ? __ldg(kscale + fr) : kDefaultQuadScale;
            if (f < F) {
                const float4 p4 = __ldg(reinterpret_cast<const float4*>(P + fr * ld + f));
                const float4 v4 = __ldg(reinterpret_cast<const float4*>(Vb + fr * ld + f));
                const float4 b4 = *reinterpret_cast<const float4*>(bias_log2 + f);
                w[0] = pv_word(p4.x, v4.x, b4.x, 0, k);
                w[1] = (f + 1 < F) ? pv_word(p4.y, v4.y, b4.y, 1, k) : pv_pad_word(1, k);
                w[2] = (f + 2 < F) ? pv_word(p4.z, v4.z, b4.z, 2, k) : pv_pad_word(2, k);
                w[3] = (f + 3 < F) ? pv_word(p4.w, v4.w, b4.w, 3, k) : pv_pad_word(3, k);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) w[j] = pv_pad_word(j, k);
            }
        }
        sm[ql * (TM + 1) + row] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < PPV_Q * TM / 256; ++k) {
        const int e = threadIdx.x + 256 * k;
        const int ql = e / TM, row = e % TM, q = q0 + ql;
        if (q < NQ) dst[(tile * NQ + q) * TM + row] = sm[ql * (TM + 1) + row];
    }
}

// Per-frame quad scale of the sampler's likelihood (loglik16_pv): k = 2^(-2 c) with the frame's level 2^c = 2^-16 x the loudest
// bin of the frame's bias-free spectrum P 2^-b.  The quad product k^2 X0 X1 X2 X3 of X = Vx 2^-b then has 2^15.75 of headroom per
// factor above the loudest observation (a model that overshoots it by more than 55 000 x is rejected as Inf) and, with the Vb'
// floor of pack_pv 30 octaves below the level, 138 dB of range below it.  (The first version centred on the MEAN of log2 P: a
// frame with one loud partial over a quiet floor - geometric mean near the floor - overflowed.)  P does not change during a run,
// so this runs once per batch.  One warp per frame: deterministic and independent of the batch a frame sits in.  Frames without
// energy keep the default 2^15; c is clamped to +-30 so that P' / k stays a normal number.
__global__ void row_scale_kernel(const float* __restrict__ P, const float* __restrict__ bias_log2, int64_t NT, int F, int ld,
                                 float* __restrict__ kscale) {
    const int64_t n = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (n >= NT) return;
    float top = -1e30f;
    for (int f = lane; f < F; f += 32) {
        const float p = P[n * ld + f];
        if (p > 0.f) top = fmaxf(top, log2f(p) - bias_log2[f]);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) top = fmaxf(top, __shfl_xor_sync(0xffffffffu, top, o));
    if (lane == 0) {
        float k = kDefaultQuadScale;
        if (top > -1e29f) {
            const float c = fminf(fmaxf(rintf(top) - 16.0f, -30.f), 30.f);
            k = exp2f(-2.0f * c);
        }
        kscale[n] = k;
    }
}

// ----------------------------------------------------------------------------- kernel
struct Params {
    Dims d;
    const unsigned char* image;
    int64_t rows;                 // rows of Zin
    int C;                        // label row divisor: row r uses y[r / C]
    const float* y;               // [rows / C][y_dim] or null
    const float* ybias;           // [rows / C][128] per-frame layer-1 bias or null
    const float* Zin;             // [rows][L]
    float* Vs;                    // [rows][ld]
    int ld;
    int* status;
};

__global__ void __launch_bounds__(NTHREADS, 1) decoder_tc_kernel(Params p) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ uint64_t bars[3];
    __shared__ uint32_t tmem_slot;
    __shared__ int dead_flag;

    const Dims& d = p.d;
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* A = base + ((d.image_bytes + 1023) & ~1023);
    const uint32_t bar12 = smem_u32(&bars[0]);
    const uint32_t bar3[2] = {smem_u32(&bars[1]), smem_u32(&bars[2])};
    uint32_t ph12 = 0, ph3[2] = {0, 0};
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = warp & 3, h = (warp >> 2) & 1;
    const int row = 32 * q + lane;
    const bool epi = warp < 8, owner = warp < 4, ctrl = (warp == 8 && lane == 0);

    {   // weights -> shared memory (generic proxy writes, made visible to the tensor core by the fence before S1)
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(base);
        for (int i = threadIdx.x; i < d.image_bytes / 16; i += NTHREADS) dst[i] = __ldg(src + i);
    }
    if (threadIdx.x == 0) {
        dead_flag = 0;
        mbar_init(bar12, 1);
        mbar_init(bar3[0], 1);
        mbar_init(bar3[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    volatile int* dead = &dead_flag;

    const uint32_t a_addr = smem_u32(A);
    const uint32_t w1_addr = smem_u32(base), w2_addr = smem_u32(base + d.off_w2), w3_addr = smem_u32(base + d.off_w3);
    const float* bias = reinterpret_cast<const float*>(base + d.off_bias);
    const float* b2 = (d.n_hidden == 2) ? bias : nullptr;
    const float* b3 = bias + (d.n_hidden == 2 ? HID : 0);
    const int L = d.L;
    const int64_t n_tiles = (p.rows + TM - 1) / TM;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row_g = tile * TM + row;
        const bool valid = row_g < p.rows;
        if (owner) {
            float z[DVAE_MAX_L], yrow[8];
            if (valid) {
                for (int l = 0; l < L; ++l) z[l] = p.Zin[row_g * L + l];
                for (int i = 0; i < d.y_dim; ++i) yrow[i] = p.y[(row_g / p.C) * d.y_dim + i];
            } else {
                for (int l = 0; l < L; ++l) z[l] = 0.f;
            }
            write_a1_row(d, A, row, z, yrow, valid);
        }
        fence_async_smem();
        __syncthreads();                                                            // S1

        // ---- layer 1 (bias rides on the constant-one column)
        if (ctrl) {
            tc_fence_after();
            issue_gemm2(a_addr, 16384, w1_addr, 16384, d.nkb1, tmem, HID);
            umma_commit(bar12);
        }
        if (epi) {
            mbar_wait(bar12, ph12, dead, p.status);
            tc_fence_after();
            hidden_epilogue_rows(tmem, A, q, h, row, (p.ybias && valid) ? p.ybias + (row_g / p.C) * HID : nullptr);
            fence_async_smem();
            tc_fence_before();
        }
        ph12 ^= 1;
        __syncthreads();                                                            // S2

        // ---- layer 2
        if (d.n_hidden == 2) {
            if (ctrl) {
                tc_fence_after();
                issue_gemm2(a_addr, 16384, w2_addr, 16384, 2, tmem, HID);
                umma_commit(bar12);
            }
            if (epi) {
                mbar_wait(bar12, ph12, dead, p.status);
                tc_fence_after();
                hidden_epilogue_rows(tmem, A, q, h, row, b2);
                fence_async_smem();
                tc_fence_before();
            }
            ph12 ^= 1;
            __syncthreads();                                                        // S3
        }

        // ---- layer 3 in 5 chunks, TMEM double buffer at columns 128 / 256
        if (ctrl) {
            tc_fence_after();
            issue_gemm2(a_addr, 16384, w3_addr, NPAD * 128, 2, tmem + 128, 128);
            umma_commit(bar3[0]);
            issue_gemm2(a_addr, 16384, w3_addr + 16384, NPAD * 128, 2, tmem + 256, 128);
            umma_commit(bar3[1]);
        }
        for (int j = 0; j < 5; ++j) {
            const int b = j & 1;
            if (epi) {
                mbar_wait(bar3[b], ph3[b], dead, p.status);
                tc_fence_after();
                const uint32_t tbuf = tmem + 128 + 128 * b + ((uint32_t)(32 * q) << 16);
                if (j < 4) {
                    float v[32];
#pragma unroll
                    for (int part = 0; part < 2; ++part) {
                        const int col0 = 64 * h + 32 * part;                // column inside the chunk
                        const int f0 = 128 * j + col0;                      // global bin
                        tmem_ld32(tbuf + col0, v);
                        tmem_wait_ld();
                        if (valid) {
                            float* dst = p.Vs + row_g * p.ld + f0;
#pragma unroll
                            for (int qd = 0; qd < 8; ++qd) {
                                const float4 bb = *reinterpret_cast<const float4*>(b3 + f0 + 4 * qd);
                                float4 o;
                                o.x = ex2_approx(v[4 * qd + 0] + bb.x);
                                o.y = ex2_approx(v[4 * qd + 1] + bb.y);
                                o.z = ex2_approx(v[4 * qd + 2] + bb.z);
                                o.w = ex2_approx(v[4 * qd + 3] + bb.w);
                                *reinterpret_cast<float4*>(dst + 4 * qd) = o;
                            }
                        }
                    }
                } else if (h == 0) {                                       // tail chunk: only bin 512 is real
                    float v[4];
                    tmem_ld4(tbuf, v);
                    tmem_wait_ld();
                    if (valid && d.F > 512) p.Vs[row_g * p.ld + 512] = ex2_approx(v[0] + b3[512]);
                }
                tc_fence_before();
            }
            ph3[b] ^= 1;
            __syncthreads();                                                        // S4..S8
            if (ctrl && j + 2 < 5) {
                tc_fence_after();
                const int jn = j + 2;
                issue_gemm2(a_addr, 16384, w3_addr + jn * 16384, NPAD * 128, 2, tmem + 128 + 128 * b, jn < 4 ? 128 : 16);
                umma_commit(bar3[b]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512) : "memory");
    }
}

size_t smem_bytes(const Dims& d) { return (size_t)((d.image_bytes + 1023) & ~1023) + A_BYTES + 512 + 1024; }

int check_dims(const DvaeMlp* dec, int L, int y_dim, const char* who, Dims* out) {
    DVAE_REQUIRE(dec != nullptr, "%s: null decoder", who);
    DVAE_REQUIRE(dec->n_layers == 2 || dec->n_layers == 3, "%s: the tensor-core path supports 1 or 2 hidden layers", who);
    for (int i = 1; i < dec->n_layers; ++i) DVAE_REQUIRE(dec->dims[i] == HID, "%s: hidden width must be %d", who, HID);
    const int F = dec->dims[dec->n_layers];
    DVAE_REQUIRE(F > 512 && F <= 513, "%s: the tensor-core path is specialised for F=513 bins (got %d)", who, F);
    DVAE_REQUIRE(L >= 1 && L <= DVAE_MAX_L && y_dim >= 0 && y_dim <= 8, "%s: bad L / y_dim", who);
    DVAE_REQUIRE(dec->dims[0] == L + y_dim, "%s: decoder takes %d inputs, L+y_dim=%d", who, dec->dims[0], L + y_dim);
    *out = make_dims(L, y_dim, dec->n_layers - 1, F);
    DVAE_REQUIRE(out->nkb1 <= 2, "%s: 2L+2y+1 must be <= 128", who);
    DVAE_REQUIRE(smem_bytes(*out) <= 227 * 1024, "%s: weights do not fit in shared memory", who);
    return 0;
}

}  // namespace tc
}  // namespace dvae

using namespace dvae;
using namespace dvae::tc;

extern "C" int64_t dvae_tc_image_bytes(const DvaeMlp* dec, int L, int y_dim) {
    Dims d;
    if (check_dims(dec, L, y_dim, "dvae_tc_image_bytes", &d)) return -1;
    return d.image_bytes;
}

extern "C" int dvae_tc_pack_decoder(const DvaeMlp* dec, int L, int y_dim, void* image, void* stream) {
    Dims d;
    int rc = check_dims(dec, L, y_dim, "dvae_tc_pack_decoder", &d);
    if (rc) return rc;
    DVAE_REQUIRE(image != nullptr && (reinterpret_cast<uintptr_t>(image) & 15) == 0, "dvae_tc_pack_decoder: image must be 16-byte aligned");
    const bool two = d.n_hidden == 2;
    pack_decoder_kernel<<<148, 256, 0, (cudaStream_t)stream>>>(d, dec->wt[0], dec->bias[0], two ? dec->wt[1] : nullptr,
                                                              two ? dec->bias[1] : nullptr, dec->wt[two ? 2 : 1],
                                                              dec->bias[two ? 2 : 1], (unsigned char*)image);
    return check_launch("pack_decoder_kernel");
}

// max over bins of log2(e) * sum_k |W3[k][f]|: the layer-3 pre-activation (log2 domain, bias excluded) cannot exceed it
// because the hidden activations are tanh outputs
__global__ void exponent_bound_kernel(const float* __restrict__ wt, int K, int F, float* __restrict__ out) {
    __shared__ float red[256];
    float m = 0.f;
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < K; ++k) s += fabsf(wt[k * F + f]);
        m = fmaxf(m, s);
    }
    red[threadIdx.x] = m;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = red[0] * kLog2e;
}

extern "C" int dvae_tc_decoder_exponent_bound(const DvaeMlp* dec, int L, int y_dim, float* bound_host, void* stream) {
    Dims d;
    int rc = check_dims(dec, L, y_dim, "dvae_tc_decoder_exponent_bound", &d);
    if (rc) return rc;
    DVAE_REQUIRE(bound_host, "dvae_tc_decoder_exponent_bound: null pointer");
    float* dev = nullptr;
    cudaError_t e = cudaMalloc(&dev, sizeof(float));
    if (e != cudaSuccess) { set_error("cudaMalloc: %s", cudaGetErrorString(e)); return (int)e; }
    const bool two = d.n_hidden == 2;
    cudaStream_t st = (cudaStream_t)stream;
    exponent_bound_kernel<<<1, 256, 0, st>>>(dec->wt[two ? 2 : 1], HID, d.F, dev);
    e = cudaMemcpyAsync(bound_host, dev, sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (e != cudaSuccess) { set_error("dvae_tc_decoder_exponent_bound: %s", cudaGetErrorString(e)); return (int)e; }
    return 0;
}

extern "C" int64_t dvae_tc_image_bias_offset(const DvaeMlp* dec, int L, int y_dim) {
    Dims d;
    if (check_dims(dec, L, y_dim, "dvae_tc_image_bias_offset", &d)) return -1;
    return d.off_bias + 4 * (d.n_hidden == 2 ? HID : 0);           // the layer-3 bias follows the hidden-2 bias (pack_decoder_kernel)
}

// The samplers' hidden activation (hidden_rows_bf_part) over every BF16 input: table[x] = tanh.approx.bf16x2 of pattern x
__global__ void tanh_bf16_table_kernel(uint16_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;      // one pair of patterns per thread
    if (i >= 32768u) return;
    const uint32_t y = tanh_bf16x2((2u * i) | ((2u * i + 1u) << 16));
    out[2 * i] = (uint16_t)(y & 0xffffu);
    out[2 * i + 1] = (uint16_t)(y >> 16);
}

extern "C" int dvae_tc_tanh_bf16_table(uint16_t* out, void* stream) {
    DVAE_REQUIRE(out != nullptr, "dvae_tc_tanh_bf16_table: null pointer");
    tanh_bf16_table_kernel<<<128, 256, 0, (cudaStream_t)stream>>>(out);
    return check_launch("tanh_bf16_table_kernel");
}

// The decode kernels' hidden activation (hidden_epilogue_rows, ds_hidden_row): y[i] = tanh.approx.f32(x[i]); tests only
__global__ void tanh_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y[i] = tanh_approx(x[i]);
}

extern "C" int dvae_tc_tanh_f32(const float* x, float* y, int64_t n, void* stream) {
    DVAE_REQUIRE(x && y && n >= 0, "dvae_tc_tanh_f32: bad arguments");
    if (n == 0) return 0;
    const int64_t blocks = (n + 255) / 256;
    tanh_f32_kernel<<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), 256, 0, (cudaStream_t)stream>>>(x, y, n);
    return check_launch("tanh_f32_kernel");
}

extern "C" int64_t dvae_tc_packed_pv_bytes(int64_t chains) {
    if (chains <= 0) return 0;
    return ((chains + TM - 1) / TM) * (int64_t)NQ * TM * 16;
}

extern "C" int dvae_tc_row_scale(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* P, int64_t NT, int F, int ld,
                                 float* kscale, void* stream) {
    Dims d;
    int rc = check_dims(dec, L, y_dim, "dvae_tc_row_scale", &d);
    if (rc) return rc;
    DVAE_REQUIRE(image && P && kscale && NT >= 0 && F == d.F && ld >= F, "dvae_tc_row_scale: bad arguments");
    if (NT == 0) return 0;
    const float* bias_log2 = reinterpret_cast<const float*>((const unsigned char*)image + d.off_bias) + (d.n_hidden == 2 ? HID : 0);
    row_scale_kernel<<<(unsigned)((NT + 7) / 8), 256, 0, (cudaStream_t)stream>>>(P, bias_log2, NT, F, ld, kscale);
    return check_launch("row_scale_kernel");
}

extern "C" int dvae_tc_pack_pv(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* P, const float* Vb,
                               const float* kscale, int64_t NT, int n_chains, int F, int ld, void* dst, void* stream) {
    Dims d;
    int rc = check_dims(dec, L, y_dim, "dvae_tc_pack_pv", &d);
    if (rc) return rc;
    DVAE_REQUIRE(image && P && Vb && dst && NT >= 0 && n_chains >= 1 && F == d.F && ld >= F, "dvae_tc_pack_pv: bad arguments");
    DVAE_REQUIRE((reinterpret_cast<uintptr_t>(dst) & 15) == 0, "dvae_tc_pack_pv: 16-byte alignment required");
    if (NT == 0) return 0;
    // layer-3 bias (log2 domain) inside the decoder image: after the hidden-2 bias if there is one
    const float* bias_log2 = reinterpret_cast<const float*>((const unsigned char*)image + d.off_bias) + (d.n_hidden == 2 ? HID : 0);
    const int64_t chains = NT * n_chains, n_tiles = (chains + TM - 1) / TM;
    if ((ld & 3) == 0 && ld >= ((F + 3) & ~3) && ((reinterpret_cast<uintptr_t>(P) | reinterpret_cast<uintptr_t>(Vb)) & 15) == 0 && n_tiles < 65536) {
        pack_pv_tiled_kernel<<<dim3((NQ + PPV_Q - 1) / PPV_Q, (unsigned)n_tiles), 256, 0, (cudaStream_t)stream>>>(P, Vb, bias_log2, kscale, chains,
                                                                                                                n_chains, F, ld, (uint4*)dst);
        return check_launch("pack_pv_tiled_kernel");
    }
    pack_pv_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(P, Vb, bias_log2, kscale, chains, n_chains, F, ld, (uint4*)dst);
    return check_launch("pack_pv_kernel");
}

extern "C" int dvae_decode_tc(const DvaeMlp* dec, const void* image, const float* Zs, int64_t rows, int L, const float* y,
                              int y_dim, const float* ybias, int x2_row_div, float* Vs, int ld, int* status, void* stream) {
    Params p{};
    int rc = check_dims(dec, L, y_dim, "dvae_decode_tc", &p.d);
    if (rc) return rc;
    DVAE_REQUIRE(image && Zs && Vs && status, "dvae_decode_tc: null pointer");
    DVAE_REQUIRE((y_dim == 0 || y) && x2_row_div >= 1, "dvae_decode_tc: bad label arguments");
    DVAE_REQUIRE(rows >= 0 && ld >= p.d.F && (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(Vs) & 15) == 0, "dvae_decode_tc: bad sizes / alignment");
    if (rows == 0) return 0;
    p.image = (const unsigned char*)image;
    p.rows = rows; p.C = x2_row_div < 1 ? 1 : x2_row_div; p.y = y; p.ybias = ybias;
    p.Zin = Zs; p.Vs = Vs; p.ld = ld; p.status = status;
    const size_t smem = smem_bytes(p.d);
    const int64_t n_tiles = (p.rows + TM - 1) / TM;
    const int grid = (int)(n_tiles < 148 ? n_tiles : 148);
    cudaError_t e = cudaFuncSetAttribute(decoder_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return (int)e; }
    decoder_tc_kernel<<<grid, NTHREADS, smem, (cudaStream_t)stream>>>(p);
    return check_launch("decoder_tc_kernel");
}
