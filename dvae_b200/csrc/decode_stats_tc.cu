// Warp-specialised tcgen05 decode of the kept samples with per-frame reciprocal statistics (third decode kernel).
//
// Replaces packages/models/mcem.py:280-290 (compute_Vs) and the inner sums of mcem.py:108-110:
//
//   Vs[n][r][f] = D([Z_r(n); y(n)])[f]                         (FP32, written once, 128-byte coalesced warp stores)
//   A1[n][f]    = sum_r 1 / Vx,   A2[n][f] = sum_r 1 / Vx^2,   Vx = g[n] Vs[n][r][f] + Vb[n][f]
//
// The W update then only needs  num[f,k] = sum_n P A2 H,  den[f,k] = sum_n A1 H  (w_from_frame_stats_kernel): no per-bin
// accumulators have to live in registers across tiles, which is what allows the schedule below.
//
// Phase timing of the previous, unpipelined kernel (round 1): 26 k cycles per 120-row tile, of
// which the serial front (operand write, layers 1-2) took 10 k and each layer-3 chunk epilogue 5 k with two warps per
// scheduler.  Here the CTA is a two-stage pipeline over tiles:
//
//   front  (warps 0-3,  thread = row)      z -> layer-1 operand -> MMA -> tanh -> MMA -> tanh -> h2 in A[tile & 1]
//   back   (warps 4-19, thread = bin,      layer 3 TRANSPOSED (A = 128 bins of W3, B = h2): TMEM lanes are bins, a warp
//           warp = lane quadrant x frame)   stores 128 contiguous bytes of Vs; two chunk buffers in TMEM; W3 is streamed
//                                           from L2 chunk by chunk (cp.async.bulk) into two 32 KB slots
//
// so layers 1-2 of tile i+1 overlap layer 3 of tile i, and 4 back warps per scheduler keep MUFU / LSU busy.
// Shared memory: W1 | W2 | biases resident (51 KB) + 2 activation buffers (64 KB) + 2 W3 slots (64 KB).
// TMEM: [0,128) layers 1-2, [128,256) / [256,384) layer-3 chunks.
#include "tc_common.cuh"

namespace dvae {
namespace tc {

constexpr int DS_THREADS = 672;                       // 4 front warps + 16 back warps + 1 issue warp
constexpr int DS_BACK = 512;
// Depth of the layer-3 ring (W3 chunk slot in shared memory + accumulator buffer in TMEM per stage).  With two stages the GEMM
// of chunk c+2 could only be issued once chunk c was drained and every chunk hand-over cost the back warps ~0.5 k cycles of
// waiting; with three, it is issued one chunk earlier.
constexpr int DS_NS = 3;

struct DsParams {
    Dims d;
    const unsigned char* image;
    const float* Zs;        // [NT][R][L]
    const float* y;         // [NT][y_dim] or null
    const float* ybias;     // [NT][128] per-frame layer-1 bias or null
    const float* Vb;        // [NT][ld]
    const float* g;         // [NT]
    float* Vs;              // [NT][R][ld]
    float* A1;              // [NT][ld] (STORE)
    float* A2;              // [NT][ld] (STORE)
    float* WFs;             // [NT][ld] (!STORE) mask sums sum_r g Vs / Vx ...
    float* WFn;             // [NT][ld] (!STORE) ... and sum_r Vb / Vx
    int64_t NT;
    int ld;
    int zs_rtot, zs_r0;     // samples per frame in Zs (and Vs) and the first one this launch decodes (R of them)
    int acc;                // != 0: add to A1 / A2 (WFs / WFn) instead of overwriting (later sample windows of the same frames)
    int* status;
};

__device__ __forceinline__ void ds_bar_front() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ void ds_bar_tail() { asm volatile("bar.sync 2, 128;" ::: "memory"); }

__device__ __forceinline__ void ds_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void ds_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}

template <int RL> __device__ __forceinline__ void ds_tmem_ld(uint32_t taddr, float* v);
template <> __device__ __forceinline__ void ds_tmem_ld<32>(uint32_t taddr, float* v) { tmem_ld32(taddr, v); }
template <> __device__ __forceinline__ void ds_tmem_ld<16>(uint32_t taddr, float* v) { tmem_ld16(taddr, v); }

// front epilogue: the thread's row, all 128 hidden units: D12[row][0..128) -> tanh(+bias) -> bf16 -> activation operand
__device__ __forceinline__ void ds_hidden_row(uint32_t tmem, unsigned char* A, int q, int row, const float* bias) {
#pragma unroll 1
    for (int part = 0; part < 4; ++part) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(32 * q) << 16) + 32 * part, v);
        tmem_wait_ld();
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            float t[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float x = v[8 * cc + e];
                if (bias) x += bias[32 * part + 8 * cc + e];
                t[e] = tanh_approx(x);
            }
            const int kb = part >> 1, chunk = 4 * (part & 1) + cc;
            uint4 pk = make_uint4(pack_bf16x2(t[0], t[1]), pack_bf16x2(t[2], t[3]), pack_bf16x2(t[4], t[5]), pack_bf16x2(t[6], t[7]));
            *reinterpret_cast<uint4*>(A + kb * 16384 + row * 128 + ((chunk ^ (row & 7)) << 4)) = pk;
        }
    }
}

// LDC: compile-time row pitch of Vs / Vb / A1 / A2 (520 for F = 513: store offsets become immediates), 0 = take p.ld
// STORE = false: the Wiener mask sums of the final filter (mcem.py:325-327) instead of Vs / A1 / A2, so its 75 (25) samples
// are never written to memory: WFn = Vb sum_r 1 / Vx and WFs = g sum_r Vs / Vx.  The speech sum is accumulated, not taken
// as R - Vb A1: where g Vs << Vb (collapsed gains, spectral nulls) that difference cancels to FP32 noise, even negative.
template <int R, int L, int LDC, bool STORE>
__global__ void __launch_bounds__(DS_THREADS, 1) decode_stats_kernel(DsParams p) {
    constexpr int RL = (R <= 16) ? 16 : 32;
    constexpr int FT = (R == 25) ? 4 : 128 / R;        // frames per tile (R = 25: 4 x 25 = 100 rows, so that FT stays a multiple of 4)
    constexpr int FS = FT / 4;                         // frames per back warp
    static_assert(FT % 4 == 0 && (FT - 1) * R + RL <= 128 && FT * R <= 128, "tile geometry");
    extern __shared__ unsigned char smem_raw[];
    __shared__ uint64_t bars[5 + 3 * DS_NS];
    __shared__ uint32_t tmem_slot;
    __shared__ int dead_flag;
    __shared__ float tailS[256];

    const Dims& d = p.d;
    const int ldv = (LDC > 0) ? LDC : p.ld;
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool front = warp < 4;
    const int shared_bytes = (d.off_w3 + 4 * ((d.n_hidden == 2 ? HID : 0) + NPAD) + 1023) & ~1023;
    float* biasp = reinterpret_cast<float*>(base + d.off_w3);
    unsigned char* Abuf = base + shared_bytes;                       // 2 x 32 KB
    unsigned char* Wslot = Abuf + 65536;                             // DS_NS x 32 KB
    const uint32_t bar12 = smem_u32(&bars[0]);
    const uint32_t a_full0 = smem_u32(&bars[1]), a_full1 = smem_u32(&bars[2]);
    const uint32_t a_free0 = smem_u32(&bars[3]), a_free1 = smem_u32(&bars[4]);
    // ring stage sl: W3 slot loaded / layer-3 accumulator ready / accumulator drained (8 bytes apart)
    const uint32_t w_full = smem_u32(&bars[5]), bar3 = smem_u32(&bars[5 + DS_NS]), barf = smem_u32(&bars[5 + 2 * DS_NS]);

    {
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(base);
        for (int i = threadIdx.x; i < d.off_w3 / 16; i += DS_THREADS) dst[i] = __ldg(src + i);
        const uint4* bsrc = reinterpret_cast<const uint4*>(p.image + d.off_bias);
        uint4* bdst = reinterpret_cast<uint4*>(biasp);
        for (int i = threadIdx.x; i < (d.image_bytes - d.off_bias) / 16; i += DS_THREADS) bdst[i] = __ldg(bsrc + i);
    }
    if (threadIdx.x == 0) {
        dead_flag = 0;
        mbar_init(bar12, 1);
        mbar_init(a_full0, 128); mbar_init(a_full1, 128);
        mbar_init(a_free0, 1); mbar_init(a_free1, 1);
        for (int i = 0; i < DS_NS; ++i) { mbar_init(w_full + 8 * i, 1); mbar_init(bar3 + 8 * i, 1); mbar_init(barf + 8 * i, DS_BACK); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    volatile int* dead = &dead_flag;

    const uint32_t w1_addr = smem_u32(base), w2_addr = smem_u32(base + d.off_w2);
    const float* b2 = (d.n_hidden == 2) ? biasp : nullptr;
    const float* b3 = biasp + (d.n_hidden == 2 ? HID : 0);
    const unsigned char* w3g = p.image + d.off_w3;
    const int y_dim = d.y_dim, nkb1 = d.nkb1;
    const bool two_hidden = d.n_hidden == 2;
    const int64_t n_tiles = (p.NT + FT - 1) / FT;

    if (front) {
        // =========================================== front: layers 1-2 ===========================================
        const int q = warp, row = 32 * warp + lane;
        const int fi = row / R, r = row - fi * R;
        uint32_t ph12 = 0, phfree0 = 0, phfree1 = 0;
        int k = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
            const int buf = k & 1;
            unsigned char* A = Abuf + buf * 32768;
            const uint32_t a_addr = smem_u32(A);
            const int64_t n = tile * FT + fi;
            const bool valid = (fi < FT) && (n < p.NT);
            float z[L];
            float y0 = 0.f, y1 = 0.f, y2 = 0.f;
            if (valid) {
                const float4* src = reinterpret_cast<const float4*>(p.Zs + (n * p.zs_rtot + p.zs_r0 + r) * (int64_t)L);
#pragma unroll
                for (int l = 0; l < L / 4; ++l) {
                    const float4 t4 = __ldg(src + l);
                    z[4 * l] = t4.x; z[4 * l + 1] = t4.y; z[4 * l + 2] = t4.z; z[4 * l + 3] = t4.w;
                }
                if (y_dim > 0) y0 = p.y[n * y_dim];
                if (y_dim > 1) y1 = p.y[n * y_dim + 1];
                if (y_dim > 2) y2 = p.y[n * y_dim + 2];
            } else {
#pragma unroll
                for (int l = 0; l < L; ++l) z[l] = 0.f;
            }
            if (k >= 2) {                              // the layer-3 MMAs of tile k-2 have finished reading this buffer
                if (buf == 0) { mbar_wait(a_free0, phfree0, dead, p.status); phfree0 ^= 1; }
                else { mbar_wait(a_free1, phfree1, dead, p.status); phfree1 ^= 1; }
            }
            write_a1_static<L>(y_dim, nkb1, A, row, z, y0, y1, y2, valid);
            fence_async_smem();
            ds_bar_front();
            if (threadIdx.x == 0) {
                tc_fence_after();
                issue_gemm2(a_addr, 16384, w1_addr, 16384, nkb1, tmem, HID);
                umma_commit(bar12);
            }
            mbar_wait(bar12, ph12, dead, p.status);
            ph12 ^= 1;
            tc_fence_after();
            ds_hidden_row(tmem, A, q, row, (p.ybias && valid) ? p.ybias + n * HID : nullptr);
            fence_async_smem();
            tc_fence_before();
            ds_bar_front();
            if (two_hidden) {
                if (threadIdx.x == 0) {
                    tc_fence_after();
                    issue_gemm2(a_addr, 16384, w2_addr, 16384, 2, tmem, HID);
                    umma_commit(bar12);
                }
                mbar_wait(bar12, ph12, dead, p.status);
                ph12 ^= 1;
                tc_fence_after();
                ds_hidden_row(tmem, A, q, row, b2);
                fence_async_smem();
                tc_fence_before();
            }
            mbar_arrive2(buf ? a_full1 : a_full0);      // h2 of this tile is in A[buf]
        }
    } else if (warp < 20) {
        // =========================================== back: layer 3, Vs, statistics ===========================================
        const int bw = warp - 4;
        const int q = bw & 3, s = bw >> 2;              // TMEM lane quadrant (bins 32q..), frame slot
        const uint32_t lane_off = (uint32_t)(32 * q) << 16;
        int sl = 0;                                     // ring stage of the current chunk and the parity of its use count
        uint32_t par = 0;
        int k = 0;
        // Vb and g of the NEXT chunk are fetched while the current one is processed (their DRAM latency otherwise sits in
        // front of every chunk: 18 % of the stall samples in profiles/r01_tc_ncu_decode_stats.txt)
        float vbn[FS], ggn[FS];
        auto prefetch = [&](int64_t tl, int j) {
#pragma unroll
            for (int ff = 0; ff < FS; ++ff) {
                const int64_t n = tl * FT + s * FS + ff;
                const bool ok = (tl < n_tiles) && (n < p.NT);
                vbn[ff] = ok ? __ldg(p.Vb + n * ldv + 128 * j + 32 * q + lane) : 0.f;
                ggn[ff] = ok ? __ldg(p.g + n) : 0.f;
            }
        };
        prefetch(blockIdx.x, 0);
        // The thread's four layer-3 biases (one per 128-bin chunk) live in registers: read from shared memory at the start of
        // every chunk, the load queued behind the chunk's 30 stores per thread and its first consumer collected 29 % of the
        // kernel's stall samples (profiles/r01_tc_ncu_decode_stats.txt).
        const float bias_c0 = b3[32 * q + lane], bias_c1 = b3[128 + 32 * q + lane], bias_c2 = b3[256 + 32 * q + lane],
                    bias_c3 = b3[384 + 32 * q + lane];
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
            const int64_t t0 = tile * FT;
#pragma unroll 1
            for (int j = 0; j < 5; ++j) {
                mbar_wait(bar3 + 8 * sl, par, dead, p.status);
                tc_fence_after();
                const uint32_t tb = tmem + 128 + 128 * sl;
                if (j < 4) {
                    const int f = 128 * j + 32 * q + lane;
                    const float bias = (j == 0) ? bias_c0 : ((j == 1) ? bias_c1 : ((j == 2) ? bias_c2 : bias_c3));
                    float vbc[FS], ggc[FS];
#pragma unroll
                    for (int ff = 0; ff < FS; ++ff) { vbc[ff] = vbn[ff]; ggc[ff] = ggn[ff]; }
                    if (j < 3) prefetch(tile, j + 1);
                    else prefetch(tile + gridDim.x, 0);
#pragma unroll
                    for (int ff = 0; ff < FS; ++ff) {
                        const int fi = s * FS + ff;
                        const int64_t n = t0 + fi;
                        if (n < p.NT) {
                            const float gg = ggc[ff];
                            const float vb = vbc[ff];
                            float* dst = p.Vs + (n * p.zs_rtot + p.zs_r0) * (int64_t)ldv + f;
                            // packed FP32 pairs; four samples share two reciprocals: X = (Vx_r, Vx_r+1), Y = (Vx_r+2, Vx_r+3),
                            // 1 / (X Y) gives 1 / X = Y / (X Y) and 1 / Y = X / (X Y) lane by lane
                            const f32x2 g2 = pk2(gg, gg), vb2 = pk2(vb, vb), bias2 = pk2(bias, bias);
                            f32x2 a1p = 0ull, a2p = 0ull, asp = 0ull;
                            float a1 = 0.f, a2 = 0.f, as = 0.f;          // as: sum_r Vs / Vx (STORE = false)
                            // CNT samples (rows r0 .. r0 + CNT of the frame) held in v[0 .. CNT)
                            auto quad = [&](const float* v, int k, int r0) {
                                float e0, e1, e2, e3;
                                upk2(add2(pk2(v[k], v[k + 1]), bias2), e0, e1);
                                upk2(add2(pk2(v[k + 2], v[k + 3]), bias2), e2, e3);
                                const float s0 = ex2_approx(e0), s1 = ex2_approx(e1), s2 = ex2_approx(e2), s3 = ex2_approx(e3);
                                if (STORE) {
                                    dst[(int64_t)(r0 + k) * ldv] = s0;
                                    dst[(int64_t)(r0 + k + 1) * ldv] = s1;
                                    dst[(int64_t)(r0 + k + 2) * ldv] = s2;
                                    dst[(int64_t)(r0 + k + 3) * ldv] = s3;
                                }
                                const f32x2 X = fma2(g2, pk2(s0, s1), vb2), Y = fma2(g2, pk2(s2, s3), vb2);
                                float m0, m1;
                                upk2(mul2(X, Y), m0, m1);
                                const f32x2 rr = pk2(rcp_approx(m0), rcp_approx(m1));
                                const f32x2 i0 = mul2(Y, rr), i1 = mul2(X, rr);
                                a1p = add2(a1p, add2(i0, i1));
                                if (STORE) a2p = fma2(i0, i0, fma2(i1, i1, a2p));
                                else asp = fma2(pk2(s0, s1), i0, fma2(pk2(s2, s3), i1, asp));
                            };
                            auto pair = [&](const float* v, int k, int r0) {
                                const float s0 = ex2_approx(v[k] + bias), s1 = ex2_approx(v[k + 1] + bias);
                                if (STORE) {
                                    dst[(int64_t)(r0 + k) * ldv] = s0;
                                    dst[(int64_t)(r0 + k + 1) * ldv] = s1;
                                }
                                const float x0 = fmaf(gg, s0, vb), x1 = fmaf(gg, s1, vb);
                                const float rr = rcp_approx(x0 * x1);
                                const float i0 = x1 * rr, i1 = x0 * rr;
                                a1 += i0 + i1;
                                if (STORE) a2 = fmaf(i0, i0, fmaf(i1, i1, a2));
                                else as = fmaf(s0, i0, fmaf(s1, i1, as));
                            };
                            auto single = [&](const float* v, int k, int r0) {
                                const float s0 = ex2_approx(v[k] + bias);
                                if (STORE) dst[(int64_t)(r0 + k) * ldv] = s0;
                                const float i0 = rcp_approx(fmaf(gg, s0, vb));
                                a1 += i0;
                                if (STORE) a2 = fmaf(i0, i0, a2);
                                else as = fmaf(s0, i0, as);
                            };
                            static_assert(R == 30 || R == 25 || R == 10, "sample count of the back epilogue");
                            float v0[16];
                            tmem_ld16(tb + lane_off + fi * R, v0);
                            tmem_wait_ld();
                            if (R == 30) {
                                // second half of the samples: requested now, consumed after the first half has been processed
                                // (all 16 back warps read TMEM at the same moment: the load queue is ~1 k cycles deep)
                                float v1[16];
                                tmem_ld16(tb + lane_off + fi * R + 16, v1);
                                quad(v0, 0, 0); quad(v0, 4, 0); quad(v0, 8, 0); quad(v0, 12, 0);
                                tmem_wait_ld();
                                quad(v1, 0, 16); quad(v1, 4, 16); quad(v1, 8, 16); pair(v1, 12, 16);
                            } else if (R == 25) {
                                float v1[16];
                                tmem_ld16(tb + lane_off + fi * R + 16, v1);
                                quad(v0, 0, 0); quad(v0, 4, 0); quad(v0, 8, 0); quad(v0, 12, 0);
                                tmem_wait_ld();
                                quad(v1, 0, 16); quad(v1, 4, 16); single(v1, 8, 16);
                            } else {
                                quad(v0, 0, 0); quad(v0, 4, 0); pair(v0, 8, 0);
                            }
                            {
                                float lo, hi;
                                upk2(a1p, lo, hi);
                                a1 += lo + hi;
                                upk2(STORE ? a2p : asp, lo, hi);
                                if (STORE) a2 += lo + hi;
                                else as += lo + hi;
                            }
                            const int64_t i = n * ldv + f;
                            bool finite;
                            if (STORE) {
                                if (p.acc) { a1 += p.A1[i]; a2 += p.A2[i]; }
                                p.A1[i] = a1;
                                p.A2[i] = a2;
                                finite = isfinite(a1) && isfinite(a2);
                            } else {
                                float wn = __fmul_rn(vb, a1), ws = __fmul_rn(gg, as);   // no FMA contraction: WFn = fl(Vb A1)
                                if (p.acc) { wn += p.WFn[i]; ws += p.WFs[i]; }
                                p.WFn[i] = wn;
                                p.WFs[i] = ws;
                                finite = isfinite(wn) && isfinite(ws);
                            }
                            if (!finite) atomicOr(p.status, DVAE_STATUS_NONFINITE);
                        }
                    }
                } else if (s == 0) {
                    // bin 512: the MMA ran untransposed, TMEM lane = row of the tile, column 0 = bin 512
                    const int row = 32 * q + lane;
                    const int fi = row / R, r = row - fi * R;
                    const int64_t n = t0 + fi;
                    float v[4];
                    tmem_ld4(tb + lane_off, v);
                    tmem_wait_ld();
                    float inv = 0.f, vs = 0.f;
                    if (fi < FT && n < p.NT && d.F > 512) {
                        vs = ex2_approx(v[0] + b3[512]);
                        if (STORE) p.Vs[(n * p.zs_rtot + p.zs_r0 + r) * (int64_t)ldv + 512] = vs;
                        inv = rcp_approx(fmaf(__ldg(p.g + n), vs, __ldg(p.Vb + n * ldv + 512)));
                    }
                    tailS[row] = inv;
                    tailS[128 + row] = STORE ? inv * inv : vs * inv;
                    ds_bar_tail();
                    if (row < 2 * FT) {
                        const int fj = row >> 1, which = row & 1;
                        const int64_t nn = t0 + fj;
                        if (nn < p.NT && d.F > 512) {
                            float sum = 0.f;
                            for (int rr = 0; rr < R; ++rr) sum += tailS[which * 128 + fj * R + rr];
                            float* dst512;
                            if (STORE) {
                                dst512 = (which ? p.A2 : p.A1) + nn * ldv + 512;
                            } else {
                                dst512 = (which ? p.WFs : p.WFn) + nn * ldv + 512;
                                sum = __fmul_rn(which ? __ldg(p.g + nn) : __ldg(p.Vb + nn * ldv + 512), sum);
                            }
                            const float tot = p.acc ? *dst512 + sum : sum;
                            *dst512 = tot;
                            if (!isfinite(tot)) atomicOr(p.status, DVAE_STATUS_NONFINITE);
                        }
                    }
                    ds_bar_tail();
                }
                tc_fence_before();
                mbar_arrive2(barf + 8 * sl);
                if (++sl == DS_NS) { sl = 0; par ^= 1; }
            }
        }
    } else if (lane == 0) {
        // =========================================== issue warp: W3 stream + layer-3 MMAs ===========================================
        uint32_t phfull0 = 0, phfull1 = 0;
        const uint32_t slot_addr = smem_u32(Wslot);
        // chunk c of the CTA's stream: tile k = c / 5, j = c % 5; ring stage sl = c % DS_NS, used for the (c / DS_NS)-th time
        auto load_chunk = [&](int j, int sl) {          // issuer only
            const uint32_t bytes = (j < 4) ? 16384u : 2048u;
            const uint32_t bar = w_full + 8 * sl;
            ds_expect_tx(bar, 2 * bytes);
            ds_bulk_g2s(slot_addr + sl * 32768, w3g + (size_t)j * 128 * 128, bytes, bar);
            ds_bulk_g2s(slot_addr + sl * 32768 + 16384, w3g + NPAD * 128 + (size_t)j * 128 * 128, bytes, bar);
        };
        auto issue_chunk = [&](int64_t c2, int sl, bool first_use) {   // issuer only
            const int kk = (int)(c2 / 5), j = (int)(c2 % 5);
            const uint32_t use = (uint32_t)((c2 / DS_NS) & 1);
            const int buf = kk & 1;
            const uint32_t a_addr = smem_u32(Abuf + buf * 32768);
            mbar_wait(w_full + 8 * sl, use, dead, p.status);
            if (j == 0) {
                if (buf == 0) { mbar_wait(a_full0, phfull0, dead, p.status); phfull0 ^= 1; }
                else { mbar_wait(a_full1, phfull1, dead, p.status); phfull1 ^= 1; }
            }
            if (!first_use) mbar_wait(barf + 8 * sl, use ^ 1u, dead, p.status);      // the accumulator was drained by chunk c2 - DS_NS
            tc_fence_after();
            const uint32_t tb = tmem + 128 + 128 * sl;
            if (j < 4) issue_gemm2(slot_addr + sl * 32768, 16384, a_addr, 16384, 2, tb, 128);      // D^T = W3 chunk x h2^T
            else issue_gemm2(a_addr, 16384, slot_addr + sl * 32768, 16384, 2, tb, 16);             // bin 512: D = h2 x w^T
            umma_commit(bar3 + 8 * sl);
            if (j == 4) umma_commit(buf ? a_free1 : a_free0);                                       // A[buf] may be rewritten
        };

        const int64_t my_tiles = (n_tiles > blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
        const int64_t n_chunks = my_tiles * 5;
        for (int i = 0; i < DS_NS && i < n_chunks; ++i) load_chunk(i % 5, i);
        for (int i = 0; i < DS_NS && i < n_chunks; ++i) issue_chunk(i, i, true);
        int sl = 0;
        uint32_t par = 0;
        for (int64_t c = 0; c + DS_NS < n_chunks; ++c) {
            mbar_wait(bar3 + 8 * sl, par, dead, p.status);                                          // GEMM of chunk c done: W slot free
            const int64_t c2 = c + DS_NS;
            load_chunk((int)(c2 % 5), sl);
            issue_chunk(c2, sl, false);
            if (++sl == DS_NS) { sl = 0; par ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512) : "memory");
    }
}

// W <- W * sqrt(num / den), num[f,k] = sum_n P A2 H, den[f,k] = sum_n A1 H   (mcem.py:108-111)
// One thread per bin; the utterance's H rows are staged in shared memory (12 floats per frame, read back as three
// 16-byte broadcasts) and (num_k, den_k) is one packed FP32 pair updated by a single FFMA2 per rank.
constexpr int WFS_MAXFR = 256;                     // frames staged per pass (12 KB)
__global__ void __launch_bounds__(128, 6) w_from_frame_stats_kernel(const float* __restrict__ A1, const float* __restrict__ A2,
                                                                 const float* __restrict__ P, const float* __restrict__ H,
                                                                 const float* __restrict__ W, const int64_t* __restrict__ fr_off,
                                                                 int F, int K, int ld, float* __restrict__ Wtmp) {
    constexpr int KT = 10;
    __shared__ __align__(16) float Hs[WFS_MAXFR * 12];
    const int u = blockIdx.y;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = f < F;
    f32x2 nd[KT];
#pragma unroll
    for (int k = 0; k < KT; ++k) nd[k] = 0ull;
    const int64_t n0 = fr_off[u], n1 = fr_off[u + 1];
    for (int64_t base = n0; base < n1; base += WFS_MAXFR) {
        const int cnt = (int)((n1 - base < WFS_MAXFR) ? n1 - base : WFS_MAXFR);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt * 12; i += blockDim.x) {
            const int fr = i / 12, k = i - fr * 12;
            Hs[i] = (k < K) ? __ldg(H + (base + fr) * K + k) : 0.f;
        }
        __syncthreads();
        if (live) {
            const float* a1p = A1 + base * ld + f;
            const float* a2p = A2 + base * ld + f;
            const float* pp = P + base * ld + f;
#pragma unroll 8                            // 24 loads in flight per thread: the kernel is a pure HBM stream (3 x 4 x ld x N bytes per utterance)
            for (int i = 0; i < cnt; ++i) {
                const float a1 = __ldg(a1p + (int64_t)i * ld);
                const float pa2 = __ldg(pp + (int64_t)i * ld) * __ldg(a2p + (int64_t)i * ld);
                const f32x2 x = pk2(pa2, a1);
                const float4 h0 = *reinterpret_cast<const float4*>(Hs + 12 * i);
                const float4 h1 = *reinterpret_cast<const float4*>(Hs + 12 * i + 4);
                const float4 h2 = *reinterpret_cast<const float4*>(Hs + 12 * i + 8);
                nd[0] = fma2(x, pk2(h0.x, h0.x), nd[0]); nd[1] = fma2(x, pk2(h0.y, h0.y), nd[1]);
                nd[2] = fma2(x, pk2(h0.z, h0.z), nd[2]); nd[3] = fma2(x, pk2(h0.w, h0.w), nd[3]);
                nd[4] = fma2(x, pk2(h1.x, h1.x), nd[4]); nd[5] = fma2(x, pk2(h1.y, h1.y), nd[5]);
                nd[6] = fma2(x, pk2(h1.z, h1.z), nd[6]); nd[7] = fma2(x, pk2(h1.w, h1.w), nd[7]);
                nd[8] = fma2(x, pk2(h2.x, h2.x), nd[8]); nd[9] = fma2(x, pk2(h2.y, h2.y), nd[9]);
            }
        }
    }
    if (!live) return;
#pragma unroll
    for (int k = 0; k < KT; ++k)
        if (k < K) {
            float num, den;
            upk2(nd[k], num, den);
            const int64_t i = ((int64_t)u * K + k) * ld + f;
            Wtmp[i] = W[i] * sqrtf(num / den);
        }
}

}  // namespace tc
}  // namespace dvae

using namespace dvae;
using namespace dvae::tc;

static int launch_decode_stats(const char* who, const DvaeMlp* dec, const void* image, const float* Zs, int R_total, int r0, int R,
                               int L, const float* y, int y_dim, const float* ybias, const float* Vb, const float* g, int64_t NT, int ld, float* Vs,
                               float* A1, float* A2, float* WFs, float* WFn, int accumulate, int* status, void* stream) {
    DsParams p{};
    int rc = check_dims(dec, L, y_dim, who, &p.d);
    if (rc) return rc;
    const bool store = Vs != nullptr;
    DVAE_REQUIRE(image && Zs && Vb && g && status && (store ? (A1 && A2) : (WFs && WFn)), "%s: null pointer", who);
    DVAE_REQUIRE(store ? (R == 10 || R == 30) : (R == 10 || R == 25 || R == 30), "%s: unsupported sample count %d", who, R);
    DVAE_REQUIRE(r0 >= 0 && r0 + R <= R_total, "%s: sample window [%d, %d) outside [0, %d)", who, r0, r0 + R, R_total);
    DVAE_REQUIRE(L == 16 || L == 32, "%s: latent size must be 16 or 32 (got %d)", who, L);
    DVAE_REQUIRE(y_dim <= 3 && (y_dim == 0 || y), "%s: bad label arguments", who);
    DVAE_REQUIRE(NT >= 0 && ld >= p.d.F, "%s: bad sizes", who);
    DVAE_REQUIRE((reinterpret_cast<uintptr_t>(Zs) & 15) == 0 && (reinterpret_cast<uintptr_t>(image) & 15) == 0,
                 "%s: Zs and image must be 16-byte aligned", who);
    if (NT == 0) return 0;
    p.image = (const unsigned char*)image;
    p.Zs = Zs; p.y = y; p.ybias = ybias; p.Vb = Vb; p.g = g; p.Vs = Vs; p.A1 = A1; p.A2 = A2; p.WFs = WFs; p.WFn = WFn; p.NT = NT; p.ld = ld; p.status = status;
    p.zs_rtot = R_total; p.zs_r0 = r0; p.acc = accumulate;
    const int shared_bytes = (p.d.off_w3 + 4 * ((p.d.n_hidden == 2 ? HID : 0) + NPAD) + 1023) & ~1023;
    const size_t smem = (size_t)shared_bytes + 65536 + (size_t)DS_NS * 32768 + 1024;
    DVAE_REQUIRE(smem <= 227 * 1024, "%s: shared memory budget exceeded", who);
    const int FT = (R == 25) ? 4 : 128 / R;
    const int64_t n_tiles = (NT + FT - 1) / FT;
    const int grid = (int)(n_tiles < 148 ? n_tiles : 148);
    cudaStream_t st = (cudaStream_t)stream;
#define DS_LAUNCH(RR, LL, LD, SS)                                                                                       \
    do {                                                                                                                \
        cudaFuncSetAttribute(decode_stats_kernel<RR, LL, LD, SS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        decode_stats_kernel<RR, LL, LD, SS><<<grid, DS_THREADS, smem, st>>>(p);                                         \
    } while (0)
#define DS_PICK(RR, SS)                                                 \
    do {                                                                \
        if (L == 16 && ld == 520) DS_LAUNCH(RR, 16, 520, SS);           \
        else if (L == 16) DS_LAUNCH(RR, 16, 0, SS);                     \
        else if (ld == 520) DS_LAUNCH(RR, 32, 520, SS);                 \
        else DS_LAUNCH(RR, 32, 0, SS);                                  \
    } while (0)
    if (store) {
        if (R == 10) DS_PICK(10, true);
        else DS_PICK(30, true);
    } else {
        if (R == 10) DS_PICK(10, false);
        else if (R == 25) DS_PICK(25, false);
        else DS_PICK(30, false);
    }
#undef DS_PICK
#undef DS_LAUNCH
    return check_launch("decode_stats_kernel");
}

extern "C" int dvae_decode_stats_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R, int L, const float* y,
                                    int y_dim, const float* ybias, const float* Vb, const float* g, int64_t NT, int ld, float* Vs, float* A1,
                                    float* A2, int* status, void* stream) {
    DVAE_REQUIRE(Vs && A2, "dvae_decode_stats_tc: null pointer");
    return launch_decode_stats("dvae_decode_stats_tc", dec, image, Zs, R, 0, R, L, y, y_dim, ybias, Vb, g, NT, ld, Vs, A1, A2, nullptr, nullptr, 0,
                               status, stream);
}

extern "C" int dvae_decode_wiener_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R_total, int r0, int R, int L,
                                     const float* y, int y_dim, const float* ybias, const float* Vb, const float* g, int64_t NT, int ld,
                                     float* WFs, float* WFn, int accumulate, int* status, void* stream) {
    return launch_decode_stats("dvae_decode_wiener_tc", dec, image, Zs, R_total, r0, R, L, y, y_dim, ybias, Vb, g, NT, ld, nullptr, nullptr,
                               nullptr, WFs, WFn, accumulate, status, stream);
}

// sample window [r0, r0 + R) of frames that hold R_total samples each (multi-chain runs): Vs rows n * R_total + r0 + r are
// written, A1 / A2 are overwritten (accumulate == 0) or added to
extern "C" int dvae_decode_stats_win_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R_total, int r0, int R, int L,
                                        const float* y, int y_dim, const float* ybias, const float* Vb, const float* g, int64_t NT, int ld, float* Vs,
                                        float* A1, float* A2, int accumulate, int* status, void* stream) {
    DVAE_REQUIRE(Vs && A2, "dvae_decode_stats_win_tc: null pointer");
    return launch_decode_stats("dvae_decode_stats_win_tc", dec, image, Zs, R_total, r0, R, L, y, y_dim, ybias, Vb, g, NT, ld, Vs, A1, A2,
                               nullptr, nullptr, accumulate, status, stream);
}

extern "C" int dvae_nmf_w_from_frame_stats(const float* A1, const float* A2, const float* P, const float* H, const float* W,
                                           const int64_t* fr_off, int B, int F, int K, int ld, float* Wtmp, void* stream) {
    DVAE_REQUIRE(A1 && A2 && P && H && W && fr_off && Wtmp && B >= 1 && K >= 1 && K <= 10 && ld >= F,
                 "dvae_nmf_w_from_frame_stats: bad arguments");
    w_from_frame_stats_kernel<<<dim3((F + 127) / 128, B), 128, 0, (cudaStream_t)stream>>>(A1, A2, P, H, W, fr_off, F, K, ld, Wtmp);
    return check_launch("w_from_frame_stats_kernel");
}
