// Second-generation tcgen05 Metropolis-Hastings sampler (the default "tc" sampler).
//
// Operand images and the layer plan are described in tc_decode.cu / DESIGN.md section 4; this file is the schedule inside the
// CTA, driven by ncu captures: the first sampler of round 1 ran at 0.7 IPC per SM because every phase was serialised behind
// CTA barriers with only two warps per scheduler and a long single-warp "owner" phase.
//
// A second capture (an intermediate 16-warp build) showed 38 % of all stalls on local-memory traffic: with 223 KB of shared
// memory carved out the L1 is tiny, so every spilled register or dynamically indexed array costs an L2 round trip.
// Hence, in this version:
//   * 8 warps only (2 per scheduler -> up to 255 registers per thread): nothing spills, nothing is indexed
//     dynamically (latent size is a template parameter, every loop over chunks is fully unrolled);
//   * the L2 latency of the P / Vb stream is hidden in software: the quads of sub-chunk t+2 (16 bins) are requested
//     while sub-chunk t is evaluated (three rotating register buffers);
//   * the layer-3 chunks are handed over with mbarriers only (chunk ready: tcgen05.commit; buffer free: 256 thread
//     arrivals), no CTA barrier inside the chunk loop;
//   * the random draws of the next proposal are produced inside the kernel, Philox-4x32-10 with the counters every sampler of
//     this library uses (utterance id, frame | chain << 20, global iteration, block), under the layer-2 GEMM, where all
//     warps would otherwise wait on an mbarrier; injected draws (parity runs) are read from global memory instead;
//   * on kept iterations the decoder output of the proposal, 2^v without the output-layer bias, is written to global
//     memory in BF16 (tiled layout, see Mh2Params::VsT) together with, per chain and kept sample, the index of the slot
//     that holds the chain's state: the E-step needs no second decode of the kept samples (mcem.py:280-290);
//   * the tcgen05.mma groups are issued by lane 0 of warps 1 / 2 / 3 / 5 (layer 1, layer 2, layer-3 chunks 0 + 1, chunk 2);
//   * the chain state of row 32*q + lane is split over the two threads (column halves) that share the row: each carries
//     half of the latent dimensions and takes the same accept decision from the same shared-memory partial sums;
//   * every TMEM read is double-buffered, the layer-2 bias is preloaded into the layer-2 accumulator (tcgen05.st) while
//     the layer-1 GEMM runs, and the first P / Vb sub-chunks are requested two phases before the layer-3 loop
//     (phase clocks before / after in DESIGN.md section 4).
#include <type_traits>

#include "tc_common.cuh"

namespace dvae {
namespace tc {

constexpr int MH2_THREADS = 256;             // 8 warps: warp w -> TMEM lane quadrant w&3, column half w>>2

struct Mh2Params {
    Dims d;
    const unsigned char* image;
    int64_t rows;                 // NT*C chains
    int C;
    const float* y;
    const float* ybias;           // per-frame layer-1 bias [frames][128] or null (label inputs folded into a bias, see dvae_b200.h)
    const uint4* PVpk;            // [tile][quad][128] {P0P1, P2P3, V0V1, V2V3} in BF16
    const float* g;
    const float* kscale;          // [frames] per-frame quad scale (power of two) the stream was packed with, or null: 2^15
    float* Z;
    float* Zs;
    const float* eps;             // injected draws [n_iter][rows][L] standard normals, or null: Philox inside the kernel
    const float* u;               // injected draws [n_iter][rows] uniforms
    const int32_t* frame_gid;     // Philox counter words per frame: global utterance id, frame index inside the utterance
    const int32_t* frame_idx;
    PhiloxKeys keys;              // round keys of the run seed (read from the parameter bank)
    uint32_t iter0;
    uint32_t* n_accept;
    float* a_trace;
    int n_burn, n_keep;
    float sd;
    int* status;
    // Emission of the kept samples' variances (null: off).  VsT[tile][slot][bg][row][16] in BF16: tile = chain / 128,
    // row = chain % 128, bg = bin / 16 (33 groups, bins 513..527 are padding), slot 0 = the state at the end of the burn-in,
    // slot 1 + r = the proposal of kept iteration r.  vs_idx[chain][32]: byte r = slot holding kept sample r.
    uint4* VsT;
    uint8_t* vs_idx;
    const uint32_t* iter0_frame;  // per-frame iter0 [frames] (mh2_kernel<.., .., true>) or null
};


// 16 bins of the log-likelihood (loglik16_pv of tc_common.cuh) that also hands back 2^v of the 16 bins as eight "VsT words"
// (common.cuh: bin 2j as bf16 in the low half, the whole word nearest to bin 2j+1): the emission of the kept samples' variances.
template <int POLY>
__device__ __forceinline__ void loglik16_pv_emit(const float* v, const uint4* pv, float g_row, float k_row, float& acc, float& accl,
                                                 uint32_t* out) {
    const f32x2 g2 = pk2(g_row, g_row), g2k = pk2(g_row * k_row, g_row * k_row);
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
        const uint4 w = pv[qd];
        const f32x2 e01 = (POLY >= 2) ? ex2_poly2(pk2(v[4 * qd + 0], v[4 * qd + 1])) : pk2(ex2_approx(v[4 * qd + 0]), ex2_approx(v[4 * qd + 1]));
        const f32x2 A = fma2(g2k, e01, pk2(__uint_as_float(w.x << 16), __uint_as_float(w.y << 16)));
        const f32x2 e23 = POLY ? ex2_poly2(pk2(v[4 * qd + 2], v[4 * qd + 3])) : pk2(ex2_approx(v[4 * qd + 2]), ex2_approx(v[4 * qd + 3]));
        const f32x2 B = fma2(g2, e23, pk2(__uint_as_float(w.z << 16), __uint_as_float(w.w << 16)));
        {
            float e0, e1, e2, e3;
            upk2(e01, e0, e1);
            upk2(e23, e2, e3);
out[2 * qd] = vst_word(e0, e1);
            out[2 * qd + 1] = vst_word(e2, e3);
        }
        const f32x2 M = mul2(A, B);
        const f32x2 N = fma2(pk2(__uint_as_float(w.x), __uint_as_float(w.y)), B,
                             mul2(pk2(__uint_as_float(w.z), __uint_as_float(w.w)), A));
        float mlo, mhi, nlo, nhi;
        upk2(M, mlo, mhi);
        upk2(N, nlo, nhi);
        const float pq = mlo * mhi;
        acc = fmaf(fmaf(nlo, mhi, nhi * mlo), rcp_approx(pq), acc);
        accl += lg2_approx(pq);
    }
}

// One Philox block -> four standard normals (the arithmetic of mh_draws / rng_dump4_kernel: bit-identical draws); block 0
// also carries the accept uniform (u01_low_bytes)
__device__ __forceinline__ float4 philox_normals4(uint32_t utt, uint32_t fc, uint32_t iter, uint32_t b, const PhiloxKeys& keys, float& u) {
    const Philox4 r = philox4x32_10_rk(utt, fc, iter, b, keys);
    u = u01_low_bytes(r);
    float4 o;
    box_muller(r.x, r.y, o.x, o.y);
    box_muller(r.z, r.w, o.z, o.w);
    return o;
}

// One 32-byte cell of the emission as a single 256-bit store (STG.E.ENL2.256: a whole sector per lane, 1 KB contiguous per warp).
// Measured on the E-step call at B = 512 (tools/bench_sampler.py): two 16-byte st.global.cs (evict-first) stores per cell cost
// +0.37 ms per call (half-sector writes that leave L2 before their second half arrives), two plain 16-byte stores +0.04 ms,
// the 256-bit store nothing (2.48 ms with emission against 2.52 ms without).
// One 32-byte cell of the emission as a single 256-bit store (STG.E.ENL2.256: a whole sector per lane, 1 KB contiguous per warp)
// with an evict-first L2 policy; the P / Vb stream, which every evaluation re-reads from L2, is loaded with an evict-last
// policy.  ncu on the E-step call at B = 512 (profiles/r02_ncu_mh2_emit_vs_plain.txt): the 3 GB the kept iterations write
// push clean lines out of L2 -- part of the P / Vb stream (DRAM reads 208 -> 445 MB) and the kernel's own instructions
// (no_instruction stalls 0.46 per issued instruction) -- which costs 0.55 ms per call without the policies and 0.3 ms with them.
// (Reserving part of L2 for evict-last lines with cudaLimitPersistingL2CacheSize made it worse: 32 MB +0.02 ms, 64 MB +0.3 ms,
// and the frame-statistics kernel that follows lost up to 0.6 ms.)
__device__ __forceinline__ void st_cell(uint4* p, const uint32_t (&o)[8], uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8}, %9;" :: "l"(p), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
                 "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]), "l"(pol) : "memory");
}
__device__ __forceinline__ uint4 ld_pv(const uint4* p, uint64_t pol) {
    uint4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
}

// PER_FRAME: the Philox iteration base comes from p.iter0_frame (a separate instantiation, so that the kernel without it keeps
// its instruction stream)
template <int L, int POLY, bool PER_FRAME>
__global__ void __launch_bounds__(MH2_THREADS, 1) mh2_kernel(Mh2Params p) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ uint64_t bars[6];                       // layer 1/2 ready, chunk ready x3, buffer free x2
    __shared__ uint32_t tmem_slot;
    __shared__ int dead_flag;

    const Dims& d = p.d;
    unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* A = base + ((d.image_bytes + 1023) & ~1023);
    float2* red2 = reinterpret_cast<float2*>(A + A_BYTES);       // [2][128] {partial l(z'), partial prior term} of each column half
    float* u_sh = reinterpret_cast<float*>(red2 + 2 * TM);       // [128] accept uniform of the next proposal (written by half 0)
    uint32_t* it0_sh = reinterpret_cast<uint32_t*>(u_sh + TM);    // [128] the row's Philox iteration base, with iter0_frame only
    const uint32_t bar12 = smem_u32(&bars[0]);
    const uint32_t bar3_0 = smem_u32(&bars[1]), bar3_1 = smem_u32(&bars[2]);
    const uint32_t barf_0 = smem_u32(&bars[3]);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = warp & 3, h = warp >> 2;             // TMEM lane quadrant, column half
    const bool owner = h == 0;                         // warps 0-3 also write the label / constant chunk, the trace and the accept count
    // tcgen05.mma issue is spread over lane 0 of different warps so that no single warp pays for all of it:
    // layer 1: warp 1, layer 2: warp 2, layer-3 chunks 0 + 1: warp 3, chunk 2: warp 5
    const bool lead = lane == 0;
    const int row = 32 * q + lane;
    uint32_t ph12 = 0, ph3_0 = 0, ph3_1 = 0, phf_0 = 0;

    {
        const uint4* src = reinterpret_cast<const uint4*>(p.image);
        uint4* dst = reinterpret_cast<uint4*>(base);
        for (int i = threadIdx.x; i < d.image_bytes / 16; i += MH2_THREADS) dst[i] = __ldg(src + i);
    }
    if (threadIdx.x == 0) {
        dead_flag = 0;
        mbar_init(bar12, 1);
        mbar_init(bar3_0, 1);
        mbar_init(bar3_1, 1);
        mbar_init(barf_0, MH2_THREADS);
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

    const uint32_t a_addr = smem_u32(A);
    const uint32_t w1_addr = smem_u32(base), w2_addr = smem_u32(base + d.off_w2), w3_addr = smem_u32(base + d.off_w3);
    const float* biasp = reinterpret_cast<const float*>(base + d.off_bias);
    const float* b2 = (d.n_hidden == 2) ? biasp : nullptr;
    const int n_iter = p.n_burn + p.n_keep;
    const int64_t n_tiles = (p.rows + TM - 1) / TM;
    const int y_dim = d.y_dim, nkb1 = d.nkb1;
    const bool two_hidden = d.n_hidden == 2;
    const uint32_t lane_off = (uint32_t)(32 * q) << 16;
    const bool emit = p.VsT != nullptr;
    uint64_t pol_last, pol_first;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
    // evaluations of a tile: the start state, the burn-in proposals, [the state again: its variances become slot 0 of the
    // emission], the kept proposals
    const int n_eval = n_iter + 1 + (emit ? 1 : 0);
    const int ev_rescore = emit ? p.n_burn + 1 : -1;
    const int n_slots = p.n_keep + 1;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row_g = tile * TM + row;
        const bool valid = row_g < p.rows;
        const int64_t fr = valid ? row_g / p.C : 0;
        const float g_row = valid ? p.g[fr] : 1.f;
        const float k_row = (valid && p.kscale) ? __ldg(p.kscale + fr) : kDefaultQuadScale;      // the frame's quad scale (pack_pv used the same)
        const uint4* PVt = p.PVpk + (tile * NQ) * TM + row;
        const float* ybias_row = p.ybias ? p.ybias + fr * HID : nullptr;
        // this thread's 32 bytes of bin group 0 in slot 0 of the tile's emission
        uint4* VsTt = emit ? p.VsT + ((size_t)tile * n_slots * (NPAD / 16) * TM + row) * 2 : nullptr;
        uint32_t ph_utt = 0, ph_fc = 0;                 // Philox counter words 0 and 1 of this chain
        if (!p.eps && valid) {
            ph_utt = (uint32_t)__ldg(p.frame_gid + fr);
            ph_fc = (uint32_t)__ldg(p.frame_idx + fr) | ((uint32_t)(row_g - fr * p.C) << 20);
        }

        // Chain state, split over the two column halves: thread (row, h) carries latent dimensions [h L/2, (h+1) L/2) of its
        // row's chain plus a copy of the scalars.  The proposal / accept code is a chain of dependent operations that runs
        // with one warp per scheduler, so halving its length matters more than the duplicated scalar work.  Both halves take
        // the accept decision from the same shared-memory operands in the same order, so they always agree bit for bit.
        constexpr int LH = L / 2;
        float zh[LH], zph[LH];
        float4 enn[LH / 4];                                // this half's draws of the next proposal
        float y0 = 0.f, y1 = 0.f, y2 = 0.f, ll_cur = 0.f, u_cur = 0.5f, prior_h = 0.f;
        uint32_t n_acc = 0, state_slot = 0;
        int prop = 0;                                      // index of the next proposal to draw
        // the frame's own iter0 (DvaeRng.iter0_frame) waits in shared memory: one more register would make the kernel spill
        if constexpr (PER_FRAME) it0_sh[row] = valid ? __ldg(p.iter0_frame + fr) : 0u;
#pragma unroll
        for (int l = 0; l < LH; ++l) { zh[l] = valid ? p.Z[row_g * L + h * LH + l] : 0.f; zph[l] = 0.f; }
#pragma unroll
        for (int l = 0; l < LH / 4; ++l) enn[l] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (owner && valid) {
            if (y_dim > 0) y0 = p.y[fr * y_dim];
            if (y_dim > 1) y1 = p.y[fr * y_dim + 1];
            if (y_dim > 2) y2 = p.y[fr * y_dim + 2];
        }

        // Draws of the next proposal (if the next evaluation is one), consumed at the top of the next evaluation.  Philox mode:
        // this thread's LH / 4 blocks are produced in two parts that sit under two different GEMM waits (part 0 under the
        // layer-2 GEMM, part 1 under the first layer-3 chunk; ~150 integer / MUFU instructions per block and thread, which
        // two warps per scheduler cannot hide under one wait); the accept uniform rides on block 0 and reaches the other
        // column half through shared memory.
        auto draw_part = [&](int ev, int part) {
            const int nxt = ev + 1;
            if (nxt >= n_eval || nxt == ev_rescore) return;
            if (p.eps) {
                if (part == 0 && valid) {
                    const float4* e = reinterpret_cast<const float4*>(p.eps + ((int64_t)prop * p.rows + row_g) * L + h * LH);
#pragma unroll
                    for (int l = 0; l < LH / 4; ++l) enn[l] = __ldg(e + l);
                    if (owner) u_sh[row] = __ldg(p.u + (int64_t)prop * p.rows + row_g);
                }
            } else {
                const uint32_t iter = (PER_FRAME ? it0_sh[row] : p.iter0) + (uint32_t)prop;
                constexpr int HALF = (LH / 4 + 1) / 2;              // blocks in part 0
#pragma unroll
                for (int l = 0; l < LH / 4; ++l) {
                    if ((l < HALF) != (part == 0)) continue;
                    float u;
                    enn[l] = philox_normals4(ph_utt, ph_fc, iter, (uint32_t)(h * (LH / 4) + l), p.keys, u);
                    if (l == 0 && owner) u_sh[row] = u;             // block 0 belongs to half 0
                }
            }
            if (part == 1) ++prop;
        };

        // One evaluation.  EMIT (compile time): the evaluation writes its variances to slot `store_slot` of the emission.  The
        // body exists twice, once per flag, and a tile runs [start + burn-in] through the plain copy and then [state again + kept
        // proposals] through the emitting copy: with ONE copy that branched around the stores in each of its 17 sub-chunks the
        // interleaved dead code cost 0.33 ms per call (13 %) even when nothing was emitted (instruction fetch; tools/bench_sampler.py).
        auto evaluate = [&](auto emit_c, const int ev) {
            constexpr bool EMIT = decltype(emit_c)::value;
            const bool score_only = (ev == 0) || (ev == ev_rescore);     // evaluates the chain's state, no decision
            const int it = ev - 1 - ((emit && ev > ev_rescore) ? 1 : 0);  // proposal index (meaningless when score_only)
            // slot of the emission this evaluation's variances go to
            const int store_slot = (ev == ev_rescore) ? 0 : 1 + (it - p.n_burn);
            if (!score_only) {
                u_cur = u_sh[row];
                prior_h = 0.f;
#pragma unroll
                for (int l = 0; l < LH / 4; ++l) {
                    zph[4 * l + 0] = __fadd_rn(zh[4 * l + 0], __fmul_rn(p.sd, enn[l].x));
                    zph[4 * l + 1] = __fadd_rn(zh[4 * l + 1], __fmul_rn(p.sd, enn[l].y));
                    zph[4 * l + 2] = __fadd_rn(zh[4 * l + 2], __fmul_rn(p.sd, enn[l].z));
                    zph[4 * l + 3] = __fadd_rn(zh[4 * l + 3], __fmul_rn(p.sd, enn[l].w));
                }
#pragma unroll
                for (int l = 0; l < LH; ++l) prior_h += __fsub_rn(__fmul_rn(zh[l], zh[l]), __fmul_rn(zph[l], zph[l]));
                write_a1_half<L>(y_dim, nkb1, A, row, h, zph, y0, y1, y2, valid);
            } else {
                write_a1_half<L>(y_dim, nkb1, A, row, h, zh, y0, y1, y2, valid);
            }
            fence_async_smem();
            __syncthreads();                                                    // S1: layer-1 operand ready

            if (warp == 1 && lead) {
                tc_fence_after();
                issue_gemm2(a_addr, 16384, w1_addr, 16384, nkb1, tmem + 384, HID);
                umma_commit(bar12);
            }
            if (two_hidden) {
                // Layer-2 bias preloaded into the layer-2 accumulator, TMEM columns [0, 128), while the layer-1 GEMM runs (every
                // warp would only spin on its mbarrier here; the stores take ~0.6 k cycles).  Every thread writes the 64 columns
                // it will read back in the layer-2 epilogue.  The columns are free (the previous evaluation's reads of them
                // completed before its S4; the first layer-3 chunk is issued after S3), the layer-2 GEMM, issued after S2,
                // accumulates onto the bias, and its epilogue needs no bias loads / adds.
                tc_fence_after();
                tmem_preload_bias64(tmem + lane_off + 64 * h, b2 + 64 * h);
                tmem_wait_st();
                tc_fence_before();
            }
            mbar_wait(bar12, ph12, dead, p.status);
            ph12 ^= 1;
            tc_fence_after();
            if (ybias_row) hidden_epilogue_rows_bf(tmem + 384, A, q, h, row, ybias_row);  // label inputs folded into a per-frame bias
            else hidden_epilogue_rows_bf(tmem + 384, A, q, h, row, nullptr);         // bias rides on the constant-one column
            fence_async_smem();
            tc_fence_before();
            __syncthreads();                                                    // S2
            float acc = 0.f, accl = 0.f;
            uint4 pv0[4], pv1[4], pv2[4];
            // sub-chunk t: chunk c = t/6 (capped at 2), column inside the chunk = h*W_c + 16*(t - 6c), W = 96, 96, 80
#define MH2_CH(t) ((t) < 6 ? 0 : ((t) < 12 ? 1 : 2))
#define MH2_COL(t) (h * (MH2_CH(t) == 2 ? 80 : 96) + 16 * ((t) - 6 * MH2_CH(t)))
#define MH2_BIN(t) (192 * MH2_CH(t) + MH2_COL(t))
#define MH2_LOAD(t, PV)                                                                              \
    do {                                                                                             \
        _Pragma("unroll") for (int qd = 0; qd < 4; ++qd) PV[qd] = ld_pv(PVt + ((MH2_BIN(t) >> 2) + qd) * TM, pol_last); \
    } while (0)
            // the first two sub-chunks of the P / Vb stream are requested here, two phases ahead of their use (the wait for
            // them at the start of the layer-3 loop was 3.6 % of the kernel's stall samples: profiles/r01_tc_ncu_mh2.txt)
            MH2_LOAD(0, pv0);
            MH2_LOAD(1, pv1);
            if (two_hidden) {
                if (warp == 2 && lead) {
                    tc_fence_after();
                    issue_gemm2(a_addr, 16384, w2_addr, 16384, 2, tmem, HID, 1);
                    umma_commit(bar12);
                }
                draw_part(ev, 0);                                               // in the shadow of the layer-2 GEMM
                mbar_wait(bar12, ph12, dead, p.status);
                ph12 ^= 1;
                tc_fence_after();
                hidden_epilogue_rows_bf(tmem, A, q, h, row, nullptr);
                fence_async_smem();
                tc_fence_before();
                __syncthreads();                                                // S3
            }
            // ---- layer 3 as three chunks of 192 / 192 / 160 bins (the last one over-reads 16 rows of padding):
            // chunk 0 -> TMEM columns [0,192), chunk 1 -> [192,384), chunk 2 -> [0,160) once chunk 0 is drained
            // one thread issues chunk 0 and then chunk 1: issued from two warps at once the two GEMMs interleaved in the tensor
            // pipe and chunk 0 (the one the epilogue is waiting for) completed 0.6 k cycles later
            if (warp == 3 && lead) {
                tc_fence_after();
                issue_gemm2(a_addr, 16384, w3_addr, NPAD * 128, 2, tmem, 192);
                umma_commit(bar3_0);
                issue_gemm2(a_addr, 16384, w3_addr + 192 * 128, NPAD * 128, 2, tmem + 192, 192);
                umma_commit(bar3_1);
            }
            if (!two_hidden) draw_part(ev, 0);
            draw_part(ev, 1);                                                   // in the shadow of the first layer-3 chunk

            // per thread 17 (h = 0) or 16 (h = 1) sub-chunks of 16 bins; the P / Vb quads of sub-chunk t+2 are requested
            // while sub-chunk t is evaluated (three rotating register buffers, everything statically indexed)
            // The TMEM reads are double-buffered: the 16 columns of sub-chunk t+1 are requested right after those of t have
            // arrived, so their latency runs under the arithmetic of t (with two warps per scheduler the other warp alone
            // cannot cover it: the single-buffer version spent half of the layer-3 phase with neither XU nor issue slots busy).
            float va[16], vb[16];
            uint4* vs_dst = EMIT ? VsTt + (size_t)store_slot * ((NPAD / 16) * TM * 2) : nullptr;
            mbar_wait(bar3_0, ph3_0, dead, p.status); ph3_0 ^= 1; tc_fence_after();
            tmem_ld16(tmem + lane_off + MH2_COL(0), va);
#define MH2_EVAL(V, PV, t)                                                                    \
    do {                                                                                      \
        if constexpr (EMIT) {                                                                 \
            uint32_t o[8];                                                                    \
            loglik16_pv_emit<POLY>(V, PV, g_row, k_row, acc, accl, o);                               \
            uint4* dst = vs_dst + (MH2_BIN(t) >> 4) * (TM * 2);                               \
            st_cell(dst, o, pol_first);                                                       \
        } else {                                                                              \
            loglik16_pv<POLY>(V, PV, g_row, k_row, acc, accl);                                       \
        }                                                                                     \
    } while (0)
            // The 17 sub-chunks are spelled out through a compile-time index (a `#pragma unroll` loop over this body was left
            // partly rolled by the compiler once the emission was added, which turned the statically indexed register buffers into
            // select chains: 1.8 x the instructions)
            auto step = [&](auto tc_) {
                constexpr int t = decltype(tc_)::value;
                const bool live = (t < 16) || (h == 0);                         // bins 528..543 do not exist
                if (t + 2 < 17 && ((t + 2 < 16) || (h == 0))) {
                    if constexpr ((t + 2) % 3 == 0) MH2_LOAD(t + 2, pv0);
                    else if constexpr ((t + 2) % 3 == 1) MH2_LOAD(t + 2, pv1);
                    else MH2_LOAD(t + 2, pv2);
                }
                if (live) tmem_wait_ld();                                       // sub-chunk t is in registers
                if constexpr (t == 5) {                                         // chunk 0 drained by this thread
                    tc_fence_before();
                    mbar_arrive2(barf_0);
                }
                if (t + 1 < 17 && ((t + 1 < 16) || (h == 0))) {
                    if constexpr (t + 1 == 6) { mbar_wait(bar3_1, ph3_1, dead, p.status); ph3_1 ^= 1; tc_fence_after(); }
                    if constexpr (t + 1 == 12) { mbar_wait(bar3_0, ph3_0, dead, p.status); ph3_0 ^= 1; tc_fence_after(); }
                    if constexpr ((t + 1) % 2 == 0) tmem_ld16(tmem + 192 * (MH2_CH(t + 1) & 1) + lane_off + MH2_COL(t + 1), va);
                    else tmem_ld16(tmem + 192 * (MH2_CH(t + 1) & 1) + lane_off + MH2_COL(t + 1), vb);
                }
                if (live) {
                    if constexpr (t % 2 == 0) {
                        if constexpr (t % 3 == 0) MH2_EVAL(va, pv0, t);
                        else if constexpr (t % 3 == 1) MH2_EVAL(va, pv1, t);
                        else MH2_EVAL(va, pv2, t);
                    } else {
                        if constexpr (t % 3 == 0) MH2_EVAL(vb, pv0, t);
                        else if constexpr (t % 3 == 1) MH2_EVAL(vb, pv1, t);
                        else MH2_EVAL(vb, pv2, t);
                    }
                }
                if constexpr (t == 5) {
                    if (warp == 5) {
                        if (lead) {
                            mbar_wait(barf_0, phf_0, dead, p.status);
                            tc_fence_after();
                            issue_gemm2(a_addr, 16384, w3_addr + 384 * 128, NPAD * 128, 2, tmem, 160);
                            umma_commit(bar3_0);
                        }
                        __syncwarp();
                    }
                    phf_0 ^= 1;
                }
            };
#define MH2_STEP(T) step(std::integral_constant<int, T>{})
            MH2_STEP(0); MH2_STEP(1); MH2_STEP(2); MH2_STEP(3); MH2_STEP(4); MH2_STEP(5); MH2_STEP(6); MH2_STEP(7); MH2_STEP(8);
            MH2_STEP(9); MH2_STEP(10); MH2_STEP(11); MH2_STEP(12); MH2_STEP(13); MH2_STEP(14); MH2_STEP(15); MH2_STEP(16);
#undef MH2_STEP
#undef MH2_EVAL
#undef MH2_LOAD
#undef MH2_BIN
#undef MH2_COL
#undef MH2_CH
            tc_fence_before();
            const float part = fmaf(kLn2, accl, acc * k_row);
            red2[h * TM + row] = make_float2(part, prior_h);
            __syncthreads();                                                    // S4: both halves of l(z') and of the prior term
            {
                const float2 r0 = red2[row], r1 = red2[TM + row];
                const float ll_prop = r0.x + r1.x;
                if (valid && !(fabsf(ll_prop) <= 3.0e38f)) atomicOr(p.status, DVAE_STATUS_NONFINITE);     // NaN / Inf likelihood
                if (score_only) {
                    ll_cur = ll_prop;
                    state_slot = 0;
                } else if (valid) {
                    const float a = (ll_cur - ll_prop) + 0.5f * (r0.y + r1.y);
                    if (owner && p.a_trace) p.a_trace[(int64_t)it * p.rows + row_g] = a;
                    if (__logf(u_cur) < a) {
#pragma unroll
                        for (int l = 0; l < LH; ++l) zh[l] = zph[l];
                        ll_cur = ll_prop;
                        ++n_acc;
                        if (EMIT) state_slot = (uint32_t)store_slot;
                    }
                    if (it >= p.n_burn) {
                        float4* dst = reinterpret_cast<float4*>(p.Zs + (row_g * p.n_keep + (it - p.n_burn)) * L + h * LH);
#pragma unroll
                        for (int l = 0; l < LH / 4; ++l) dst[l] = make_float4(zh[4 * l], zh[4 * l + 1], zh[4 * l + 2], zh[4 * l + 3]);
                        if (EMIT && owner) p.vs_idx[row_g * 32 + (it - p.n_burn)] = (uint8_t)state_slot;
                    }
                }
            }
        };
        {
            const int n_plain = emit ? ev_rescore : n_eval;
            for (int ev = 0; ev < n_plain; ++ev) evaluate(std::false_type{}, ev);
            for (int ev = n_plain; ev < n_eval; ++ev) evaluate(std::true_type{}, ev);
        }
        if (valid) {
#pragma unroll
            for (int l = 0; l < LH; ++l) p.Z[row_g * L + h * LH + l] = zh[l];
            if (owner && p.n_accept) p.n_accept[row_g] += n_acc;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512) : "memory");
    }
}

}  // namespace tc
}  // namespace dvae

using namespace dvae;
using namespace dvae::tc;

extern "C" int64_t dvae_vst_bytes(int64_t chains, int n_keep) {
    if (chains <= 0 || n_keep < 1) return 0;
    return ((chains + TM - 1) / TM) * (int64_t)(n_keep + 1) * (NPAD / 16) * TM * 32;
}

extern "C" int dvae_mh_chain_tc2(const DvaeMlp* dec, const void* image, const void* PVpk, const float* kscale, const float* g,
                                 const float* y, int y_dim, const float* ybias, const int32_t* frame_utt, const int32_t* frame_idx,
                                 float* Z, float* Zs,
                                 int64_t NT, int L, int n_chains, int n_burn, int n_keep, float var_rw, const DvaeRng* rng,
                                 uint32_t* n_accept, float* a_trace, void* VsT, uint8_t* vs_idx, int flags, int* status, void* stream) {
    Mh2Params p{};
    int rc = check_dims(dec, L, y_dim, "dvae_mh_chain_tc2", &p.d);
    if (rc) return rc;
    DVAE_REQUIRE(L == 16 || L == 32, "dvae_mh_chain_tc2: latent size must be 16 or 32 (got %d)", L);
    DVAE_REQUIRE(y_dim <= 3, "dvae_mh_chain_tc2: at most 3 label inputs");
    DVAE_REQUIRE(image && PVpk && g && Z && Zs && rng && status, "dvae_mh_chain_tc2: null pointer");
    DVAE_REQUIRE(y_dim == 0 || y, "dvae_mh_chain_tc2: y_dim=%d but y is null", y_dim);
    DVAE_REQUIRE(!ybias || (reinterpret_cast<uintptr_t>(ybias) & 15) == 0, "dvae_mh_chain_tc2: ybias must be 16-byte aligned");
    DVAE_REQUIRE(NT >= 0 && n_chains >= 1 && n_chains < 4096 && n_burn >= 0 && n_keep >= 1 && var_rw > 0.f, "dvae_mh_chain_tc2: bad sizes");
    DVAE_REQUIRE((rng->eps == nullptr) == (rng->u == nullptr), "dvae_mh_chain_tc2: eps and u must be injected together");
    DVAE_REQUIRE(!(rng->eps && rng->iter0_frame), "dvae_mh_chain_tc2: iter0_frame applies to Philox draws only");
    DVAE_REQUIRE(rng->eps || (frame_utt && frame_idx), "dvae_mh_chain_tc2: Philox mode needs frame_utt / frame_idx");
    DVAE_REQUIRE((reinterpret_cast<uintptr_t>(Zs) & 15) == 0 && (reinterpret_cast<uintptr_t>(rng->eps) & 15) == 0,
                 "dvae_mh_chain_tc2: Zs and eps must be 16-byte aligned");
    DVAE_REQUIRE((VsT == nullptr) == (vs_idx == nullptr), "dvae_mh_chain_tc2: VsT and vs_idx go together");
    DVAE_REQUIRE(!VsT || (n_keep <= 31 && (reinterpret_cast<uintptr_t>(VsT) & 31) == 0),
                 "dvae_mh_chain_tc2: the emission holds at most 31 kept samples per chain, 32-byte aligned");
    if (NT == 0) return 0;
    p.image = (const unsigned char*)image;
    p.rows = NT * n_chains; p.C = n_chains; p.y = y; p.ybias = ybias;
    p.PVpk = (const uint4*)PVpk; p.kscale = kscale; p.g = g; p.Z = Z; p.Zs = Zs;
    p.eps = rng->eps; p.u = rng->u;
    p.frame_gid = frame_utt; p.frame_idx = frame_idx;
    p.keys = philox_keys((uint32_t)(rng->seed & 0xffffffffu), (uint32_t)(rng->seed >> 32)); p.iter0 = rng->iter0;
    p.iter0_frame = rng->iter0_frame;
    p.n_accept = n_accept; p.a_trace = a_trace; p.n_burn = n_burn; p.n_keep = n_keep;
    p.sd = sqrtf(var_rw);
    p.status = status;
    p.VsT = (uint4*)VsT; p.vs_idx = vs_idx;
    // + red2 [2][128] float2, u_sh [128] and, with iter0_frame, it0_sh [128] behind the activation operand
    const size_t smem = smem_bytes(p.d) + (size_t)TM * (rng->iter0_frame ? 24 : 20);
    DVAE_REQUIRE(smem <= 227 * 1024, "dvae_mh_chain_tc2: shared memory budget exceeded");
    const int64_t n_tiles = (p.rows + TM - 1) / TM;
    const int grid = (int)(n_tiles < 148 ? n_tiles : 148);
    cudaStream_t st = (cudaStream_t)stream;
    const int poly = (flags & DVAE_TC_POLY_EX2_ALL) ? 2 : ((flags & DVAE_TC_POLY_EX2) ? 1 : 0);
#define MH2_LAUNCH2(LL, PP, PF)                                                                                  \
    do {                                                                                                         \
        cudaFuncSetAttribute(mh2_kernel<LL, PP, PF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);    \
        mh2_kernel<LL, PP, PF><<<grid, MH2_THREADS, smem, st>>>(p);                                              \
    } while (0)
#define MH2_LAUNCH(LL, PP)                          \
    do {                                            \
        if (p.iter0_frame) MH2_LAUNCH2(LL, PP, true); \
        else MH2_LAUNCH2(LL, PP, false);            \
    } while (0)
    if (L == 16 && poly == 2) MH2_LAUNCH(16, 2);
    else if (L == 16 && poly == 1) MH2_LAUNCH(16, 1);
    else if (L == 16) MH2_LAUNCH(16, 0);
    else if (poly == 2) MH2_LAUNCH(32, 2);
    else if (poly == 1) MH2_LAUNCH(32, 1);
    else MH2_LAUNCH(32, 0);
#undef MH2_LAUNCH
#undef MH2_LAUNCH2
    return check_launch("mh2_kernel");
}
