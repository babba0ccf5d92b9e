// FP32 ("exact" mode) dense tanh MLP and the Metropolis-Hastings E-step sampler built on it.
//
// Replaces packages/models/models.py:102-105,119-122 (Encoder / Decoder forward) and
// packages/models/mcem.py:207-277 (+ the M2 / M2v2 / M2v3 copies at 372-448, 544-620, 716-792).
//
// This is the CUDA-core reference mode of the product: every contraction is an FP32 FFMA chain, so the log
// acceptance ratio agrees with the CPU reference to FP32 rounding.  The tensor-core sampler (mh_tc2.cu) is checked
// against this one.  Restructuring w.r.t. the reference (exact in real arithmetic, SURVEY §7.2):
//   * the chain carries l(z) = sum_f [log Vx + P/Vx]; it only changes on accept, so the post-accept decoder
//     re-evaluation of mcem.py:268 disappears and a = l(z) - l(z') + .5 sum(z^2 - z'^2);
//   * the decoder's last layer never materialises Vs': its epilogue reduces log Vx' + P/Vx' over a 64-bin tile
//     and stores one partial per (chain, tile); partials are summed in fixed order (deterministic).
#include "common.cuh"

namespace dvae {

constexpr int BM = 64, BN = 64, BK = 16;
constexpr int kRowChunk = 1 << 18;           // rows per pass of dvae_mlp_fwd (bounds the workspace)

enum { EPI_NONE = 0, EPI_TANH = 1, EPI_EXP = 2, EPI_LOGLIK = 3 };

struct LoglikArgs {
    const float* P;      // [NT][ld]
    const float* Vb;     // [NT][ld]
    const float* g;      // [NT]
    float* partial;      // [rows][n_tiles]
    int ld;
    int row_div;         // chains per frame
    int n_tiles;
};

// out[m][n] = epi( sum_k A[m][k] * Wt[k][n] + bias[n] ),   A[m][k] = k < k1 ? x[m*ldx+k] : x2[(m/div)*ldx2 + k-k1]
template <int EPI>
__global__ void __launch_bounds__(256) linear_kernel(const float* __restrict__ x, int ldx, int k1,
                                                     const float* __restrict__ x2, int ldx2, int k2, int x2_div,
                                                     const float* __restrict__ Wt, const float* __restrict__ bias,
                                                     int64_t M, int N, float* __restrict__ out, int ldo, LoglikArgs ll) {
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int K = k1 + k2;

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int kt = 0; kt < K; kt += BK) {
        // A tile: 64 rows x 16 k, transposed into As[k][m]
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int kk = tid & 15, mm = (tid >> 4) + 16 * i;
            const int k = kt + kk;
            const int64_t m = m0 + mm;
            float v = 0.f;
            if (m < M) {
                if (k < k1) v = x[m * ldx + k];
                else if (k < K) v = x2[(m / x2_div) * ldx2 + (k - k1)];
            }
            As[kk][mm] = v;
        }
        // B tile: 16 k x 64 n
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int nn = tid & 63, kk = (tid >> 6) + 4 * i;
            const int k = kt + kk, n = n0 + nn;
            Bs[kk][nn] = (k < K && n < N) ? Wt[(int64_t)k * N + n] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }

    float bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) bv[j] = (n0 + tx * 4 + j < N) ? bias[n0 + tx * 4 + j] : 0.f;

    if (EPI != EPI_LOGLIK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t m = m0 + ty * 4 + i;
            if (m >= M) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + tx * 4 + j;
                if (n >= N) continue;
                float v = acc[i][j] + bv[j];
                if (EPI == EPI_TANH) v = tanhf(v);
                if (EPI == EPI_EXP) v = expf(v);
                out[m * ldo + n] = v;
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t m = m0 + ty * 4 + i;
            float s = 0.f;
            if (m < M) {
                const int64_t fr = m / ll.row_div;
                const float gg = ll.g[fr];
                const float* Pn = ll.P + fr * ll.ld;
                const float* Vn = ll.Vb + fr * ll.ld;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int n = n0 + tx * 4 + j;
                    if (n < N) {
                        const float vs = expf(acc[i][j] + bv[j]);
                        const float vx = __fadd_rn(__fmul_rn(gg, vs), Vn[n]);
                        s += logf(vx) + __fdiv_rn(Pn[n], vx);
                    }
                }
            }
            // the 16 threads of a row group sit in one half-warp: xor-reduce over lanes 0..15
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (tx == 0 && m < M) ll.partial[m * ll.n_tiles + blockIdx.y] = s;
        }
    }
}

static int launch_linear(int epi, const float* x, int ldx, int k1, const float* x2, int ldx2, int k2, int x2_div,
                         const float* Wt, const float* bias, int64_t M, int N, float* out, int ldo, LoglikArgs ll,
                         cudaStream_t st) {
    if (M == 0) return 0;
    dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN));
    if (x2_div < 1) x2_div = 1;
    switch (epi) {
        case EPI_NONE: linear_kernel<EPI_NONE><<<grid, 256, 0, st>>>(x, ldx, k1, x2, ldx2, k2, x2_div, Wt, bias, M, N, out, ldo, ll); break;
        case EPI_TANH: linear_kernel<EPI_TANH><<<grid, 256, 0, st>>>(x, ldx, k1, x2, ldx2, k2, x2_div, Wt, bias, M, N, out, ldo, ll); break;
        case EPI_EXP: linear_kernel<EPI_EXP><<<grid, 256, 0, st>>>(x, ldx, k1, x2, ldx2, k2, x2_div, Wt, bias, M, N, out, ldo, ll); break;
        default: linear_kernel<EPI_LOGLIK><<<grid, 256, 0, st>>>(x, ldx, k1, x2, ldx2, k2, x2_div, Wt, bias, M, N, out, ldo, ll); break;
    }
    return check_launch("linear_kernel");
}

static int max_hidden(const DvaeMlp* mlp) {
    int h = 1;
    for (int i = 1; i < mlp->n_layers; ++i) h = mlp->dims[i] > h ? mlp->dims[i] : h;
    return h;
}

static int check_mlp(const DvaeMlp* mlp, const char* who) {
    DVAE_REQUIRE(mlp != nullptr, "%s: null mlp", who);
    DVAE_REQUIRE(mlp->n_layers >= 1 && mlp->n_layers <= DVAE_MAX_LAYERS, "%s: n_layers=%d out of range", who, mlp->n_layers);
    for (int i = 0; i <= mlp->n_layers; ++i) DVAE_REQUIRE(mlp->dims[i] >= 1, "%s: dims[%d]=%d", who, i, mlp->dims[i]);
    for (int i = 0; i < mlp->n_layers; ++i) DVAE_REQUIRE(mlp->wt[i] && mlp->bias[i], "%s: null weights in layer %d", who, i);
    return 0;
}

// Layers [0, n_layers-1) with tanh; returns the pointer/ld of the last hidden activation (or the input).
// `last_epi` + out are applied to the final layer.
static int run_mlp(const DvaeMlp* mlp, const float* x, int ldx, int k1, const float* x2, int ldx2, int k2, int x2_div,
                   int64_t rows, int last_epi, float* out, int ldo, LoglikArgs ll, float* ws, cudaStream_t st) {
    const int mh = max_hidden(mlp);
    float* bufs[2] = {ws, ws + rows * (int64_t)mh};
    const float* cur = x;
    int cur_ld = ldx, cur_k1 = k1, cur_k2 = k2;
    const float* cur_x2 = x2;
    for (int i = 0; i < mlp->n_layers; ++i) {
        const bool last = (i == mlp->n_layers - 1);
        const int N = mlp->dims[i + 1];
        float* dst = last ? out : bufs[i & 1];
        const int dld = last ? ldo : N;
        int rc = launch_linear(last ? last_epi : EPI_TANH, cur, cur_ld, cur_k1, cur_x2, ldx2, cur_k2, x2_div, mlp->wt[i],
                               mlp->bias[i], rows, N, dst, dld, ll, st);
        if (rc) return rc;
        cur = dst; cur_ld = dld; cur_k1 = N; cur_k2 = 0; cur_x2 = nullptr;
    }
    return 0;
}

// ----------------------------------------------------------------------------- elementwise helpers
__global__ void reparam_kernel(const float* __restrict__ mu, const float* __restrict__ lv, const float* __restrict__ eps,
                               float* __restrict__ z, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        z[i] = fmaf(expf(0.5f * lv[i]), eps[i], mu[i]);
}

// ----------------------------------------------------------------------------- Metropolis-Hastings step
struct MhArgs {
    float* Z;            // [chains][L] current states
    float* Zp;           // [chains][L] proposals (decoder input of the next evaluation)
    float* ll_cur;       // [chains]
    float* u_next;       // [chains] uniform of the pending proposal
    const float* partial;  // [chains][n_tiles]
    float* Zs;           // [NT][C*n_keep][L]
    const int32_t* frame_utt;
    const int32_t* frame_idx;
    const float* inj_eps;  // nullable [n_iter][chains][L]
    const float* inj_u;    // nullable [n_iter][chains]
    uint32_t* n_accept;  // nullable
    float* a_trace;      // nullable [n_iter][chains]
    int64_t chains;
    int L, C, n_tiles, n_burn, n_keep;
    uint32_t seed_lo, seed_hi, iter0;
    const uint32_t* iter0_frame;  // nullable [NT]: per-frame iter0
    float sd;
};

// it = -1: initialise l(z) from the evaluation of the start state and draw proposal 0.
// it >= 0: accept/reject proposal `it`, record the kept sample, draw proposal it+1 (if any).
__global__ void __launch_bounds__(128) mh_step_kernel(MhArgs a, int it) {
    const int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (m >= a.chains) return;
    const int L = a.L;
    float* z = a.Z + m * L;
    float* zp = a.Zp + m * L;
    float ll_prop = 0.f;
    for (int t = 0; t < a.n_tiles; ++t) ll_prop += a.partial[m * a.n_tiles + t];

    if (it < 0) {
        a.ll_cur[m] = ll_prop;
    } else {
        float prior = 0.f;
        for (int l = 0; l < L; ++l) prior += __fsub_rn(__fmul_rn(z[l], z[l]), __fmul_rn(zp[l], zp[l]));
        const float acc_log = __fadd_rn(__fsub_rn(a.ll_cur[m], ll_prop), __fmul_rn(0.5f, prior));
        const float u = a.u_next[m];
        const bool accept = logf(u) < acc_log;
        if (a.a_trace) a.a_trace[(int64_t)it * a.chains + m] = acc_log;
        if (accept) {
            for (int l = 0; l < L; ++l) z[l] = zp[l];
            a.ll_cur[m] = ll_prop;
            if (a.n_accept) a.n_accept[m] += 1u;
        }
        if (it >= a.n_burn) {
            const int64_t fr = m / a.C;
            const int c = (int)(m - fr * a.C);
            float* dst = a.Zs + ((fr * a.C + c) * (int64_t)a.n_keep + (it - a.n_burn)) * L;
            for (int l = 0; l < L; ++l) dst[l] = z[l];
        }
    }
    const int nxt = it + 1;
    if (nxt < a.n_burn + a.n_keep) {
        float eps[DVAE_MAX_L];
        float u;
        if (a.inj_eps) {
            const float* e = a.inj_eps + ((int64_t)nxt * a.chains + m) * L;
            for (int l = 0; l < L; ++l) eps[l] = e[l];
            u = a.inj_u[(int64_t)nxt * a.chains + m];
        } else {
            const int64_t fr = m / a.C;
            const uint32_t c = (uint32_t)(m - fr * a.C);
            mh_draws(a.seed_lo, a.seed_hi, (uint32_t)a.frame_utt[fr], (uint32_t)a.frame_idx[fr] | (c << 20),
                     (a.iter0_frame ? a.iter0_frame[fr] : a.iter0) + (uint32_t)nxt, L, eps, u);
        }
        for (int l = 0; l < L; ++l) zp[l] = __fadd_rn(z[l], __fmul_rn(a.sd, eps[l]));
        a.u_next[m] = u;
    }
}

__global__ void copy_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

__global__ void rng_dump_kernel(uint32_t seed_lo, uint32_t seed_hi, uint32_t iter0, const uint32_t* __restrict__ iter0_frame,
                                const int32_t* __restrict__ frame_utt, const int32_t* __restrict__ frame_idx, int64_t chains, int C, int L, int n_iter,
                                float* __restrict__ eps_out, float* __restrict__ u_out) {
    const int64_t total = chains * n_iter;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int it = (int)(i / chains);
        const int64_t m = i - (int64_t)it * chains;
        const int64_t fr = m / C;
        const uint32_t c = (uint32_t)(m - fr * C);
        float eps[DVAE_MAX_L];
        float u;
        mh_draws(seed_lo, seed_hi, (uint32_t)frame_utt[fr], (uint32_t)frame_idx[fr] | (c << 20),
                 (iter0_frame ? iter0_frame[fr] : iter0) + (uint32_t)it, L, eps, u);
        for (int l = 0; l < L; ++l) eps_out[i * L + l] = eps[l];
        u_out[i] = u;
    }
}

// L % 4 == 0: one thread per Philox block (4 normals, one float4 store; consecutive threads write consecutive 16 bytes).
// Same counters and the same arithmetic as mh_draws, so the numbers are bit-identical to rng_dump_kernel.
// blockIdx.y = MH iteration, blockIdx.x covers chains * nb blocks: no 64-bit division on the index path.
__global__ void __launch_bounds__(256) rng_dump4_kernel(uint32_t seed_lo, uint32_t seed_hi, uint32_t iter0,
                                                        const uint32_t* __restrict__ iter0_frame, const int32_t* __restrict__ frame_utt, const int32_t* __restrict__ frame_idx,
                                                        uint32_t chains, uint32_t C, uint32_t nb_shift, float4* __restrict__ eps_out,
                                                        float* __restrict__ u_out) {
    const uint32_t it = blockIdx.y;
    const uint32_t per_it = chains << nb_shift;
    const uint32_t nb = 1u << nb_shift;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < per_it; j += gridDim.x * blockDim.x) {
        const uint32_t m = j >> nb_shift, b = j & (nb - 1);
        const uint32_t fr = (C == 1) ? m : m / C;
        const uint32_t c = (C == 1) ? 0u : m - fr * C;
        const uint32_t utt = (uint32_t)__ldg(frame_utt + fr), fc = (uint32_t)__ldg(frame_idx + fr) | (c << 20);
        const Philox4 r = philox4x32_10(utt, fc, (iter0_frame ? __ldg(iter0_frame + fr) : iter0) + it, b, seed_lo, seed_hi);
        float4 o;
        box_muller(r.x, r.y, o.x, o.y);
        box_muller(r.z, r.w, o.z, o.w);
        eps_out[(size_t)it * per_it + j] = o;
        if (b == 0) u_out[(size_t)it * chains + m] = u01_low_bytes(r);      // the accept uniform rides on block 0 (common.cuh)
    }
}

// box_muller on caller-supplied words; tests only (the float64 check of the normals over every 24-bit uniform)
__global__ void box_muller_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, float* __restrict__ n0,
                                  float* __restrict__ n1, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float x, y;
        box_muller(a[i], b[i], x, y);
        n0[i] = x;
        n1[i] = y;
    }
}

}  // namespace dvae

using namespace dvae;

extern "C" int64_t dvae_mlp_workspace_floats(const DvaeMlp* mlp, int64_t rows) {
    if (!mlp || rows <= 0) return 0;
    const int64_t r = rows < kRowChunk ? rows : kRowChunk;
    return 2 * r * (int64_t)max_hidden(mlp);
}

extern "C" int dvae_mlp_fwd(const DvaeMlp* mlp, const float* x, int ldx, int k1, const float* x2, int ldx2, int k2,
                            int x2_row_div, int64_t rows, int act_last, float* out, int ldo, float* ws, void* stream) {
    int rc = check_mlp(mlp, "dvae_mlp_fwd");
    if (rc) return rc;
    DVAE_REQUIRE(rows >= 0 && x && out, "dvae_mlp_fwd: bad rows/pointers");
    DVAE_REQUIRE(k1 >= 1 && k2 >= 0 && k1 + k2 == mlp->dims[0], "dvae_mlp_fwd: k1+k2=%d but the MLP takes %d inputs", k1 + k2, mlp->dims[0]);
    DVAE_REQUIRE(k2 == 0 || (x2 && ldx2 >= k2 && x2_row_div >= 1), "dvae_mlp_fwd: bad x2 arguments");
    DVAE_REQUIRE(ldx >= k1 && ldo >= mlp->dims[mlp->n_layers], "dvae_mlp_fwd: leading dimensions too small");
    DVAE_REQUIRE(act_last >= DVAE_ACT_NONE && act_last <= DVAE_ACT_EXP, "dvae_mlp_fwd: bad activation %d", act_last);
    DVAE_REQUIRE(mlp->n_layers == 1 || ws, "dvae_mlp_fwd: workspace required");
    DVAE_REQUIRE(k2 == 0 || x2_row_div <= kRowChunk, "dvae_mlp_fwd: x2_row_div too large");
    LoglikArgs none{};
    // row chunks are multiples of x2_row_div so every chunk starts on an x2 row boundary
    const int64_t div = (k2 > 0) ? x2_row_div : 1;
    const int64_t chunk = (kRowChunk / div) * div;
    for (int64_t r0 = 0; r0 < rows; r0 += chunk) {
        const int64_t r = (rows - r0 < chunk) ? rows - r0 : chunk;
        const float* x2c = (k2 > 0) ? x2 + (r0 / div) * ldx2 : nullptr;
        rc = run_mlp(mlp, x + r0 * ldx, ldx, k1, x2c, ldx2, k2, x2_row_div, r, act_last, out + r0 * ldo, ldo, none, ws,
                     (cudaStream_t)stream);
        if (rc) return rc;
    }
    return 0;
}

extern "C" int dvae_reparam(const float* mu, const float* log_var, const float* eps, float* z, int64_t n, void* stream) {
    DVAE_REQUIRE(mu && log_var && eps && z && n >= 0, "dvae_reparam: bad arguments");
    if (n == 0) return 0;
    const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
    reparam_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(mu, log_var, eps, z, n);
    return check_launch("reparam_kernel");
}

static int64_t mh_tiles(int F) { return (F + BN - 1) / BN; }

extern "C" int64_t dvae_mh_workspace_floats(const DvaeMlp* dec, int64_t chains, int F) {
    if (!dec || chains <= 0) return 0;
    // hidden ping-pong + proposals + l(z) + pending uniforms + per-tile partials
    return 2 * chains * (int64_t)max_hidden(dec) + chains * (int64_t)DVAE_MAX_L + 2 * chains + chains * mh_tiles(F);
}

extern "C" int dvae_mh_chain_f32(const DvaeMlp* dec, const float* P, const float* Vb, const float* g, const float* y,
                                 int y_dim, const int32_t* frame_utt, const int32_t* frame_idx, float* Z, float* Zs,
                                 int64_t NT, int F, int ld, int L, int n_chains, int n_burn, int n_keep, float var_rw,
                                 const DvaeRng* rng, uint32_t* n_accept, float* a_trace, float* ws, void* stream) {
    int rc = check_mlp(dec, "dvae_mh_chain_f32");
    if (rc) return rc;
    DVAE_REQUIRE(P && Vb && g && Z && Zs && ws && rng, "dvae_mh_chain_f32: null pointer");
    DVAE_REQUIRE(NT >= 0 && F >= 1 && ld >= F, "dvae_mh_chain_f32: bad sizes");
    DVAE_REQUIRE(L >= 1 && L <= DVAE_MAX_L, "dvae_mh_chain_f32: L=%d out of range", L);
    DVAE_REQUIRE(y_dim >= 0 && (y_dim == 0 || y), "dvae_mh_chain_f32: y_dim=%d but y is null", y_dim);
    DVAE_REQUIRE(dec->dims[0] == L + y_dim, "dvae_mh_chain_f32: decoder takes %d inputs, L+y_dim=%d", dec->dims[0], L + y_dim);
    DVAE_REQUIRE(dec->dims[dec->n_layers] == F, "dvae_mh_chain_f32: decoder emits %d bins, F=%d", dec->dims[dec->n_layers], F);
    DVAE_REQUIRE(n_chains >= 1 && n_chains < 4096, "dvae_mh_chain_f32: n_chains=%d", n_chains);
    DVAE_REQUIRE(n_burn >= 0 && n_keep >= 1, "dvae_mh_chain_f32: bad schedule");
    DVAE_REQUIRE(var_rw > 0.f, "dvae_mh_chain_f32: var_rw must be positive");
    DVAE_REQUIRE((rng->eps == nullptr) == (rng->u == nullptr), "dvae_mh_chain_f32: eps and u must be injected together");
    DVAE_REQUIRE(!(rng->eps && rng->iter0_frame), "dvae_mh_chain_f32: iter0_frame applies to Philox draws only");
    DVAE_REQUIRE(rng->eps || (frame_utt && frame_idx), "dvae_mh_chain_f32: Philox mode needs frame_utt/frame_idx");
    if (NT == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t chains = NT * n_chains;
    const int mh = max_hidden(dec);
    const int n_tiles = (int)mh_tiles(F);
    float* hid = ws;
    float* Zp = hid + 2 * chains * (int64_t)mh;
    float* ll_cur = Zp + chains * (int64_t)DVAE_MAX_L;
    float* u_next = ll_cur + chains;
    float* partial = u_next + chains;

    MhArgs a{};
    a.Z = Z; a.Zp = Zp; a.ll_cur = ll_cur; a.u_next = u_next; a.partial = partial; a.Zs = Zs;
    a.frame_utt = frame_utt; a.frame_idx = frame_idx; a.inj_eps = rng->eps; a.inj_u = rng->u;
    a.n_accept = n_accept; a.a_trace = a_trace; a.chains = chains; a.L = L; a.C = n_chains; a.n_tiles = n_tiles;
    a.n_burn = n_burn; a.n_keep = n_keep;
    a.seed_lo = (uint32_t)(rng->seed & 0xffffffffu); a.seed_hi = (uint32_t)(rng->seed >> 32); a.iter0 = rng->iter0;
    a.iter0_frame = rng->iter0_frame;
    a.sd = sqrtf(var_rw);

    LoglikArgs ll{P, Vb, g, partial, ld, n_chains, n_tiles};
    const int grid_c = (int)((chains + 127) / 128);
    const int n_iter = n_burn + n_keep;
    for (int it = -1; it < n_iter; ++it) {
        // evaluate l(.) at the start state (it = -1) or at proposal `it`
        const float* in = (it < 0) ? Z : Zp;
        rc = run_mlp(dec, in, L, L, y, y_dim, y_dim, n_chains, chains, EPI_LOGLIK, nullptr, 0, ll, hid, st);
        if (rc) return rc;
        mh_step_kernel<<<grid_c, 128, 0, st>>>(a, it);
        rc = check_launch("mh_step_kernel");
        if (rc) return rc;
    }
    return 0;
}

extern "C" int dvae_rng_dump(const DvaeRng* rng, const int32_t* frame_utt, const int32_t* frame_idx, int64_t NT,
                             int n_chains, int L, int n_iter, float* eps, float* u, void* stream) {
    DVAE_REQUIRE(rng && frame_utt && frame_idx && eps && u, "dvae_rng_dump: null pointer");
    DVAE_REQUIRE(NT >= 0 && n_chains >= 1 && L >= 1 && L <= DVAE_MAX_L && n_iter >= 0, "dvae_rng_dump: bad sizes");
    DVAE_REQUIRE(n_chains < 4096, "dvae_rng_dump: n_chains=%d (the chain index has 12 bits of the counter)", n_chains);
    const int64_t total = NT * n_chains * n_iter;
    if (total == 0) return 0;
    if ((L == 4 || L == 8 || L == 16 || L == 32 || L == 64) && (reinterpret_cast<uintptr_t>(eps) & 15) == 0 && n_iter <= 65535 &&
        NT * n_chains * (L / 4) < (1ll << 31)) {
        const uint32_t chains = (uint32_t)(NT * n_chains);
        uint32_t nb_shift = 0;
        while ((4 << nb_shift) < L) ++nb_shift;
        const uint32_t per_it = chains << nb_shift;
        const uint32_t bx = (per_it + 255) / 256;
        rng_dump4_kernel<<<dim3(bx < 4096 ? bx : 4096, n_iter), 256, 0, (cudaStream_t)stream>>>(
            (uint32_t)(rng->seed & 0xffffffffu), (uint32_t)(rng->seed >> 32), rng->iter0, rng->iter0_frame, frame_utt, frame_idx, chains,
            (uint32_t)n_chains, nb_shift, reinterpret_cast<float4*>(eps), u);
        return check_launch("rng_dump4_kernel");
    }
    const int grid = (int)((total + 127) / 128 < 148 * 16 ? (total + 127) / 128 : 148 * 16);
    rng_dump_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>((uint32_t)(rng->seed & 0xffffffffu), (uint32_t)(rng->seed >> 32),
                                                           rng->iter0, rng->iter0_frame, frame_utt, frame_idx, NT * n_chains, n_chains, L,
                                                           n_iter, eps, u);
    return check_launch("rng_dump_kernel");
}

extern "C" int dvae_box_muller_f32(const uint32_t* a, const uint32_t* b, float* n0, float* n1, int64_t n, void* stream) {
    DVAE_REQUIRE(a && b && n0 && n1 && n >= 0, "dvae_box_muller_f32: bad arguments");
    if (n == 0) return 0;
    const int64_t blocks = (n + 255) / 256;
    box_muller_kernel<<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), 256, 0, (cudaStream_t)stream>>>(a, b, n0, n1, n);
    return check_launch("box_muller_kernel");
}
