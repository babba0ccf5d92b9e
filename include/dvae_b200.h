/*
 * libdvae_b200 -- C ABI of the B200-native (sm_100a) MCEM VAE-NMF speech-enhancement hot path.
 *
 * The reference (sp-uhh/disentangled-vae) has no FFI layer: its "operator API" for this path is the Python call
 * surface used by scripts/evaluate_ntcd_{M1,M2,M2_info_vad}.py and scripts/reconstruct_*.py.  This header is the
 * boundary a maintainer binds instead (ctypes stub in INTEGRATION.md); every entry point names the reference
 * code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer on the current CUDA device unless marked [host];
 *   - the caller owns every buffer; the library never allocates device memory (workspace sizes are queried);
 *   - all work is enqueued on the passed stream (a cudaStream_t passed as void*); nothing synchronises;
 *   - return 0 = OK, DVAE_ERR_ARG (<0) = argument error detected before any launch, >0 = cudaError_t;
 *     dvae_last_error() returns a thread-local description of the last non-zero return;
 *   - there is no CPU fallback: the library only contains sm_100a code.
 *
 * Batch layout ("frame-major, ragged")
 *   A batch holds B utterances; utterance u owns frames [fr_off[u], fr_off[u+1]) of NT = fr_off[B] frames in total.
 *   Per-frame spectra are rows of `ld` floats (ld >= F, ld % 4 == 0; the library's Python host uses ld = 520 for
 *   F = 513): X[NT][ld] (float2), P[NT][ld], Vb[NT][ld], Vs[NT][R][ld].  Latents are Z[NT*C][L] (C chains per
 *   frame), kept samples Zs[NT][C*R][L], labels y[NT][y_dim], activations H[NT][K], gains g[NT], and the
 *   per-utterance dictionaries W[B][K][ld].  The reference's (F,N) / (K,N) / (L,N) matrices are the transposes of
 *   one utterance's slice.
 */
#ifndef DVAE_B200_H
#define DVAE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVAE_ABI_VERSION 4          /* 4: dvae_decode_wiener_tc replaces dvae_decode_a1_tc + dvae_wiener_from_a1 */
#define DVAE_ERR_ARG (-1)
#define DVAE_MAX_LAYERS 6
#define DVAE_MAX_L 64          /* latent dimension limit of the Metropolis-Hastings kernels */
#define DVAE_MAX_K 16          /* NMF rank limit */

/* bits of the device status word (`int* status`) some entry points take: it is OR-ed into, never cleared by the library */
#define DVAE_STATUS_TIMEOUT 1      /* a tcgen05 kernel's internal pipeline wait ran out: results invalid */
#define DVAE_STATUS_NONFINITE 2    /* NaN / Inf guard: a chain's log-likelihood or an utterance's cost was not finite */

/* activation applied after the LAST layer of dvae_mlp_fwd (hidden layers are always tanh, models.py:102-104,119-121) */
#define DVAE_ACT_NONE 0
#define DVAE_ACT_TANH 1
#define DVAE_ACT_EXP 2

/* A tanh MLP (Encoder trunk + one head, or Decoder) with transposed weights:
 * wt[i] is [dims[i]][dims[i+1]] row-major = nn.Linear(dims[i], dims[i+1]).weight.T, bias[i] is [dims[i+1]].
 * Replaces packages/models/models.py:91-105 (Encoder), 108-122 (Decoder).  The struct lives in HOST memory. */
typedef struct DvaeMlp {
    int32_t n_layers;
    int32_t dims[DVAE_MAX_LAYERS + 1];
    const float* wt[DVAE_MAX_LAYERS];
    const float* bias[DVAE_MAX_LAYERS];
} DvaeMlp;

/* Random draws of the Metropolis-Hastings sampler.  Either counter-based Philox-4x32-10 keyed by `seed`
 * (eps == NULL) or injected draws (parity runs): eps[it][NT*C][L] standard normals and u[it][NT*C] uniforms,
 * `it` counting the iterations of THIS call from 0.  Struct in HOST memory.  (mcem.py:243,256) */
typedef struct DvaeRng {
    uint64_t seed;
    uint32_t iter0;            /* global iteration number of this call's first iteration (Philox counter word 2) */
    uint32_t reserved;
    const float* eps;          /* nullable */
    const float* u;            /* nullable; required when eps is given */
    const uint32_t* iter0_frame;   /* nullable [NT] (device): per-frame replacement of iter0, so frames whose EM loops stopped
                                      at different iterations draw their own counters in one call; Philox mode only */
} DvaeRng;

int dvae_version(void);
const char* dvae_last_error(void);

/* ---- STFT: packages/processing/stft.py:13-60 (librosa.core.stft, center=False, periodic Hann, n_fft=1024) ----
 * x: concatenated float32 signals; utterance u = x[x_off[u] .. x_off[u]+x_len[u]).  Frame j covers samples
 * [j*hop, j*hop+n_fft) with zeros past x_len[u] (this realises the end-padding rule of stft.py:45-50; the caller
 * chooses the frame count).  Writes X[fr_off[u]+j][0..F) (complex64) and, if P != NULL, P = |X|^2 (mcem.py:47).
 * Accuracy (tests/test_gpu_stft_f64.py, bounds derived in oracle/stft_mirror.py, u = 2^-24): against the float64 rfft of
 * x * hann, every bin is within 93 u * sum_n |x_n w_n| of its frame, and every frame within 97 u * ||X||_2 in the 2-norm.
 * The per-bin bound is relative to the frame's sum |x w|, not to the bin: a bin far below its frame's peak carries the
 * frame's absolute rounding floor, whereas the reference (a float64 FFT stored as complex64) is relative-accurate in
 * every bin.  P is within the X error carried through, plus 2 u P, plus 2^-148 (subnormal results are kept). */
int dvae_stft_f32(const float* x, const int64_t* x_off, const int32_t* x_len, int B, void* X /* float2 */, float* P,
                  const int64_t* fr_off, int64_t NT, int n_fft, int hop, int ld, void* stream);

/* ---- ISTFT: packages/processing/stft.py:63-99 (librosa.core.istft, center=False, length=max_len) ----
 * y[y_off[u] .. +y_len[u]) <- overlap-add of window * irfft(frame), divided by the float32 sum of squared windows
 * where that sum exceeds FLT_MIN, zero beyond n_fft + hop*(N_u-1).  max_y_len = max_u y_len[u] (grid sizing).
 * Accuracy (tests/test_gpu_stft_f64.py, oracle/stft_mirror.py): every sample is within its own bound of the float64
 * overlap-add divided by the float32 window sum-square: per covering frame, 92 u * sum |Hermitian-extended spectrum| / 1024
 * times the window, the window and float32 overlap-add roundings, then divided by the window sum-square (so the bound grows
 * near the first and last samples, where that sum is small), plus 2 u |y|.  The Im parts of bins 0 and 512 are ignored,
 * sample 0 and the samples past the natural length are exactly 0, and a sample's value does not depend on B, the batch
 * order or y_off (bit-identical). */
int dvae_istft_f32(const void* X /* float2 */, const int64_t* fr_off, int B, float* y, const int64_t* y_off,
                   const int32_t* y_len, int max_y_len, int n_fft, int hop, int ld, void* stream);

/* ---- Wiener filter fused into the ISTFT: mcem.py:176-177 (S_hat = WFs * X) followed by stft.py:63-99 ----
 * Same as dvae_istft_f32 on the spectrum (mask[n][f] * mask_scale) * X[n][f] (real mask, row pitch ld), formed in
 * registers while the frame is loaded: bit-identical to dvae_wiener_apply + dvae_istft_f32 without the S_hat / N_hat
 * round trip through HBM (BASELINE.json configs[4]).  Accuracy as dvae_istft_f32, plus 2 u |mask * X| per bin (the two
 * products). */
int dvae_istft_masked_f32(const void* X /* float2 */, const float* mask, float mask_scale, const int64_t* fr_off, int B,
                          float* y, const int64_t* y_off, const int32_t* y_len, int max_y_len, int n_fft, int hop, int ld,
                          void* stream);

/* ---- dense tanh MLP: models.py:102-105 (Encoder trunk + head) and 119-122 (Decoder) ----
 * out[r][0..dims[n_layers]) = act_last(Linear_n(tanh(... tanh(Linear_1([x[r] ; x2[r / x2_row_div]])))))
 * x: rows x k1 (row stride ldx); x2 (nullable): k2 extra input columns (labels y), row r uses x2 row r / x2_row_div.
 * ws: workspace of dvae_mlp_workspace_floats(mlp, rows) floats. */
int64_t dvae_mlp_workspace_floats(const DvaeMlp* mlp, int64_t rows);
int dvae_mlp_fwd(const DvaeMlp* mlp, const float* x, int ldx, int k1, const float* x2, int ldx2, int k2, int x2_row_div,
                 int64_t rows, int act_last, float* out, int ldo, float* ws, void* stream);

/* z = mu + exp(0.5*log_var)*eps   (models.py:8-22) */
int dvae_reparam(const float* mu, const float* log_var, const float* eps, float* z, int64_t n, void* stream);

/* P[i] = |X[i]|^2 over n complex64 elements (mcem.py:47, for spectrograms handed in by the caller) */
int dvae_power(const void* X /* float2 */, float* P, int64_t n, void* stream);

/* ---- NMF noise model: mcem.py:36-58, 76-83, 91-153, 69-71 ---- */
/* Vb[n][f] = sum_k W[utt(n)][k][f] * H[n][k]   (compute_Vb, mcem.py:82-83) */
int dvae_nmf_vb(const float* W, const float* H, const int32_t* frame_utt, int64_t NT, int F, int K, int ld, float* Vb,
                void* stream);

/* One M-step (mcem.py:91-153) + cost (mcem.py:69-71) on materialised speech variances Vs[NT][R][ld]:
 *   W <- W*sqrt(((P*sum_r Vx^-2) H^T)/((sum_r Vx^-1) H^T)), Vb,Vx refreshed;  H likewise with W^T;  Vb,Vx refreshed;
 *   W <- W/||W||_1col, H <- H*||W||_1col (Vb NOT recomputed);  g <- g*sqrt(sum_f P sum_r Vs Vx^-2 / sum_f sum_r Vs Vx^-1);
 *   cost[u] = mean_{r,f,n in u}(log Vx + P/Vx) with the new g.
 * In/out: W[B][K][ld], H[NT][K], g[NT], Vb[NT][ld] (in: product used by the E-step; out: W_new H_new before
 * normalisation, as the reference keeps it).  cost: [B] doubles, overwritten.
 * ws: dvae_nmf_workspace_floats(B, K, ld, max_frames) floats, 8-byte aligned.
 * Supported input range (this entry point, dvae_nmf_mstep_vst and the dvae_vst_* statistics passes; DESIGN section 6): every
 * Vx = g Vs + Vb the M-step forms (E-step g and Vb, then W_new H_old, W_new H_new, g_new) lies in [2^-60, 2^60], and the
 * samples of a bin lie within 2^+-31 of the bin's first sample.  Inside, every output is within the error model of
 * tests/test_gpu_mstep_f64.py of float64.  Below 2^-63 the pair products x0 x1 of the shared reciprocals leave FP32's normal
 * range, above 2^63 their reciprocal does; a wider spread overflows the cost passes' products of four samples: such inputs end
 * in DVAE_STATUS_NONFINITE or, on the generic (IEEE reciprocal) kernels, in results that still meet the bound. */
int64_t dvae_nmf_workspace_floats(int B, int K, int ld, int max_frames);
int dvae_nmf_mstep(const float* P, const float* Vs, int R, float* W, float* H, float* g, float* Vb, double* cost,
                   const int64_t* fr_off, const int32_t* frame_utt, int B, int64_t NT, int F, int K, int ld,
                   int max_frames /* max_u frames of one utterance, for grid sizing */, float* ws,
                   const float* wstat /* nullable: frame statistics A1 | A2 (dvae_decode_stats_tc), replace the pass over Vs of
                                         the W update */,
                   int* status /* nullable: DVAE_STATUS_NONFINITE is OR-ed in when a cost is not finite */, void* stream);

/* ---- Metropolis-Hastings E-step sampler: mcem.py:207-277 / 372-448 / 544-620 / 716-792 ----
 * FP32 CUDA-core decoder ("exact" mode).  Runs n_burn + n_keep random-walk iterations on every (frame, chain):
 *   z' = z + sqrt(var_rw)*eps;  a = sum_f[log Vx - log Vx' + (1/Vx - 1/Vx')P] + .5 sum_l(z^2 - z'^2),  Vx = g*D(z)+Vb;
 *   accept iff log(u) < a.
 * Z[NT*C][L] in: chain starts, out: last states.  Zs[NT][C*n_keep][L]: kept samples, chain c sample r at slot c*n_keep+r.
 * frame_utt / frame_idx [NT]: Philox counter words (global utterance id, frame index inside the utterance).
 * n_accept (nullable): [NT*C] accepted-proposal counters, incremented.  a_trace (nullable): [n_iter][NT*C] log ratios.
 * ws: dvae_mh_workspace_floats(dec, NT*C) floats. */
int64_t dvae_mh_workspace_floats(const DvaeMlp* dec, int64_t chains, int F);
int dvae_mh_chain_f32(const DvaeMlp* dec, const float* P, const float* Vb, const float* g, const float* y, int y_dim,
                      const int32_t* frame_utt, const int32_t* frame_idx, float* Z, float* Zs, int64_t NT, int F, int ld,
                      int L, int n_chains, int n_burn, int n_keep, float var_rw, const DvaeRng* rng, uint32_t* n_accept,
                      float* a_trace, float* ws, void* stream);

/* The draws the Philox mode of dvae_mh_chain_* consumes, dumped as eps[n_iter][NT*C][L], u[n_iter][NT*C]
 * (so a parity test can inject the very same draws into the reference / oracle). */
int dvae_rng_dump(const DvaeRng* rng, const int32_t* frame_utt, const int32_t* frame_idx, int64_t NT, int n_chains,
                  int L, int n_iter, float* eps, float* u, void* stream);

/* ---- Wiener filter: mcem.py:310-329 + 176-177 ----
 * accumulate: WFs[n][f] += sum_r g*Vs/Vx, WFn[n][f] += sum_r Vb/Vx over the R samples present in Vs[NT][R][ld];
 * apply: S_hat = X*WFs/R_total, N_hat = X*WFn/R_total (complex64). */
int dvae_wiener_accum(const float* Vs, int R, const float* Vb, const float* g, int64_t NT, int F, int ld, float* WFs,
                      float* WFn, int first /* 1: overwrite instead of add */, void* stream);
int dvae_wiener_apply(const void* X, const float* WFs, const float* WFn, int R_total, int64_t NT, int F, int ld,
                      void* S_hat, void* N_hat, void* stream);

/* ---- tensor-core (tcgen05, BF16 x BF16 -> FP32) decoder path: mcem.py:207-277 + 280-290 over models.py:119-122 ----
 * Specialised for F = 513 bins, hidden width 128, 1 or 2 hidden layers, 2L + 2*y_dim + 1 <= 128.
 * dvae_tc_pack_decoder builds the shared-memory image of the decoder (UMMA K-major 128B-swizzled BF16 operands +
 * FP32 biases; W3/b3 pre-scaled by log2 e) into `image` (dvae_tc_image_bytes bytes, 16-byte aligned).
 * dvae_decode_tc: Vs[r][0..F) = decoder([Zs[r]; y[r / x2_row_div]]) for any number of rows; *status: DVAE_STATUS_* bits.
 *
 * Label inputs.  Up to three labels per frame ride in the layer-1 operand (y, y_dim <= 3).  Wider label vectors -- the
 * IBM-conditioned M2 model has y_dim = 513 (scripts/evaluate_ntcd_M2.py:66-73) -- are folded into a PER-FRAME layer-1 bias
 * instead: the caller packs the decoder WITHOUT its label columns and without its layer-1 bias (dims[0] = L, y_dim = 0) and
 * passes ybias[frame][128] = W1[:, L:] y[frame] + b1 (one dvae_mlp_fwd over the frames; the labels do not change during a
 * run), which every tensor-core kernel adds to the layer-1 pre-activation of the frame's rows.  ybias == NULL: no such bias. */
int64_t dvae_tc_image_bytes(const DvaeMlp* dec, int L, int y_dim);
int dvae_tc_pack_decoder(const DvaeMlp* dec, int L, int y_dim, void* image, void* stream);
int dvae_decode_tc(const DvaeMlp* dec, const void* image, const float* Zs, int64_t rows, int L, const float* y, int y_dim,
                   const float* ybias /* nullable: [rows / x2_row_div][128] */, int x2_row_div, float* Vs, int ld, int* status,
                   void* stream);

/* The Metropolis-Hastings sampler on tensor cores: same contract as dvae_mh_chain_f32 (Z, Zs, frame_utt / frame_idx,
 * rng, n_accept, a_trace); L in {16, 32}, y_dim <= 3.  Draws: counter-based Philox inside the kernel (rng->eps == NULL,
 * the counters of every sampler of this library) or injected eps / u (16-byte aligned).  P and Vb are streamed at BF16
 * precision (dvae_tc_pack_pv: [tile][bin quad][128 chains] x 4 words, word j = P'_j with bf16(Vb'_j) as its low half, the
 * layer-3 bias of `image` folded in as a per-bin scale; dvae_tc_packed_pv_bytes bytes).
 * Emission (VsT, vs_idx non-NULL; n_keep <= 31): the decoder output of the kept samples -- compute_Vs, mcem.py:280-290 --
 * is written by the sampler itself, in BF16 and WITHOUT the output-layer bias E[f] = exp(b3[f]):
 *   VsT[tile = chain / 128][slot 0..n_keep][bg = bin / 16 (33)][row = chain % 128][16] bf16  (dvae_vst_bytes bytes, 32-byte aligned),
 *   vs_idx[chain][32] bytes: byte r = slot of kept sample r, i.e. Vs[chain][r][f] = E[f] VsT[..][vs_idx[chain][r]][..].
 * flags: DVAE_TC_POLY_EX2 lets the sampler evaluate half of the layer-3 exponentials with a polynomial on the FMA pipe
 * (relative error 7.5e-5) instead of MUFU.EX2; only valid when the pre-activation stays inside +-120 in the log2
 * domain, i.e. when dvae_tc_decoder_exponent_bound (a one-off, synchronising query: log2(e) * max_f sum_k |W3[k][f]|)
 * reports less than DVAE_TC_POLY_EX2_LIMIT for the decoder.
 * *status: DVAE_STATUS_TIMEOUT / DVAE_STATUS_NONFINITE are OR-ed in. */
#define DVAE_TC_POLY_EX2 1
#define DVAE_TC_POLY_EX2_ALL 2      /* all layer-3 exponentials from the polynomial (same validity condition) */
#define DVAE_TC_POLY_EX2_LIMIT 120.0f
int64_t dvae_tc_packed_pv_bytes(int64_t chains);
/* kscale[NT] (nullable everywhere: 2^15): a power of two per frame that centres the sampler's four-fold variance products in
 * the FP32 range for THIS frame's spectrum and THIS decoder's output bias; dvae_tc_row_scale derives it once per batch from
 * P (k = 2^-2c, 2^c = 2^-16 x the frame's loudest bin of P 2^-b); the stream must be packed and sampled with the same array.  dvae_tc_pack_pv keeps
 * every factor of those products within 30 octaves of the frame's level 2^c: it floors Vb' at 2^(c-30) (90 dB below the frame,
 * identical under l(z) and l(z'), in bins that carry no energy) and packs the observation-free padding bins 513..543 as the
 * constant 1 in the quad's scale, so that a collapsed gain g or a spectral null cannot underflow the product. */
int dvae_tc_row_scale(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* P, int64_t NT, int F, int ld,
                      float* kscale, void* stream);
int dvae_tc_pack_pv(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* P, const float* Vb,
                    const float* kscale, int64_t NT, int n_chains, int F, int ld, void* dst, void* stream);
int dvae_tc_decoder_exponent_bound(const DvaeMlp* dec, int L, int y_dim, float* bound_host, void* stream);
/* Byte offset inside the decoder image of the FP32 layer-3 bias in the log2 domain (b3 * log2 e, the per-bin scale the P / Vb
 * stream is packed with), or -1. */
int64_t dvae_tc_image_bias_offset(const DvaeMlp* dec, int L, int y_dim);
/* The samplers' hidden-layer activation (tanh.approx.bf16x2 on the BF16-rounded pre-activation) as a table over every input:
 * out[x] (65536 BF16 bit patterns, device memory) = the activation of the BF16 number with bit pattern x.  For parity tests:
 * the instruction is not the correctly rounded tanh. */
int dvae_tc_tanh_bf16_table(uint16_t* out, void* stream);
/* y[i] = tanh.approx.f32(x[i]), the activation of the decode kernels' hidden layers (tests: the float64 mirror's activation) */
int dvae_tc_tanh_f32(const float* x, float* y, int64_t n, void* stream);
/* (n0[i], n1[i]) = the samplers' Box-Muller normals of the Philox words (a[i], b[i]) (csrc/common.cuh box_muller); tests only */
int dvae_box_muller_f32(const uint32_t* a, const uint32_t* b, float* n0, float* n1, int64_t n, void* stream);
int64_t dvae_vst_bytes(int64_t chains, int n_keep);
int dvae_mh_chain_tc2(const DvaeMlp* dec, const void* image, const void* PVpk, const float* kscale, const float* g, const float* y, int y_dim,
                      const float* ybias /* nullable: [NT][128] */, const int32_t* frame_utt, const int32_t* frame_idx, float* Z,
                      float* Zs, int64_t NT, int L,
                      int n_chains, int n_burn, int n_keep, float var_rw, const DvaeRng* rng, uint32_t* n_accept,
                      float* a_trace, void* VsT /* nullable */, uint8_t* vs_idx /* nullable */, int flags, int* status,
                      void* stream);

/* Consumers of the emission.  n_chains = 1: chain = frame.  n_chains = 2^c <= 128 (dvae_vst_w_partials, dvae_nmf_mstep_vst,
 * R = kept samples PER CHAIN): chain row m belongs to frame m / n_chains, the frame's n_chains x R samples enter every sum, the
 * segment tables are cut on the chain-row axis (tile boundaries and n_chains x the utterances' frame offsets) and the M-step
 * needs wpart; dvae_vst_unpack with NT = the number of chain rows gives Vs[NT][n_chains * R][ld].
 * dvae_vst_frame_stats: A1[n][f] = sum_r 1/Vx, A2[n][f] = sum_r 1/Vx^2 with Vx = g[n] Vs[n][r][f] + Vb[n][f]: the inner
 *   sums of the W update (mcem.py:108-110); R <= 31.
 * dvae_vst_w_partials: the same pass, but instead of writing A1 / A2 it multiplies them with the activations H and reduces over
 *   the frames of every SEGMENT (a maximal run of frames inside one 128-frame tile and one utterance; seg_start[S+1] ascending
 *   frame boundaries, tile_seg[n_tiles+1] first segment per tile): Wpart[seg][k][0|1][f] = sum_n P A2 H | sum_n A1 H
 *   (dvae_vst_w_partial_floats floats).  dvae_nmf_w_from_partials sums an utterance's segments (utt_seg[B+1]) in order and
 *   applies the W update; deterministic, and the A1 / A2 round trip through memory disappears.
 * dvae_nmf_mstep_vst: dvae_nmf_mstep on the emission (F = 513, ld = 520, K <= 10, R in {10, 30}); exactly one of
 *   fstat = A1 | A2 (A2 = A1 + NT*ld, from dvae_vst_frame_stats) and wpart (+ utt_seg, from dvae_vst_w_partials).
 * dvae_vst_unpack / dvae_vst_pack: conversion to / from dense FP32 Vs[NT][R][ld] (pack: sample r -> slot 1 + r). */
int dvae_vst_frame_stats(const DvaeMlp* dec, const void* image, int L, int y_dim, const void* VsT, const uint8_t* vs_idx,
                         int R, const float* Vb, const float* g, int64_t NT, int ld, float* A1, float* A2, void* stream);
int dvae_nmf_mstep_vst(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* P, const void* VsT,
                       const uint8_t* vs_idx, int R, float* W, float* H, float* g, float* Vb, double* cost,
                       const int64_t* fr_off, int B, int64_t NT, int K, int ld, int max_frames, float* ws,
                       const float* fstat /* nullable */, const float* wpart /* nullable */, const int32_t* utt_seg, int n_chains,
                       int* status, void* stream);
int64_t dvae_vst_w_partial_floats(int64_t n_segments, int K, int ld);
int dvae_vst_w_partials(const DvaeMlp* dec, const void* image, int L, int y_dim, const void* VsT, const uint8_t* vs_idx, int R,
                        const float* P, const float* Vb, const float* g, const float* H, int K, int64_t NT, int n_chains, int ld,
                        const int64_t* seg_start, const int32_t* tile_seg, float* Wpart, void* stream);
int dvae_nmf_w_from_partials(const float* Wpart, const int32_t* utt_seg, const float* W, int B, int F, int K, int ld, float* Wtmp,
                             void* stream);
int dvae_vst_unpack(const DvaeMlp* dec, const void* image, int L, int y_dim, const void* VsT, const uint8_t* vs_idx, int R,
                    int64_t NT, int ld, float* Vs, void* stream);
int dvae_vst_pack(const DvaeMlp* dec, const void* image, int L, int y_dim, const float* Vs, int R, int64_t NT, int ld,
                  void* VsT, uint8_t* vs_idx, void* stream);

/* Warp-specialised decode with per-frame statistics (R in {10,30}): writes FP32 Vs[NT][R][ld], A1[n][f] = sum_r 1/Vx and
 * A2[n][f] = sum_r 1/Vx^2; dvae_nmf_mstep takes them as wstat = A1 (A2 = A1 + NT*ld).  Used when the sampler's emission
 * does not apply (several chains per frame, injected kept samples). */
int dvae_decode_stats_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R, int L, const float* y, int y_dim,
                         const float* ybias /* nullable */, const float* Vb, const float* g, int64_t NT, int ld, float* Vs, float* A1, float* A2, int* status,
                         void* stream);
/* dvae_decode_stats_tc for frames that hold R_total samples (multi-chain runs): decodes the window r0 .. r0+R (R in {10, 30}),
 * writes the rows n * R_total + r0 + r of Vs and overwrites (accumulate == 0) or adds to A1 / A2 */
int dvae_decode_stats_win_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R_total, int r0, int R, int L,
                             const float* y, int y_dim, const float* ybias /* nullable */, const float* Vb, const float* g, int64_t NT, int ld, float* Vs, float* A1,
                             float* A2, int accumulate, int* status, void* stream);
/* Final filter without materialising its samples: dvae_decode_wiener_tc decodes the samples r0 .. r0+R (R in {10, 25, 30}) of
 * every frame of Zs [NT][R_total][L] and writes the mask sums of compute_WF (mcem.py:325-327) for them, overwriting
 * (accumulate == 0) or adding to WFs / WFn [NT][ld]:  WFs = g sum_r Vs / Vx,  WFn = Vb sum_r 1 / Vx.  Both sums are
 * accumulated term by term (positive terms: FP32 relative precision in every bin, however small g Vs is against Vb).
 * Supported range (this entry point, dvae_decode_stats_tc and dvae_decode_stats_win_tc; DESIGN section 6): every
 * Vx = g Vs + Vb in [2^-60, 2^60], as for the M-step (the margin of 2^3 keeps A2 = sum_r Vx^-2 finite for R <= 256).
 * Inside, Vs, A1 / A2 and the mask sums are within the error model of tests/test_gpu_decode_f64.py of float64.  Outside,
 * the shared reciprocal of a pair of samples leaves FP32's normal range (at 2^-63 / 2^63): below, the pair product
 * underflows, A1 / A2 / the mask sums become Inf or NaN and DVAE_STATUS_NONFINITE is OR-ed into *status; above, the pair
 * product overflows, its reciprocal flushes to zero and those samples drop out of A1 / A2 / the sums: finite, too small,
 * no status bit. */
int dvae_decode_wiener_tc(const DvaeMlp* dec, const void* image, const float* Zs, int R_total, int r0, int R, int L, const float* y,
                          int y_dim, const float* ybias /* nullable */, const float* Vb, const float* g, int64_t NT, int ld, float* WFs,
                          float* WFn, int accumulate, int* status, void* stream);
/* W <- W sqrt(num / den), num[f,k] = sum_n P A2 H, den[f,k] = sum_n A1 H (mcem.py:108-111); Wtmp: un-normalised result */
int dvae_nmf_w_from_frame_stats(const float* A1, const float* A2, const float* P, const float* H, const float* W,
                                const int64_t* fr_off, int B, int F, int K, int ld, float* Wtmp, void* stream);

/* ---- evaluation metric on the device (packages/metrics.py:12-82: si_sdr_components, energy_ratios, si_sdr_leroux) ----
 * Ragged batch: utterance u occupies [off[u], off[u] + len[u]) of s_hat / s / n (n nullable).  out[u] = {SI-SDR, SI-SIR,
 * SI-SAR} in dB (float64, inner products accumulated in double); SI-SIR / SI-SAR are NaN when n is null, SI-SDR then
 * equals si_sdr_leroux. */
int dvae_energy_ratios(const float* s_hat, const float* s, const float* n, const int64_t* off, const int32_t* len, int B,
                       double* out, void* stream);

/* ---- 16-bit PCM quantisation (batch_io.write_wav: np.clip(np.rint(x * 32768), -32768, 32767).astype("<i2")) ----
 * Over the flat buffer x[0..n): q = clamp(rint(x * 32768), -32768, 32767), round half to even, +-Inf saturating, NaN -> 0.
 * pcm[i] = q (the samples of the wav file) and xq[i] = q / 32768 (what read_wav returns for it, exact in FP32); either
 * output may be null, not both.  16-byte aligned x / xq and 8-byte aligned pcm take the vectorised path. */
int dvae_pcm16_f32(const float* x, int64_t n, int16_t* pcm /* nullable */, float* xq /* nullable */, void* stream);

/* ---- STOI / ESTOI on the device (pystoi.stoi, called by scripts/run_metrics.py) ----
 * Ragged batch of (clean x, processed y) pairs: utterance u occupies [off[u], off[u] + len[u]) of x and y, sampled at fs_sig.
 * dvae_resample_taps [host only, no GPU needed]: Octave's anti-aliasing filter that pystoi hands to scipy's resample_poly
 *   for 10 kHz / fs_sig, designed in double and normalised to unit sum; writes it to taps[0..count) (host, nullable) and
 *   returns count (1 tap, the identity, at fs_sig = 10000) or DVAE_ERR_ARG.
 * dvae_resample_poly_f32: xr / yr [r_off[u] .. + ceil(len[u] p / q)) = scipy.signal.resample_poly(x_u, 10000, fs_sig, window=taps)
 *   (same length, delay and zero edges; a copy at fs_sig = 10000); y / yr nullable; taps: a device copy of
 *   dvae_resample_taps(fs_sig); r_off ascending with room for every output, r_total >= the end of the last one.
 * dvae_stoi_envelopes: resampling, pystoi's silent-frame removal (40 dB below the loudest clean frame, energies in double)
 *   and the 15 third-octave band envelopes of every STFT frame of the desilenced signals (FP32
 *   resampled samples, FFT in double, FP32 envelopes).  Frame-indexed
 *   outputs hold dvae_stoi_frame_capacity(B, total, fs_sig) rows; utterance u owns rows frame_off[u] ...:
 *   keep[frame_off[u] + i] (energy frame i kept), env[frame_off[u] + k][2][15] (clean, processed envelopes of STFT frame k),
 *   counts[u] = {energy frames, STFT frames} with STFT frames = -1 when the score is undefined (no complete frame, an
 *   all-zero or non-finite clean signal).  total >= sum_u len[u] sizes the workspace (dvae_stoi_workspace_bytes,
 *   256-byte aligned); an utterance that does not fit is scored NaN.
 * dvae_stoi_scores: out[u] = {STOI, ESTOI} (double statistics); 1e-5 below 30 STFT frames, NaN where counts[u][1] = -1. */
int dvae_resample_taps(int fs_sig, float* taps /* [host], nullable */, int cap);
int dvae_resample_poly_f32(const float* x, const float* y, const int64_t* off, const int32_t* len, int B, int fs_sig,
                           const float* taps, float* xr, float* yr, const int64_t* r_off, int64_t r_total, void* stream);
int64_t dvae_stoi_workspace_bytes(int B, int64_t total, int fs_sig);
int64_t dvae_stoi_frame_capacity(int B, int64_t total, int fs_sig);
int dvae_stoi_envelopes(const float* x, const float* y, const int64_t* off, const int32_t* len, int B, int64_t total, int fs_sig,
                        const float* taps, void* ws, float* env, uint8_t* keep, int64_t* frame_off, int32_t* counts,
                        void* stream);
int dvae_stoi_scores(const float* env, const int64_t* frame_off, const int32_t* counts, int B, double* out, void* stream);

/* ---- label front end on the device (packages/processing/target.py:5-105; center=False, end-pad rule of the STFT) ----
 * dvae_vad_labels: vad[n] = 1 where the power of frame n of the zero-padded signal exceeds 10^vad_threshold times the
 *   utterance's minimum frame power (clean_speech_VAD, target.py:5-56); ws: dvae_vad_workspace_bytes(NT) bytes.
 * dvae_ibm_labels: mask[n][f] = 20 log10(|S| + eps) > max over the utterance - ibm_threshold_db (clean_speech_IBM,
 *   target.py:58-70), multiplied by vad[n] when vad is given (noise_robust_clean_speech_IBM, 72-105); ws: 4 B bytes. */
int64_t dvae_vad_workspace_bytes(int64_t NT);
int dvae_vad_labels(const float* x, const int64_t* x_off, const int32_t* x_len, int B, const int32_t* frame_utt,
                    const int64_t* fr_off, int64_t NT, int n_fft, int hop, float vad_threshold, float* vad, void* ws,
                    void* stream);
int dvae_ibm_labels(const void* S, const int32_t* frame_utt, const int64_t* fr_off, int B, int64_t NT, int F, int ld,
                    float eps, float ibm_threshold_db, const float* vad, float* mask, void* ws, void* stream);

/* ---- per-utterance stopping of the EM loop ----
 * dvae_em_stop_check: after EM iteration n (1-based) with window w (n >= 2w), for the columns u < B_active of the cost matrix
 * cost[niter][ld_cost] (row k = the costs after iteration k, 0-based): m_old = (cost[n-2w][u] + ... + cost[n-w-1][u]) / w and
 * m_new = (cost[n-w][u] + ... + cost[n-1][u]) / w, both summed in ascending k in double; stop[u] = 1 when
 * m_old - m_new <= tol * |m_new| (never when a cost is NaN), else 0. */
int dvae_em_stop_check(const double* cost, int ld_cost, int B_active, int n, int w, double tol, uint8_t* stop, void* stream);

/* dvae_permute_rows: gathers of rows by index maps, every job of the list in one launch:
 *   dst + r * pitch + i * row_bytes <- src + r * pitch + map[i] * row_bytes   for i < n_rows, r < n_rep.
 * row_bytes a positive multiple of 4; 16-byte vector copies when row_bytes, pitch, src and dst are multiples of 16.  src and dst
 * must not overlap.  jobs [host]: up to DVAE_PERMUTE_MAX_JOBS. */
#define DVAE_PERMUTE_MAX_JOBS 16
typedef struct DvaePermuteJob {
    const void* src;
    void* dst;
    const int32_t* map;        /* [n_rows] source row of each destination row */
    int64_t n_rows;
    int64_t row_bytes;
    int64_t n_rep;             /* >= 1 planes `pitch` bytes apart (the columns of a row-major matrix: row_bytes = element size) */
    int64_t pitch;
} DvaePermuteJob;
int dvae_permute_rows(const DvaePermuteJob* jobs, int n_jobs, void* stream);

/* uniform [eps,1) initialisation of W, H and g = 1 from Philox (mcem.py:42-44: max(rand, eps)) */
int dvae_nmf_init(uint64_t seed, const int32_t* utt_ids /*[B] global ids*/, const int64_t* fr_off, int B, int64_t NT, int F,
                  int K, int ld, float eps, float* W, float* H, float* g, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVAE_B200_H */
