// Scale-invariant energy ratios on the device (SURVEY §8(f) N1): SI-SDR, SI-SIR, SI-SAR of a ragged batch.
//
// Replaces packages/metrics.py:12-82 (si_sdr_components / energy_ratios / si_sdr_leroux), which works on one pair of
// host vectors at a time.  With the six inner products  a = <s_hat,s>, b = <s_hat,n>, c = <s,s>, d = <n,n>,
// e = <s_hat,s_hat>, f = <s,n>  (accumulated in double) the reference's vectors never have to be formed:
//
//   alpha_s = a / c, alpha_n = b / d
//   |s_target|^2        = alpha_s^2 c
//   |e_noise|^2         = alpha_n^2 d
//   |e_noise + e_art|^2 = |s_hat - s_target|^2 = e - 2 alpha_s a + alpha_s^2 c
//   |e_art|^2           = e + alpha_s^2 c + alpha_n^2 d - 2 alpha_s a - 2 alpha_n b + 2 alpha_s alpha_n f
//
// One CTA per utterance; per-thread double partial sums in a fixed order, fixed-order tree reduction: deterministic.
// HBM-bound: 3 x 4 T bytes read per utterance.
#include <algorithm>

#include "common.cuh"

namespace dvae {

__global__ void __launch_bounds__(256) energy_ratios_kernel(const float* __restrict__ s_hat, const float* __restrict__ s,
                                                            const float* __restrict__ n, const int64_t* __restrict__ off,
                                                            const int32_t* __restrict__ len, double* __restrict__ out) {
    __shared__ double red[6][8];
    const int u = blockIdx.x;
    const int64_t o = off[u];
    const int T = len[u];
    double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        const double x = (double)s_hat[o + i], y = (double)s[o + i], z = n ? (double)n[o + i] : 0.0;
        acc[0] = fma(x, y, acc[0]);
        acc[1] = fma(x, z, acc[1]);
        acc[2] = fma(y, y, acc[2]);
        acc[3] = fma(z, z, acc[3]);
        acc[4] = fma(x, x, acc[4]);
        acc[5] = fma(y, z, acc[5]);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const double v = warp_sum_d(acc[k]);
        if (lane == 0) red[k][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            double v = 0.0;
            for (int w = 0; w < 8; ++w) v += red[k][w];
            t[k] = v;
        }
        const double a = t[0], b = t[1], c = t[2], d = t[3], e = t[4], f = t[5];
        const double as = a / c;
        const double tgt = as * as * c;
        const double dist = e - 2.0 * as * a + tgt;                      // |s_hat - s_target|^2
        double* r = out + 3 * (int64_t)u;
        r[0] = 10.0 * log10(tgt / dist);
        if (n) {
            const double an = b / d;
            const double noise = an * an * d;
            const double art = e + tgt + noise - 2.0 * as * a - 2.0 * an * b + 2.0 * as * an * f;
            r[1] = 10.0 * log10(tgt / noise);
            r[2] = 10.0 * log10(tgt / art);
        } else {
            r[1] = nan("");
            r[2] = nan("");
        }
    }
}

// 16-bit PCM quantisation of batch_io.write_wav: q = clip(rint(x * 32768), -32768, 32767), round half to even.  x * 32768 is
// exact in FP32 (a power-of-two scale), so this equals numpy's float64 expression; +-Inf saturate, NaN maps to 0.  xq = q / 32768
// is what read_wav returns for the written file (exact in FP32).
__device__ __forceinline__ int pcm16_of(float v) {
    const float r = fminf(fmaxf(rintf(v * 32768.0f), -32768.0f), 32767.0f);
    return v == v ? (int)r : 0;
}

// V samples per thread and iteration (V = 4: 16-byte loads, 8-byte PCM stores, 16-byte xq stores; V = 1 for unaligned pointers).
// HBM-bound: 4 bytes read and up to 6 written per sample.
template <int V>
__global__ void __launch_bounds__(256) pcm16_kernel(const float* __restrict__ x, int64_t n, int16_t* __restrict__ pcm,
                                                    float* __restrict__ xq) {
    const int64_t nv = n / V, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
        float v[V];
        int q[V];
        if constexpr (V == 4) {
            const float4 t = reinterpret_cast<const float4*>(x)[i];
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
            v[0] = x[i];
        }
#pragma unroll
        for (int k = 0; k < V; ++k) q[k] = pcm16_of(v[k]);
        if constexpr (V == 4) {
            if (pcm) {
                const uint2 w = make_uint2(((uint32_t)q[0] & 0xffffu) | ((uint32_t)q[1] << 16),
                                           ((uint32_t)q[2] & 0xffffu) | ((uint32_t)q[3] << 16));
                reinterpret_cast<uint2*>(pcm)[i] = w;
            }
            if (xq) reinterpret_cast<float4*>(xq)[i] = make_float4(q[0] * (1.0f / 32768.0f), q[1] * (1.0f / 32768.0f),
                                                                   q[2] * (1.0f / 32768.0f), q[3] * (1.0f / 32768.0f));
        } else {
            if (pcm) pcm[i] = (int16_t)q[0];
            if (xq) xq[i] = q[0] * (1.0f / 32768.0f);
        }
    }
    if (V > 1 && blockIdx.x == 0 && threadIdx.x < n - nv * V) {          // the last n % V samples
        const int64_t j = nv * V + threadIdx.x;
        const int q = pcm16_of(x[j]);
        if (pcm) pcm[j] = (int16_t)q;
        if (xq) xq[j] = q * (1.0f / 32768.0f);
    }
}

}  // namespace dvae

using namespace dvae;

extern "C" int dvae_pcm16_f32(const float* x, int64_t n, int16_t* pcm, float* xq, void* stream) {
    DVAE_REQUIRE(x && n >= 0 && (pcm || xq), "dvae_pcm16_f32: bad arguments (x, n >= 0 and at least one of pcm / xq)");
    if (n == 0) return 0;
    const bool vec = ((uintptr_t)x % 16 == 0) && ((uintptr_t)pcm % 8 == 0) && ((uintptr_t)xq % 16 == 0);
    const int64_t items = vec ? n / 4 : n;
    const int64_t grid = std::min<int64_t>(std::max<int64_t>((items + 255) / 256, 1), 148 * 8);
    if (vec) pcm16_kernel<4><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(x, n, pcm, xq);
    else pcm16_kernel<1><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(x, n, pcm, xq);
    return check_launch("pcm16_kernel");
}

extern "C" int dvae_energy_ratios(const float* s_hat, const float* s, const float* n, const int64_t* off, const int32_t* len,
                                  int B, double* out, void* stream) {
    DVAE_REQUIRE(s_hat && s && off && len && out && B >= 0, "dvae_energy_ratios: bad arguments");
    if (B == 0) return 0;
    energy_ratios_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(s_hat, s, n, off, len, out);
    return check_launch("energy_ratios_kernel");
}
