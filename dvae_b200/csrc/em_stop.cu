// Per-utterance stopping of the EM loop: the convergence test on the cost matrix and the row gathers that move stopped
// utterances out of the active range of the batch (engine.py, McemConfig.stop_tol).
#include "common.cuh"

namespace dvae {

// One thread per utterance; the two window sums run in ascending iteration order, in double.
__global__ void em_stop_check_kernel(const double* __restrict__ cost, int ld_cost, int B_active, int n, int w, double tol,
                                     uint8_t* __restrict__ stop) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= B_active) return;
    double s_old = 0.0, s_new = 0.0;
    for (int k = n - 2 * w; k < n - w; ++k) s_old += cost[(int64_t)k * ld_cost + u];
    for (int k = n - w; k < n; ++k) s_new += cost[(int64_t)k * ld_cost + u];
    const double m_old = s_old / w, m_new = s_new / w;
    stop[u] = (m_old - m_new <= tol * fabs(m_new)) ? 1 : 0;         // false for NaN
}

struct PermuteJobs {
    DvaePermuteJob j[DVAE_PERMUTE_MAX_JOBS];
};

// blockIdx.y = job; the grid strides over the job's (plane, row, word) elements, 16-byte words when the job allows them
__global__ void __launch_bounds__(256) permute_rows_kernel(PermuteJobs jobs) {
    const DvaePermuteJob& jb = jobs.j[blockIdx.y];
    const bool vec = ((jb.row_bytes | jb.pitch | (int64_t)(uintptr_t)jb.src | (int64_t)(uintptr_t)jb.dst) & 15) == 0;
    const int64_t wb = vec ? 16 : 4;
    const int64_t words = jb.row_bytes / wb, per_rep = jb.n_rows * words, total = per_rep * jb.n_rep;
    const char* src = static_cast<const char*>(jb.src);
    char* dst = static_cast<char*>(jb.dst);
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / per_rep, rem = e - r * per_rep;
        const int64_t i = rem / words, k = rem - i * words;
        const int64_t s_off = r * jb.pitch + (int64_t)__ldg(jb.map + i) * jb.row_bytes + k * wb;
        const int64_t d_off = r * jb.pitch + i * jb.row_bytes + k * wb;
        if (vec) *reinterpret_cast<uint4*>(dst + d_off) = __ldg(reinterpret_cast<const uint4*>(src + s_off));
        else *reinterpret_cast<uint32_t*>(dst + d_off) = __ldg(reinterpret_cast<const uint32_t*>(src + s_off));
    }
}

}  // namespace dvae

using namespace dvae;

extern "C" int dvae_em_stop_check(const double* cost, int ld_cost, int B_active, int n, int w, double tol, uint8_t* stop,
                                  void* stream) {
    DVAE_REQUIRE(cost && stop, "dvae_em_stop_check: null pointer");
    DVAE_REQUIRE(B_active >= 0 && ld_cost >= B_active, "dvae_em_stop_check: B_active=%d, ld_cost=%d", B_active, ld_cost);
    DVAE_REQUIRE(w >= 1 && n >= 2 * w, "dvae_em_stop_check: needs n >= 2w (n=%d, w=%d)", n, w);
    DVAE_REQUIRE(tol >= 0.0 && tol <= 1.79e308, "dvae_em_stop_check: tol must be finite and >= 0");
    if (B_active == 0) return 0;
    em_stop_check_kernel<<<(B_active + 127) / 128, 128, 0, (cudaStream_t)stream>>>(cost, ld_cost, B_active, n, w, tol, stop);
    return check_launch("em_stop_check_kernel");
}

extern "C" int dvae_permute_rows(const DvaePermuteJob* jobs, int n_jobs, void* stream) {
    DVAE_REQUIRE(jobs && n_jobs >= 0 && n_jobs <= DVAE_PERMUTE_MAX_JOBS, "dvae_permute_rows: 0..%d jobs", DVAE_PERMUTE_MAX_JOBS);
    PermuteJobs pj{};
    int m = 0;
    int64_t most = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const DvaePermuteJob& jb = jobs[i];
        DVAE_REQUIRE(jb.n_rows >= 0 && jb.n_rep >= 1 && jb.row_bytes > 0 && jb.row_bytes % 4 == 0,
                     "dvae_permute_rows: job %d: bad sizes (row_bytes must be a positive multiple of 4)", i);
        DVAE_REQUIRE(jb.n_rep == 1 || jb.pitch >= jb.n_rows * jb.row_bytes, "dvae_permute_rows: job %d: planes overlap", i);
        DVAE_REQUIRE(jb.pitch % 4 == 0, "dvae_permute_rows: job %d: pitch must be a multiple of 4", i);
        if (jb.n_rows == 0) continue;
        DVAE_REQUIRE(jb.src && jb.dst && jb.map, "dvae_permute_rows: job %d: null pointer", i);
        DVAE_REQUIRE(((uintptr_t)jb.src & 3) == 0 && ((uintptr_t)jb.dst & 3) == 0, "dvae_permute_rows: job %d: unaligned pointer", i);
        pj.j[m++] = jb;
        const int64_t e = jb.n_rep * jb.n_rows * (jb.row_bytes / 4);
        most = e > most ? e : most;
    }
    if (m == 0) return 0;
    const int64_t bx = (most + 255) / 256;
    permute_rows_kernel<<<dim3((unsigned)(bx < 148 * 8 ? bx : 148 * 8), m), 256, 0, (cudaStream_t)stream>>>(pj);
    return check_launch("permute_rows_kernel");
}
