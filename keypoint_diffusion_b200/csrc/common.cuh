// Shared device/host helpers for the kpdiff_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/kpdiff_b200.h"

namespace kpd {

// ------------------------------------------------------------------ error plumbing
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define KPD_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            kpd::set_error(__VA_ARGS__);       \
            return -1;                         \
        }                                      \
    } while (0)

#define KPD_TRY(expr)                          \
    do {                                       \
        int _rc = (expr);                      \
        if (_rc != 0) return _rc;              \
    } while (0)

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// carve aligned sub-buffers out of a caller-owned workspace
struct Carver {
    char* base;
    int64_t off;
    explicit Carver(void* p) : base(static_cast<char*>(p)), off(0) {}
    template <typename T>
    T* take(int64_t n) {
        off = align_up(off, 256);
        T* r = reinterpret_cast<T*>(base + off);
        off += n * (int64_t)sizeof(T);
        return r;
    }
    int64_t bytes() const { return align_up(off, 256); }
};

constexpr int TE = KPD_TILE_EDGES;   // rows per CTA tile
constexpr int NT = 256;              // threads per CTA in the tile kernels
constexpr int KC = 16;               // K chunk staged per pipeline stage
constexpr int BS_FLOATS = 2 * KC * 256;  // double-buffered weight stage (floats)

// ------------------------------------------------------------------ math
// accurate (not --use_fast_math) forms: parity mode is fp32-faithful
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ------------------------------------------------------------------ the tile GEMM
// acc[i][4*j+q] (+)= sum_k As[(ty*RM+i)*lda + k] * WT[k*ldw + 4*tx + 64*j + q]
//   256 threads, ty = tid/16, tx = tid%16; rows = 16*RM; up to 256 output columns per call.
//   WT global, K-major, 16-byte aligned rows (ldw % 4 == 0); only columns < nmain are read
//   (nmain % 4 == 0); columns >= nmain of Bs must have been zeroed by the caller once.
//   Weight chunks of KC rows stream through a 2-stage cp.async pipeline in Bs.
//   Ends with a __syncthreads(): As may be overwritten by the caller afterwards.
template <int RM>
__device__ __forceinline__ void tile_gemm(const float* __restrict__ As, int lda,
                                          const float* __restrict__ WT, int ldw, int K, int nmain,
                                          float* __restrict__ Bs, float (&acc)[RM][16]) {
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int nchunks = (K + KC - 1) / KC;

    auto stage = [&](int chunk, int buf) {
        const int k0 = chunk * KC;
        float* dstb = Bs + buf * (KC * 256);
#pragma unroll
        for (int i = 0; i < (KC * 64) / NT; ++i) {
            int idx = tid + NT * i;
            int row = idx >> 6, c4 = idx & 63;
            if (k0 + row < K && 4 * c4 < nmain)
                cp_async16(dstb + row * 256 + 4 * c4, WT + (size_t)(k0 + row) * ldw + 4 * c4);
        }
        cp_async_commit();
    };

    stage(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        const int buf = c & 1;
        if (c + 1 < nchunks) {
            stage(c + 1, buf ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float* B = Bs + buf * (KC * 256) + 4 * tx;
        const float* A = As + (size_t)(ty * RM) * lda + c * KC;
        const int kmax = min(KC, K - c * KC);
        if (kmax == KC) {
#pragma unroll
            for (int k4 = 0; k4 < KC; k4 += 4) {
                float4 a4[RM];
#pragma unroll
                for (int i = 0; i < RM; ++i) a4[i] = *reinterpret_cast<const float4*>(A + i * lda + k4);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    float4 b[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4*>(B + (k4 + kk) * 256 + 64 * j);
#pragma unroll
                    for (int i = 0; i < RM; ++i) {
                        float a = kk == 0 ? a4[i].x : kk == 1 ? a4[i].y : kk == 2 ? a4[i].z : a4[i].w;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            acc[i][4 * j + 0] = fmaf(a, b[j].x, acc[i][4 * j + 0]);
                            acc[i][4 * j + 1] = fmaf(a, b[j].y, acc[i][4 * j + 1]);
                            acc[i][4 * j + 2] = fmaf(a, b[j].z, acc[i][4 * j + 2]);
                            acc[i][4 * j + 3] = fmaf(a, b[j].w, acc[i][4 * j + 3]);
                        }
                    }
                }
            }
        } else {
            for (int kk = 0; kk < kmax; ++kk) {
                float4 b[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4*>(B + kk * 256 + 64 * j);
#pragma unroll
                for (int i = 0; i < RM; ++i) {
                    float a = A[i * lda + kk];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[i][4 * j + 0] = fmaf(a, b[j].x, acc[i][4 * j + 0]);
                        acc[i][4 * j + 1] = fmaf(a, b[j].y, acc[i][4 * j + 1]);
                        acc[i][4 * j + 2] = fmaf(a, b[j].z, acc[i][4 * j + 2]);
                        acc[i][4 * j + 3] = fmaf(a, b[j].w, acc[i][4 * j + 3]);
                    }
                }
            }
        }
        __syncthreads();
    }
}

// zero the weight stage once per kernel (columns >= nmain are never written by tile_gemm)
__device__ __forceinline__ void zero_stage(float* Bs) {
    for (int i = threadIdx.x; i < BS_FLOATS; i += blockDim.x) Bs[i] = 0.0f;
}

// leading dimension for an fp32 row tile of `w` columns: multiple of 4 (float4 rows) and
// == 4 (mod 8) so that the RM rows two half-warps read land in different banks
static inline __host__ __device__ int tile_ld(int w) {
    int p = (w + 3) & ~3;
    return (p % 8 == 4) ? p : p + 4;
}

// ------------------------------------------------------------------ segmented tile reduction
// Rows of a tile are edges sorted by destination.  For column `col` walk the n rows in order
// and emit one sum per run of equal dst.  A run that lies completely inside [tile_begin,
// tile_end) and is the whole CSR row goes straight to out[dst]; a run continuing from the
// previous tile goes to part[0]; a run continuing into the next tile goes to part[1].
// The node-side consumer recombines them in tile order (deterministic, no atomics).
struct SegOut {
    float* out;        // [n_dst][ld_out]
    int ld_out;
    float* part0;      // this tile's "continues from previous tile" slot  [width]
    float* part1;      // this tile's "continues into next tile" slot      [width]
};

__device__ __forceinline__ void seg_reduce_column(const float* __restrict__ C, int ldc, int col, int n,
                                                  const int* __restrict__ dst_s,
                                                  const int* __restrict__ rowptr, int tile_begin,
                                                  const SegOut& o, int out_col) {
    int i = 0;
    while (i < n) {
        const int d = dst_s[i];
        float s = 0.0f;
        int j = i;
        while (j < n && dst_s[j] == d) {
            s += C[j * ldc + col];
            ++j;
        }
        const bool from_prev = (i == 0) && (rowptr[d] < tile_begin);
        const bool into_next = (j == n) && (rowptr[d + 1] > tile_begin + n);
        if (from_prev) o.part0[out_col] = s;
        else if (into_next) o.part1[out_col] = s;
        else o.out[(size_t)d * o.ld_out + out_col] = s;
        i = j;
    }
}

// Node-side recombination for destination node d and column c:
//   rows [r0,r1) of the CSR; tiles of TE edges; part is [ntiles][2][pw].
__device__ __forceinline__ float seg_gather(const float* __restrict__ out, int ld_out,
                                            const float* __restrict__ part, int pw, int r0, int r1,
                                            int d, int c, int tile = TE) {
    if (r1 <= r0) return 0.0f;
    const int t0 = r0 / tile, t1 = (r1 - 1) / tile;
    if (t0 == t1) {
        // complete inside one tile -- unless the tile boundary coincides, still a direct store
        return out[(size_t)d * ld_out + c];
    }
    float s = part[((size_t)t0 * 2 + 1) * pw + c];
    for (int t = t0 + 1; t <= t1; ++t) s += part[((size_t)t * 2 + 0) * pw + c];
    return s;
}

// ------------------------------------------------------------------ row ops (row_ops.cu)
int launch_linear(const float* X, int ldx, const float* WT, int ldw, const float* bias, const float* R,
                  int ldr, float* Y, int ldy, int M, int K, int N, int act, cudaStream_t st);
int launch_layernorm_pair(const float* in0, float* out0, int M0, const float* w0, const float* b0, const float* in1, float* out1,
                          int M1, const float* w1, const float* b1, int ldi, int ldo, int H, cudaStream_t st);
int launch_layernorm(const float* in, int ldi, float* out, int ldo, int M, int H, const float* w,
                     const float* b, cudaStream_t st);
int launch_set_time_col(float* out, int ld, int col, int n, const float* t_ptr, const int* batch,
                        int per_complex, cudaStream_t st);
int launch_concat_time(const float* in, int w, float* out, int ldo, int n, const float* t_ptr,
                       const int* batch, int per_complex, cudaStream_t st);
int launch_copy_rows(const float* in, int ldi, float* out, int ldo, int n, int w, cudaStream_t st);
int launch_sub(const float* a, const float* b, float* out, int n, cudaStream_t st);

// ------------------------------------------------------------------ step ops (ddpm_step.cu)
struct MultistepParams {  // DPM-Solver++(2M) (DESIGN.md section 6.5); a multistep sampler keeps it in device memory,
                          // so that a captured graph can be re-pointed, like RecordParams
    const float* ms_coef; // [rows][4] = (c, alpha_t, sigma_t, 0) of the active schedule (schedule.multistep_rows)
    float* hist_x;        // [n_lig][3] the previous executed row's clean-ligand estimate, frame of the next step
    float* hist_h;        // [n_lig][F]
};
struct RunParams {        // lives in device memory so that a captured graph can be re-pointed
    const float* noise;   // NULL or slots of [n_lig][3+F] (x first), numbered by noise_slot()
    uint64_t seed;
    int T;                // the step the run starts from (the sampler's T, or t0 of a run from a start ligand): the
                          // injected-noise slots of executed steps are counted from it
    int atom_offset;     // added to the atom index of the Philox counter: a batch sampled as several sub-batches draws
                          // the same noise as when it is sampled whole (kpd_sampler_set_atom_offset)
};

// injected-noise slot of draw k of step s in a run from step T: slot 0 is the initial draw (s = -1), then every executed
// step holds per_step draws (1 in the plain loop; 3r-1 with inpainting: posterior, known part, re-noise but after the last pass)
__device__ __forceinline__ int noise_slot(int T, int s, int per_step, int k) {
    return s < 0 ? 0 : 1 + (T - 1 - s) * per_step + k;
}

// where a step kernel's draws come from: in a sampler run (rp) the run's seed, atom offset and injected slot
// noise_slot(T, s, per_step, k); in a stand-alone call the caller's noise and seed.  noise == NULL: Philox.
struct StepDraws {
    const float* noise;
    uint64_t seed;
    int atom_offset;
};
__device__ __forceinline__ StepDraws step_draws(const RunParams* rp, const float* noise, uint64_t seed, int s,
                                                int per_step, int k, size_t slot_len) {
    if (!rp) return {noise, seed, 0};
    return {rp->noise ? rp->noise + (size_t)noise_slot(rp->T, s, per_step, k) * slot_len : nullptr, rp->seed,
            rp->atom_offset};
}

// One CTA per complex.  mean3: out = the mean of rows [r0, r0+n) of x[][3], threads 0..2 summing in row order
// (bit-identical to the oracle's sequential mean); the caller syncs before reading out.  sub3: those rows -= v.
__device__ __forceinline__ void mean3(const float* x, int r0, int n, float* out) {
    if (threadIdx.x < 3) {
        float acc = 0.0f;
        for (int j = 0; j < n; ++j) acc = __fadd_rn(acc, x[3 * (r0 + j) + threadIdx.x]);
        out[threadIdx.x] = __fdiv_rn(acc, (float)n);
    }
}
__device__ __forceinline__ void sub3(float* x, int r0, int n, const float* v) {
    for (int i = threadIdx.x; i < n * 3; i += blockDim.x) x[3 * r0 + i] = __fsub_rn(x[3 * r0 + i], v[i % 3]);
}
// the ligand COM (into com[3], shared) removed from the complex's ligand and keypoint rows
__device__ __forceinline__ void remove_ligand_com(float* x_lig, float* x_kp, int l0, int nl, int k0, int nk, float* com) {
    mean3(x_lig, l0, nl, com);
    __syncthreads();
    sub3(x_lig, l0, nl, com);
    sub3(x_kp, k0, nk, com);
}

// msp (device, a multistep sampler's) or msv (host copy, a stand-alone call) selects the DPM-Solver++(2M) step; first_row
// is the row a stand-alone call treats as the run's first (no correction); a sampler's run takes RunParams.T - 1
int launch_ddpm_step(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                     const float* eps_h, int F, const float* coef, const int* step_ptr, const float* noise_x,
                     const float* noise_h, uint64_t seed, const RunParams* rp, cudaStream_t st,
                     const struct MultistepParams* msp = nullptr, const struct MultistepParams* msv = nullptr,
                     int first_row = 0);
int launch_com(const kpd_batch* b, float* x_lig, float* x_kp, int which, int shift, float* com_out, cudaStream_t st);
int launch_shift(float* x, const int* node_batch, int n, const float* v, float sign, cudaStream_t st);
int launch_randn_init(float* x_lig, float* h_lig, int n_lig, int F, uint64_t seed, const RunParams* rp, cudaStream_t st);
int launch_scale(float* x, int n, float s, cudaStream_t st);
int launch_step_prologue(int* counter, int* step, float* t_cur, const float* coef, cudaStream_t st);

// ------------------------------------------------------------------ fragment-conditioned sampling (inpaint.cu)
struct InpaintParams {    // a sampler keeps it in device memory, so that a captured graph can be re-pointed
    const uint8_t* mask;  // NULL (no fixed atom) or [n_lig], nonzero = fixed
    const float* x_fix;   // [n_lig][3] fragment positions, frame of the keypoints the caller passed
    const float* h_fix;   // [n_lig][F] fragment features, returned (un-normalised) feature space
    const float* coef2;   // [T][4] rows (alpha_s, sigma_s, alpha_t|s, sigma_t|s)
};
// noise: NULL or the draws of this call ([2][n_lig][3+F] posterior then known part; [n_lig][3+F] for renoise), x first;
// with rp (a sampler's run) and ip (its fragment) the slot and the buffers come from device memory instead
int launch_ddpm_inpaint_step(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                             const float* eps_h, int F, const float* coef, const int* step_ptr, int u, int r,
                             const InpaintParams& fr, const InpaintParams* ip, const float* init_kp_com, float norm_c,
                             const float* noise, uint64_t seed, const RunParams* rp, cudaStream_t st);
int launch_renoise(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, int F, const int* step_ptr, int u, int r,
                   const float* coef2, const InpaintParams* ip, const float* noise, uint64_t seed, const RunParams* rp,
                   cudaStream_t st);
// ------------------------------------------------------------------ partial noising of a start ligand (partial_noise.cu)
// noise: NULL or [n_lig][3+F] (x first) for the stand-alone call; with rp (a sampler's run) seed, noise slot 0 and the
// atom offset come from device memory instead
int launch_partial_noise(const kpd_batch* b, const float* x_start, const float* h_start, float* x_lig, float* h_lig,
                         float* x_kp, int F, float alpha, float sigma, float norm_c, const float* noise, uint64_t seed,
                         const RunParams* rp, cudaStream_t st);
// ------------------------------------------------------------------ trajectory recording (trajectory.cu)
struct RecordParams {     // a recording sampler keeps it in device memory, so that a captured graph can be re-pointed
    int every;            // frame stride k >= 1: executed step i is recorded when i % k == 0, as frame i / k
    float* x_frames;      // NULL (record nothing) or [m+1][n_lig][3] state frames, output frame of reference
    float* h_frames;      // [m+1][n_lig][F]
    float* x_pred;        // [m][n_lig][3] clean-ligand estimates (x - sigma_t eps_x) / alpha_t, same frame
    float* h_pred;        // [m][n_lig][F]
    const float* pred_coef;   // [rows][2] (alpha_t, sigma_t) of the state each row starts from
};
int launch_record_frame(const kpd_batch* b, const float* x_lig, const float* h_lig, const float* x_kp,
                        const float* eps_x, const float* eps_h, int F, const int* step_ptr, const RunParams* rp,
                        const RecordParams* rec, const float* init_kp_com, float norm_c, cudaStream_t st);
long long launch_count();  // kernels launched through check_launch() so far (this process)

// optional per-kernel CUDA-event timing (bench.py's roofline leg); no-ops unless enabled and
// never active while a stream is being captured
enum ProfId { PROF_EGNN_EDGE = 1, PROF_GVP_EDGE = 2, PROF_GRAPH = 3, PROF_STEP = 4, PROF_GVP_NODE = 5,
              PROF_GVP_HEAD = 6, PROF_EGNN_NODE = 7, PROF_EGNN_PRE = 8, PROF_ENCDEC = 9 };
void prof_begin(int id, cudaStream_t st);
void prof_end(int id, cudaStream_t st);
bool prof_enabled();      // a kernel id is being timed: callers keep to one stream and one launch per stage

int build_graph_impl(const kpd_batch* batch, const float* x_lig, const float* x_kp, const kpd_graph_params* p,
                     kpd_csr* ll, kpd_csr* kl, kpd_csr* lk, int32_t* counts_ll, int32_t* counts_kl, void* workspace,
                     long long* edge_accum, cudaStream_t st);

}  // namespace kpd
