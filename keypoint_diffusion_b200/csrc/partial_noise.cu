// Ligand optimisation by partial noising: the start of a reverse-diffusion run from a given ligand at step t0
// (SDEdit-style, DiffSBDD's molecule optimisation; DESIGN.md section 6.2).
//
// Replaces the plain loop's frame setup after the keypoint mean (shift by init_lig_pos, randn_init, ligand COM
// removal) with one launch, one CTA per complex:
//   c_b  = mean of x_start over the complex's atoms                 (sequential sum in atom order, then a division)
//   x_kp = x_kp - c_b
//   z_x  = alpha*(x_start - c_b) + sigma*e_x,  z_h = alpha*(h_start / norm_c) + sigma*e_h
//   then the ligand COM of z_x is removed from ligand and keypoints.
// alpha = alpha_t0, sigma = sigma_t0 (schedule.start_coefficients); e is the plain loop's initial draw: Philox
// (seed, step = -1, atom, channel), or injected-noise slot 0.  The arithmetic is unfused __f*_rn like ddpm_step_kernel,
// so with injected draws the state equals the op-by-op PyTorch evaluation of oracle/optimize.py.
#include "common.cuh"
#include "philox.cuh"

namespace kpd {

// ddpm_step.cu's philox_normal, draw for draw (the same counter, key and Box-Muller arithmetic); a copy so that the
// plain step's translation unit stays untouched
__device__ float philox_normal_start(uint64_t seed, int step, int atom, int ch) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)atom, (uint32_t)(step + 1), (uint32_t)(ch >> 2), 0u),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const int q = ch & 3;
    const uint32_t ua = q < 2 ? r.x : r.z, ub = q < 2 ? r.y : r.w;
    const float u1 = ((float)ua + 1.0f) * 2.3283064365386963e-10f;
    const float u2 = (float)ub * 2.3283064365386963e-10f;
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincosf(6.283185307179586f * u2, &sn, &cs);
    return (q & 1) ? rad * sn : rad * cs;
}

__global__ void __launch_bounds__(128)
partial_noise_kernel(kpd_batch b, const float* __restrict__ x_start, const float* __restrict__ h_start,
                     float* __restrict__ x_lig, float* __restrict__ h_lig, float* __restrict__ x_kp, int F, float alpha,
                     float sigma, float norm_c, const float* noise, uint64_t seed, const RunParams* rp) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    int aoff = 0;
    if (rp) { seed = rp->seed; noise = rp->noise; aoff = rp->atom_offset; }
    __shared__ float cb[3], com[3];
    if (threadIdx.x < 3) {
        float acc = 0.0f;
        for (int j = 0; j < nl; ++j) acc = __fadd_rn(acc, x_start[3 * (l0 + j) + threadIdx.x]);
        cb[threadIdx.x] = __fdiv_rn(acc, (float)nl);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nk * 3; i += blockDim.x) x_kp[3 * k0 + i] = __fsub_rn(x_kp[3 * k0 + i], cb[i % 3]);
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) {
        const int idx = 3 * l0 + i;
        const float e = noise ? noise[idx] : philox_normal_start(seed, -1, aoff + l0 + i / 3, i % 3);
        const float x0 = __fsub_rn(x_start[idx], cb[i % 3]);
        x_lig[idx] = __fadd_rn(__fmul_rn(alpha, x0), __fmul_rn(sigma, e));
    }
    for (int i = threadIdx.x; i < nl * F; i += blockDim.x) {
        const int idx = F * l0 + i;
        const float e = noise ? noise[(size_t)b.n_lig * 3 + idx] : philox_normal_start(seed, -1, aoff + l0 + i / F, 3 + i % F);
        const float h0 = __fdiv_rn(h_start[idx], norm_c);
        h_lig[idx] = __fadd_rn(__fmul_rn(alpha, h0), __fmul_rn(sigma, e));
    }
    __syncthreads();
    // remove the ligand COM from ligand and keypoints (as the plain loop does after its initial draw)
    if (threadIdx.x < 3) {
        float acc = 0.0f;
        for (int j = 0; j < nl; ++j) acc = __fadd_rn(acc, x_lig[3 * (l0 + j) + threadIdx.x]);
        com[threadIdx.x] = __fdiv_rn(acc, (float)nl);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) x_lig[3 * l0 + i] = __fsub_rn(x_lig[3 * l0 + i], com[i % 3]);
    for (int i = threadIdx.x; i < nk * 3; i += blockDim.x) x_kp[3 * k0 + i] = __fsub_rn(x_kp[3 * k0 + i], com[i % 3]);
}

int launch_partial_noise(const kpd_batch* b, const float* x_start, const float* h_start, float* x_lig, float* h_lig,
                         float* x_kp, int F, float alpha, float sigma, float norm_c, const float* noise, uint64_t seed,
                         const RunParams* rp, cudaStream_t st) {
    partial_noise_kernel<<<b->B, 128, 0, st>>>(*b, x_start, h_start, x_lig, h_lig, x_kp, F, alpha, sigma, norm_c, noise,
                                               seed, rp);
    return check_launch("partial_noise_kernel");
}

}  // namespace kpd

using namespace kpd;

extern "C" int kpd_partial_noise(const kpd_batch* batch, const float* x_start, const float* h_start, float* x_lig,
                                 float* h_lig, float* x_kp, int32_t atom_nf, float alpha, float sigma,
                                 float lig_feat_norm_constant, const float* noise, uint64_t seed, void* stream) {
    KPD_REQUIRE(batch && x_start && h_start && x_lig && h_lig && x_kp, "kpd_partial_noise: null argument");
    KPD_REQUIRE(atom_nf >= 1 && lig_feat_norm_constant != 0.0f, "kpd_partial_noise: bad argument");
    return launch_partial_noise(batch, x_start, h_start, x_lig, h_lig, x_kp, atom_nf, alpha, sigma,
                                lig_feat_norm_constant, noise, seed, nullptr, static_cast<cudaStream_t>(stream));
}
