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

__global__ void __launch_bounds__(128)
partial_noise_kernel(kpd_batch b, const float* __restrict__ x_start, const float* __restrict__ h_start,
                     float* __restrict__ x_lig, float* __restrict__ h_lig, float* __restrict__ x_kp, int F, float alpha,
                     float sigma, float norm_c, const float* noise, uint64_t seed, const RunParams* rp) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    const StepDraws d = step_draws(rp, noise, seed, -1, 1, 0, (size_t)b.n_lig * (3 + F));
    __shared__ float cb[3], com[3];
    mean3(x_start, l0, nl, cb);
    __syncthreads();
    sub3(x_kp, k0, nk, cb);
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) {
        const int idx = 3 * l0 + i;
        const float e = d.noise ? d.noise[idx] : philox_normal(d.seed, -1, d.atom_offset + l0 + i / 3, i % 3);
        const float x0 = __fsub_rn(x_start[idx], cb[i % 3]);
        x_lig[idx] = __fadd_rn(__fmul_rn(alpha, x0), __fmul_rn(sigma, e));
    }
    for (int i = threadIdx.x; i < nl * F; i += blockDim.x) {
        const int idx = F * l0 + i;
        const float e = d.noise ? d.noise[(size_t)b.n_lig * 3 + idx]
                                : philox_normal(d.seed, -1, d.atom_offset + l0 + i / F, 3 + i % F);
        const float h0 = __fdiv_rn(h_start[idx], norm_c);
        h_lig[idx] = __fadd_rn(__fmul_rn(alpha, h0), __fmul_rn(sigma, e));
    }
    __syncthreads();
    remove_ligand_com(x_lig, x_kp, l0, nl, k0, nk, com);   // as the plain loop does after its initial draw
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
