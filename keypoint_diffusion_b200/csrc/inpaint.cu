// Fragment-conditioned sampling: the reverse step with the known atoms replaced, and the re-noise between
// resampling passes (inpainting with RePaint-style resampling, DESIGN.md section 6.1).
//
// The reference has no inpainting; this follows DiffSBDD's inpainting sampler for the same class of model, with the
// keypoints in the pocket's role.  Per reverse step s (t = s+1) and pass u = 0 .. r-1:
//   z_unk = x/alpha_t|s - var_terms*eps + sigma*noise               (ddpm_step_kernel, word 3u)
//   z_kn  = alpha_s*(x_fix - init_kp_com + kp_com_now) + sigma_s*e  (word 3u+1; features h_fix / norm)
//   dx    = mean_M(z_unk_x) - mean_M(z_kn_x), added to z_kn_x and to the complex's keypoints
//   x, h  = M ? z_kn : z_unk, then the ligand COM is removed from ligand and keypoints
// and, if u < r-1, renoise_kernel takes the state back to level t (word 3u+2) and removes the COM again.
//
// One CTA per complex, the same unfused __f*_rn arithmetic and sequential atom-order sums as ddpm_step_kernel: with
// injected draws the state matches the op-by-op PyTorch evaluation of oracle/flat.py.  A complex without a fixed atom
// runs exactly the operations of ddpm_step_kernel, so at u = 0 it gets bit-identical results.
#include "common.cuh"
#include "philox.cuh"

namespace kpd {

__global__ void __launch_bounds__(128)
ddpm_inpaint_step_kernel(kpd_batch b, float* __restrict__ x_lig, float* __restrict__ h_lig, float* __restrict__ x_kp,
                         const float* __restrict__ eps_x, const float* __restrict__ eps_h, int F,
                         const float* __restrict__ coef, const int* __restrict__ step_ptr, int u, int r,
                         InpaintParams fr, const InpaintParams* ip, const float* __restrict__ init_kp_com, float norm_c,
                         const float* noise, uint64_t seed, const RunParams* rp) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    const int s = *step_ptr;
    if (ip) fr = *ip;
    const float a = coef[4 * s], vt = coef[4 * s + 1], sg = coef[4 * s + 2];
    const float a_s = fr.coef2[4 * s], sg_s = fr.coef2[4 * s + 1];
    const size_t slot_len = (size_t)b.n_lig * (3 + F);
    // the known-part draws (kind 1) follow the posterior ones (kind 0), in a run's slots as in a stand-alone call's noise
    const StepDraws d = step_draws(rp, noise, seed, s, 3 * r - 1, 3 * u, slot_len);
    const float* nz_post = d.noise;
    const float* nz_kn = d.noise ? d.noise + slot_len : nullptr;
    const uint32_t w = 3u * (uint32_t)u;
    const uint8_t* M = fr.mask ? fr.mask + l0 : nullptr;
    extern __shared__ float z_kn[];          // [max_lig][3]: known-part positions of this complex
    __shared__ float kp_com[3], dx[3], com[3];
    __shared__ int n_fix;
    // fixed atoms of this complex and, if there are any, the keypoint COM of the current (drifting) frame
    if (threadIdx.x < 3) {
        int m = 0;
        if (M)
            for (int j = 0; j < nl; ++j) m += M[j] != 0;
        if (m) mean3(x_kp, k0, nk, kp_com);
        if (threadIdx.x == 0) n_fix = m;
    }
    __syncthreads();
    const int m = n_fix;
    // z_unk for every position (the masked mean needs it at the fixed atoms too); z_kn for the fixed ones
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) {
        const int idx = 3 * l0 + i, atom = d.atom_offset + l0 + i / 3, ch = i % 3;
        const float nz = nz_post ? nz_post[idx] : philox_normal(d.seed, s, atom, ch, w);
        const float mu = __fsub_rn(__fdiv_rn(x_lig[idx], a), __fmul_rn(vt, eps_x[idx]));
        x_lig[idx] = __fadd_rn(mu, __fmul_rn(sg, nz));
        if (m && M[i / 3]) {
            const float x0 = __fadd_rn(__fsub_rn(fr.x_fix[idx], init_kp_com[3 * c + ch]), kp_com[ch]);
            const float e = nz_kn ? nz_kn[idx] : philox_normal(d.seed, s, atom, ch, w + 1);
            z_kn[i] = __fadd_rn(__fmul_rn(a_s, x0), __fmul_rn(sg_s, e));
        }
    }
    // features: merged at once (no alignment)
    for (int i = threadIdx.x; i < nl * F; i += blockDim.x) {
        const int idx = F * l0 + i, atom = d.atom_offset + l0 + i / F, ch = 3 + i % F;
        if (m && M[i / F]) {
            const float h0 = __fdiv_rn(fr.h_fix[idx], norm_c);
            const float e = nz_kn ? nz_kn[(size_t)b.n_lig * 3 + idx] : philox_normal(d.seed, s, atom, ch, w + 1);
            h_lig[idx] = __fadd_rn(__fmul_rn(a_s, h0), __fmul_rn(sg_s, e));
        } else {
            const float nz = nz_post ? nz_post[(size_t)b.n_lig * 3 + idx] : philox_normal(d.seed, s, atom, ch, w);
            const float mu = __fsub_rn(__fdiv_rn(h_lig[idx], a), __fmul_rn(vt, eps_h[idx]));
            h_lig[idx] = __fadd_rn(mu, __fmul_rn(sg, nz));
        }
    }
    __syncthreads();
    if (m) {
        // align: dx = mean_M(z_unk_x) - mean_M(z_kn_x), sequential sums in atom order; fragment and pocket move together
        if (threadIdx.x < 3) {
            float au = 0.0f, ak = 0.0f;
            for (int j = 0; j < nl; ++j) {
                if (!M[j]) continue;
                au = __fadd_rn(au, x_lig[3 * (l0 + j) + threadIdx.x]);
                ak = __fadd_rn(ak, z_kn[3 * j + threadIdx.x]);
            }
            dx[threadIdx.x] = __fsub_rn(__fdiv_rn(au, (float)m), __fdiv_rn(ak, (float)m));
        }
        __syncthreads();
        for (int i = threadIdx.x; i < nl * 3; i += blockDim.x)
            if (M[i / 3]) x_lig[3 * l0 + i] = __fadd_rn(z_kn[i], dx[i % 3]);
        for (int i = threadIdx.x; i < nk * 3; i += blockDim.x) x_kp[3 * k0 + i] = __fadd_rn(x_kp[3 * k0 + i], dx[i % 3]);
        __syncthreads();
    }
    remove_ligand_com(x_lig, x_kp, l0, nl, k0, nk, com);
}

int launch_ddpm_inpaint_step(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                             const float* eps_h, int F, const float* coef, const int* step_ptr, int u, int r,
                             const InpaintParams& fr, const InpaintParams* ip, const float* init_kp_com, float norm_c,
                             const float* noise, uint64_t seed, const RunParams* rp, cudaStream_t st) {
    const size_t smem = sizeof(float) * 3 * (size_t)b->max_lig;
    KPD_REQUIRE(smem <= 48 * 1024, "ddpm_inpaint_step: %d atoms in one complex exceed the supported 4096", b->max_lig);
    prof_begin(PROF_STEP, st);
    ddpm_inpaint_step_kernel<<<b->B, 128, smem, st>>>(*b, x_lig, h_lig, x_kp, eps_x, eps_h, F, coef, step_ptr, u, r, fr,
                                                      ip, init_kp_com, norm_c, noise, seed, rp);
    const int rc = check_launch("ddpm_inpaint_step_kernel");
    prof_end(PROF_STEP, st);
    return rc;
}

// z_t = alpha_t|s * z_s + sigma_t|s * e for positions and features (word 3u+2), then the ligand COM is removed
__global__ void __launch_bounds__(128)
renoise_kernel(kpd_batch b, float* __restrict__ x_lig, float* __restrict__ h_lig, float* __restrict__ x_kp, int F,
               const int* __restrict__ step_ptr, int u, int r, const float* coef2, const InpaintParams* ip,
               const float* noise, uint64_t seed, const RunParams* rp) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    const int s = *step_ptr;
    if (ip) coef2 = ip->coef2;
    const float a = coef2[4 * s + 2], sg = coef2[4 * s + 3];
    const StepDraws d = step_draws(rp, noise, seed, s, 3 * r - 1, 3 * u + 2, (size_t)b.n_lig * (3 + F));
    const uint32_t w = 3u * (uint32_t)u + 2u;
    __shared__ float com[3];
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) {
        const int idx = 3 * l0 + i;
        const float e = d.noise ? d.noise[idx] : philox_normal(d.seed, s, d.atom_offset + l0 + i / 3, i % 3, w);
        x_lig[idx] = __fadd_rn(__fmul_rn(a, x_lig[idx]), __fmul_rn(sg, e));
    }
    for (int i = threadIdx.x; i < nl * F; i += blockDim.x) {
        const int idx = F * l0 + i;
        const float e = d.noise ? d.noise[(size_t)b.n_lig * 3 + idx]
                                : philox_normal(d.seed, s, d.atom_offset + l0 + i / F, 3 + i % F, w);
        h_lig[idx] = __fadd_rn(__fmul_rn(a, h_lig[idx]), __fmul_rn(sg, e));
    }
    __syncthreads();
    remove_ligand_com(x_lig, x_kp, l0, nl, k0, nk, com);
}

int launch_renoise(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, int F, const int* step_ptr, int u, int r,
                   const float* coef2, const InpaintParams* ip, const float* noise, uint64_t seed, const RunParams* rp,
                   cudaStream_t st) {
    renoise_kernel<<<b->B, 128, 0, st>>>(*b, x_lig, h_lig, x_kp, F, step_ptr, u, r, coef2, ip, noise, seed, rp);
    return check_launch("renoise_kernel");
}

}  // namespace kpd

using namespace kpd;

extern "C" int kpd_ddpm_inpaint_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                                     const float* eps_h, int32_t atom_nf, const float* coef, const float* coef2,
                                     const int32_t* step_ptr, int32_t u, const uint8_t* fixed_mask, const float* x_fix,
                                     const float* h_fix, const float* init_kp_com, float lig_feat_norm_constant,
                                     const float* noise, uint64_t seed, void* stream) {
    KPD_REQUIRE(batch && x_lig && h_lig && x_kp && eps_x && eps_h && coef && coef2 && step_ptr && init_kp_com,
                "kpd_ddpm_inpaint_step: null argument");
    KPD_REQUIRE(!fixed_mask || (x_fix && h_fix), "kpd_ddpm_inpaint_step: a fixed mask needs x_fix and h_fix");
    KPD_REQUIRE(u >= 0 && lig_feat_norm_constant != 0.0f, "kpd_ddpm_inpaint_step: bad argument");
    const InpaintParams fr = {fixed_mask, x_fix, h_fix, coef2};
    return launch_ddpm_inpaint_step(batch, x_lig, h_lig, x_kp, eps_x, eps_h, atom_nf, coef, step_ptr, u, 0, fr, nullptr,
                                    init_kp_com, lig_feat_norm_constant, noise, seed, nullptr,
                                    static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_renoise(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp, int32_t atom_nf,
                           const float* coef2, const int32_t* step_ptr, int32_t u, const float* noise, uint64_t seed,
                           void* stream) {
    KPD_REQUIRE(batch && x_lig && h_lig && x_kp && coef2 && step_ptr, "kpd_renoise: null argument");
    KPD_REQUIRE(u >= 0, "kpd_renoise: bad argument");
    return launch_renoise(batch, x_lig, h_lig, x_kp, atom_nf, step_ptr, u, 0, coef2, nullptr, noise, seed, nullptr,
                          static_cast<cudaStream_t>(stream));
}
