// (e) Reverse-diffusion step: posterior mean, noise draw, centre-of-mass removal -- one launch.
//
// Replaces KeypointDiffusion.sample_p_zs_given_zt after the denoiser call
// (models/ligand_diffuser.py:515-536) and remove_com (:185-203) of the reference, which run
// ~25 small ATen kernels plus a DGL segment-mean per step.
//
// One CTA per complex.  Arithmetic is deliberately unfused (__fdiv_rn/__fmul_rn/__fsub_rn/
// __fadd_rn) and the COM is a sequential sum in atom order, so with injected noise the state
// after a step is bit-identical to the op-by-op PyTorch evaluation the oracle performs.
// HBM-bound: 2 x (3+F) floats read + (3+F) written per ligand atom, 6 floats per keypoint.
#include "common.cuh"
#include "philox.cuh"

namespace kpd {

// MULTISTEP = true: DPM-Solver++(2M) (DESIGN.md section 6.5).  Row s is then a DDIM eta = 0 row, and the step adds
//   x^ = (z - sigma_t eps) / alpha_t,  z_s += c (x^ - x^_prev)      (c, alpha_t, sigma_t) = row s of ms_coef
// except on the first row the run executes (RunParams.T - 1, or first_row of a stand-alone call), which neither reads
// the history nor corrects: 0 * an unwritten history could be NaN.
// x^ replaces the history, which then moves with the ligand COM (positions only), so it is always in the frame of the
// next step.  MULTISTEP = false is the plain step and ignores msp / msv / first_row.
template <bool MULTISTEP>
__global__ void __launch_bounds__(128)
ddpm_step_kernel(kpd_batch b, float* __restrict__ x_lig, float* __restrict__ h_lig, float* __restrict__ x_kp,
                 const float* __restrict__ eps_x, const float* __restrict__ eps_h, int F,
                 const float* __restrict__ coef, const int* __restrict__ step_ptr,
                 const float* noise_x, const float* noise_h, uint64_t seed, const RunParams* rp,
                 const MultistepParams* msp, MultistepParams msv, int first_row) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    const int s = *step_ptr;
    const float a = coef[4 * s], vt = coef[4 * s + 1], sg = coef[4 * s + 2];
    const StepDraws d = step_draws(rp, noise_x, seed, s, 1, 0, (size_t)b.n_lig * (3 + F));
    if (rp) noise_h = d.noise ? d.noise + (size_t)b.n_lig * 3 : nullptr;   // a run's slot holds x, then h
    __shared__ float com[3];
    MultistepParams m{};
    float mc = 0.0f, ma = 1.0f, ms = 0.0f;
    bool corr = false;
    if constexpr (MULTISTEP) {
        m = msp ? *msp : msv;
        mc = m.ms_coef[4 * s]; ma = m.ms_coef[4 * s + 1]; ms = m.ms_coef[4 * s + 2];
        corr = s != (rp ? rp->T - 1 : first_row);
    }
    // mu = z/alpha_t|s - var_terms*eps ; z_s = mu + sigma*noise   (ligand_diffuser.py:522-533)
    for (int i = threadIdx.x; i < nl * 3; i += blockDim.x) {
        const int idx = 3 * l0 + i;
        const float nz = d.noise ? d.noise[idx] : philox_normal(d.seed, s, d.atom_offset + l0 + i / 3, i % 3);
        if constexpr (MULTISTEP) {
            const float z = x_lig[idx], e = eps_x[idx];
            const float zs = __fadd_rn(__fsub_rn(__fdiv_rn(z, a), __fmul_rn(vt, e)), __fmul_rn(sg, nz));
            const float xh = __fdiv_rn(__fsub_rn(z, __fmul_rn(ms, e)), ma);
            x_lig[idx] = corr ? __fadd_rn(zs, __fmul_rn(mc, __fsub_rn(xh, m.hist_x[idx]))) : zs;
            m.hist_x[idx] = xh;
        } else {
            const float mu = __fsub_rn(__fdiv_rn(x_lig[idx], a), __fmul_rn(vt, eps_x[idx]));
            x_lig[idx] = __fadd_rn(mu, __fmul_rn(sg, nz));
        }
    }
    for (int i = threadIdx.x; i < nl * F; i += blockDim.x) {
        const int idx = F * l0 + i;
        const float nz = noise_h ? noise_h[idx] : philox_normal(d.seed, s, d.atom_offset + l0 + i / F, 3 + i % F);
        if constexpr (MULTISTEP) {
            const float z = h_lig[idx], e = eps_h[idx];
            const float zs = __fadd_rn(__fsub_rn(__fdiv_rn(z, a), __fmul_rn(vt, e)), __fmul_rn(sg, nz));
            const float hh = __fdiv_rn(__fsub_rn(z, __fmul_rn(ms, e)), ma);
            h_lig[idx] = corr ? __fadd_rn(zs, __fmul_rn(mc, __fsub_rn(hh, m.hist_h[idx]))) : zs;
            m.hist_h[idx] = hh;
        } else {
            const float mu = __fsub_rn(__fdiv_rn(h_lig[idx], a), __fmul_rn(vt, eps_h[idx]));
            h_lig[idx] = __fadd_rn(mu, __fmul_rn(sg, nz));
        }
    }
    __syncthreads();
    remove_ligand_com(x_lig, x_kp, l0, nl, k0, nk, com);   // :536 -> :185-203
    if constexpr (MULTISTEP) sub3(m.hist_x, l0, nl, com);
}

int launch_ddpm_step(const kpd_batch* b, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                     const float* eps_h, int F, const float* coef, const int* step_ptr, const float* noise_x,
                     const float* noise_h, uint64_t seed, const RunParams* rp, cudaStream_t st,
                     const MultistepParams* msp, const MultistepParams* msv, int first_row) {
    prof_begin(PROF_STEP, st);
    if (msp || msv)
        ddpm_step_kernel<true><<<b->B, 128, 0, st>>>(*b, x_lig, h_lig, x_kp, eps_x, eps_h, F, coef, step_ptr, noise_x,
                                                     noise_h, seed, rp, msp, msv ? *msv : MultistepParams{}, first_row);
    else
        ddpm_step_kernel<false><<<b->B, 128, 0, st>>>(*b, x_lig, h_lig, x_kp, eps_x, eps_h, F, coef, step_ptr, noise_x,
                                                      noise_h, seed, rp, nullptr, MultistepParams{}, 0);
    const int rc = check_launch(msp || msv ? "ddpm_step_kernel<multistep>" : "ddpm_step_kernel");
    prof_end(PROF_STEP, st);
    return rc;
}

// which: 0 = ligand COM, 1 = keypoint COM.  shift != 0: subtract it from both node types.
__global__ void __launch_bounds__(128)
com_kernel(kpd_batch b, float* x_lig, float* x_kp, int which, int shift, float* com_out) {
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    __shared__ float com[3];
    mean3(which == 0 ? x_lig : x_kp, which == 0 ? l0 : k0, which == 0 ? nl : nk, com);
    if (com_out && threadIdx.x < 3) com_out[3 * c + threadIdx.x] = com[threadIdx.x];
    __syncthreads();
    if (!shift) return;
    sub3(x_lig, l0, nl, com);
    sub3(x_kp, k0, nk, com);
}

int launch_com(const kpd_batch* b, float* x_lig, float* x_kp, int which, int shift, float* com_out, cudaStream_t st) {
    com_kernel<<<b->B, 128, 0, st>>>(*b, x_lig, x_kp, which, shift, com_out);
    return check_launch("com_kernel");
}

__global__ void shift_kernel(float* x, const int* node_batch, int n, const float* v, float sign) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * n) return;
    const float d = v[3 * node_batch[i / 3] + i % 3];
    x[i] = sign > 0 ? __fadd_rn(x[i], d) : __fsub_rn(x[i], d);
}

int launch_shift(float* x, const int* node_batch, int n, const float* v, float sign, cudaStream_t st) {
    if (n <= 0) return 0;
    shift_kernel<<<cdiv(3 * n, 256), 256, 0, st>>>(x, node_batch, n, v, sign);
    return check_launch("shift_kernel");
}

// initial x_0 / h_0 (ligand_diffuser.py:366-367): Philox stream "step = -1", or noise slot 0
__global__ void randn_init_kernel(float* x_lig, float* h_lig, int n_lig, int F, uint64_t seed, const RunParams* rp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int W = 3 + F;
    if (i >= n_lig * W) return;
    const StepDraws d = step_draws(rp, nullptr, seed, -1, 1, 0, (size_t)n_lig * W);
    const int atom = i / W, ch = i % W;
    float v;
    if (d.noise) v = ch < 3 ? d.noise[3 * atom + ch] : d.noise[(size_t)3 * n_lig + (size_t)F * atom + (ch - 3)];
    else v = philox_normal(d.seed, -1, d.atom_offset + atom, ch);
    if (ch < 3) x_lig[3 * atom + ch] = v;
    else h_lig[F * atom + (ch - 3)] = v;
}

int launch_randn_init(float* x_lig, float* h_lig, int n_lig, int F, uint64_t seed, const RunParams* rp, cudaStream_t st) {
    if (n_lig <= 0) return 0;
    randn_init_kernel<<<cdiv(n_lig * (3 + F), 256), 256, 0, st>>>(x_lig, h_lig, n_lig, F, seed, rp);
    return check_launch("randn_init_kernel");
}

__global__ void scale_kernel(float* x, int n, float s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = x[i] * s;
}

int launch_scale(float* x, int n, float s, cudaStream_t st) {
    if (n <= 0) return 0;
    scale_kernel<<<cdiv(n, 256), 256, 0, st>>>(x, n, s);
    return check_launch("scale_kernel");
}

// atom type of every generated atom = argmax over its feature channels, lowest index on ties (reference test.py:199-203:
// torch.argmax(lig_feat, dim=1), then dataset.lig_atom_idx_to_element); NaN-free inputs assumed, like the reference
__global__ void decode_atom_types_kernel(const float* __restrict__ h, int n, int F, int* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* row = h + (size_t)i * F;
    float best = row[0];
    int arg = 0;
    for (int c = 1; c < F; ++c) {
        const float v = row[c];
        if (v > best) { best = v; arg = c; }
    }
    out[i] = arg;
}

// s = --counter; step = s; t_cur = coef[4 s + 3]   (ligand_diffuser.py:404-408)
__global__ void step_prologue_kernel(int* counter, int* step, float* t_cur, const float* coef) {
    const int s = *counter - 1;
    *counter = s;
    *step = s;
    *t_cur = coef[4 * s + 3];
}

int launch_step_prologue(int* counter, int* step, float* t_cur, const float* coef, cudaStream_t st) {
    step_prologue_kernel<<<1, 1, 0, st>>>(counter, step, t_cur, coef);
    return check_launch("step_prologue_kernel");
}

}  // namespace kpd

using namespace kpd;

extern "C" int kpd_ddpm_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp, const float* eps_x,
                             const float* eps_h, int32_t atom_nf, const float* coef, const int32_t* step_ptr,
                             const float* noise_x, const float* noise_h, uint64_t seed, void* stream) {
    KPD_REQUIRE(batch && x_lig && h_lig && x_kp && eps_x && eps_h && coef && step_ptr, "kpd_ddpm_step: null argument");
    KPD_REQUIRE((noise_x == nullptr) == (noise_h == nullptr), "kpd_ddpm_step: give both noise tensors or neither");
    return launch_ddpm_step(batch, x_lig, h_lig, x_kp, eps_x, eps_h, atom_nf, coef, step_ptr, noise_x, noise_h, seed,
                            nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_ddpm_multistep_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp,
                                       const float* eps_x, const float* eps_h, int32_t atom_nf, const float* coef,
                                       const float* ms_coef, const int32_t* step_ptr, int32_t first_row, float* hist_x,
                                       float* hist_h, const float* noise_x, const float* noise_h, uint64_t seed,
                                       void* stream) {
    KPD_REQUIRE(batch && x_lig && h_lig && x_kp && eps_x && eps_h && coef && ms_coef && step_ptr && hist_x && hist_h,
                "kpd_ddpm_multistep_step: null argument");
    KPD_REQUIRE((noise_x == nullptr) == (noise_h == nullptr),
                "kpd_ddpm_multistep_step: give both noise tensors or neither");
    KPD_REQUIRE(first_row >= 0, "kpd_ddpm_multistep_step: first_row must be >= 0");
    const MultistepParams msv{ms_coef, hist_x, hist_h};
    return launch_ddpm_step(batch, x_lig, h_lig, x_kp, eps_x, eps_h, atom_nf, coef, step_ptr, noise_x, noise_h, seed,
                            nullptr, static_cast<cudaStream_t>(stream), nullptr, &msv, first_row);
}

extern "C" int kpd_remove_com(const kpd_batch* batch, float* x_lig, float* x_kp, int32_t which, float* com_out,
                              void* stream) {
    KPD_REQUIRE(batch && x_lig && x_kp, "kpd_remove_com: null argument");
    KPD_REQUIRE(which == 0 || which == 1, "kpd_remove_com: which must be 0 (ligand) or 1 (keypoints)");
    return launch_com(batch, x_lig, x_kp, which, 1, com_out, static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_shift_by_complex(float* x, const int32_t* node_batch, int32_t n, const float* v, float sign,
                                    void* stream) {
    KPD_REQUIRE(x && node_batch && v, "kpd_shift_by_complex: null argument");
    return launch_shift(x, node_batch, n, v, sign, static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_randn_init(float* x_lig, float* h_lig, int32_t n_lig, int32_t atom_nf, uint64_t seed, void* stream) {
    KPD_REQUIRE(x_lig && h_lig, "kpd_randn_init: null argument");
    return launch_randn_init(x_lig, h_lig, n_lig, atom_nf, seed, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_decode_atom_types(const float* h_lig, int32_t n_lig, int32_t atom_nf, int32_t* atom_type, void* stream) {
    KPD_REQUIRE(h_lig && atom_type && atom_nf >= 1 && n_lig >= 0, "kpd_decode_atom_types: bad argument");
    if (n_lig == 0) return 0;
    decode_atom_types_kernel<<<kpd::cdiv(n_lig, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(h_lig, n_lig, atom_nf, atom_type);
    return kpd::check_launch("decode_atom_types_kernel");
}
