// Trajectory recording: one frame of the reverse-diffusion run, written from inside the captured step
// (visualize=True of sample_from_encoded_receptors; DESIGN.md section 6.4).
//
// A recording sampler (kpd_sampler_enable_recording) launches record_frame_kernel between the step's first denoiser
// pass and its posterior step.  The step index lives on the device, so the kernel itself decides whether this step is
// recorded: executed step i = T - 1 - s (T = RunParams.T, the row the run started from) is frame j = i / every when
// i % every == 0.  One CTA per complex:
//   c      = the complex's keypoint mean (mean3: sequential sum in atom order, like com_kernel)
//   frame  x_f = (x - c) + init_kp_com,   h_f = h * norm_c
//   pred   x^  = (x - sigma_t eps_x) / alpha_t,  h^ = (h - sigma_t eps_h) / alpha_t,  moved to the same frame
// (alpha_t, sigma_t) is row s of RecordParams.pred_coef.  The frame arithmetic is the final restore's (com_kernel,
// shift_kernel, scale_kernel), unfused, so state frame j equals the output of a run stopped after step j*every bit for
// bit.  The kernel only reads the state: draws, noise slots and outputs are those of a run without recording.
#include "common.cuh"

namespace kpd {

__global__ void __launch_bounds__(128)
record_frame_kernel(kpd_batch b, const float* __restrict__ x_lig, const float* __restrict__ h_lig,
                    const float* __restrict__ x_kp, const float* __restrict__ eps_x, const float* __restrict__ eps_h,
                    int F, const int* __restrict__ step_ptr, const RunParams* __restrict__ rp,
                    const RecordParams* __restrict__ rec, const float* __restrict__ init_kp_com, float norm_c) {
    const RecordParams r = *rec;
    const int s = *step_ptr;
    const int i = rp->T - 1 - s;
    if (!r.x_frames || i % r.every != 0) return;
    const size_t j = i / r.every;
    const int c = blockIdx.x;
    const int l0 = b.lig_ptr[c], nl = b.lig_ptr[c + 1] - l0;
    const int k0 = b.kp_ptr[c], nk = b.kp_ptr[c + 1] - k0;
    const float a = r.pred_coef[2 * s], sg = r.pred_coef[2 * s + 1];
    __shared__ float com[3];
    mean3(x_kp, k0, nk, com);
    __syncthreads();
    float* xf = r.x_frames + j * b.n_lig * 3;
    float* xp = r.x_pred + j * b.n_lig * 3;
    for (int t = threadIdx.x; t < nl * 3; t += blockDim.x) {
        const int idx = 3 * l0 + t;
        const float x = x_lig[idx], o = init_kp_com[3 * c + t % 3];
        const float xh = __fdiv_rn(__fsub_rn(x, __fmul_rn(sg, eps_x[idx])), a);
        xf[idx] = __fadd_rn(__fsub_rn(x, com[t % 3]), o);
        xp[idx] = __fadd_rn(__fsub_rn(xh, com[t % 3]), o);
    }
    float* hf = r.h_frames + j * b.n_lig * F;
    float* hp = r.h_pred + j * b.n_lig * F;
    const bool scale = norm_c != 1.0f;
    for (int t = threadIdx.x; t < nl * F; t += blockDim.x) {
        const int idx = F * l0 + t;
        const float h = h_lig[idx];
        const float hh = __fdiv_rn(__fsub_rn(h, __fmul_rn(sg, eps_h[idx])), a);
        hf[idx] = scale ? __fmul_rn(h, norm_c) : h;
        hp[idx] = scale ? __fmul_rn(hh, norm_c) : hh;
    }
}

int launch_record_frame(const kpd_batch* b, const float* x_lig, const float* h_lig, const float* x_kp,
                        const float* eps_x, const float* eps_h, int F, const int* step_ptr, const RunParams* rp,
                        const RecordParams* rec, const float* init_kp_com, float norm_c, cudaStream_t st) {
    record_frame_kernel<<<b->B, 128, 0, st>>>(*b, x_lig, h_lig, x_kp, eps_x, eps_h, F, step_ptr, rp, rec, init_kp_com,
                                              norm_c);
    return check_launch("record_frame_kernel");
}

}  // namespace kpd
