// The 1000-step reverse-diffusion loop as a replayed CUDA graph.
//
// Replaces the body of KeypointDiffusion.sample_from_encoded_receptors
// (models/ligand_diffuser.py:342-447, visualize=False) of the reference, where every step runs
// a Python loop that mutates a DGL graph on the host and launches O(10^2) small kernels.
// Here a step is a fixed kernel sequence
//     step_prologue -> graph_mark/scan/fill -> denoiser -> ddpm_step
// with all shapes static (edge arrays sized at capacity, counts on the device), so it is
// captured once into a CUDA graph of `steps_per_graph` steps and replayed T/steps_per_graph
// times; the step index lives on the device and is decremented by step_prologue.  An inpainting sampler
// (kpd_sampler_enable_inpainting) runs r passes per step instead:
//     step_prologue -> r x (graph_mark/scan/fill -> denoiser -> ddpm_inpaint_step [-> renoise])
// A run from a start ligand (kpd_sampler_set_start) replaces the frame setup by one partial_noise launch and starts the
// step counter at t0 instead of T; the captured graphs do not depend on the step, so they serve any t0.
// Fewer-step sampling (kpd_sampler_set_schedule) swaps the coefficient rows: the step kernels read the sampler's own
// [T,4] table, which every run fills from the active schedule, so one capture serves every schedule, eta and start.
// A recording sampler (kpd_sampler_enable_recording) adds record_frame_kernel after the step's first denoiser pass:
//     step_prologue -> graph_mark/scan/fill -> denoiser -> record_frame -> ddpm_step
// and the kernel picks its frame slot from the device step counter, so the same graphs serve any stride or buffers.
// A multistep sampler (kpd_sampler_enable_multistep) captures the DPM-Solver++(2M) instantiation of the step kernel in
// place of the plain one (same launch count); its rows and history buffers are re-pointed per run like the recording's.
#include "common.cuh"
#include <string.h>

using namespace kpd;

struct kpd_sampler {
    kpd_sampler_config cfg;
    const void* model;
    kpd_batch batch;
    kpd_graph_params gp;
    kpd_csr ll, kl, lk, kk;
    const float* coef;        // create-time tables: the default schedule (T unit steps)
    int has_lk;
    // the active schedule (kpd_sampler_set_schedule): NULL = the create-time tables, else sched_rows rows of each
    const float *sched_coef, *sched_coef2;
    int sched_rows;
    // device state carved from the caller's workspace
    float *x_lig, *h_lig, *x_kp, *h_kp, *v_kp, *eps_h, *eps_x, *kp_enc, *init_kp_com, *init_lig_pos, *t_cur;
    float* coef_run;          // [T][4]: the rows of the active schedule, copied in by every run; what the steps read
    int *counter, *step;
    long long* edge_accum;
    RunParams* rp;
    void* graph_ws;
    void* model_ws;
    int kp_width, v_width;
    // capture
    cudaStream_t stream;
    cudaEvent_t ev_in, ev_out;
    cudaGraph_t graph;
    cudaGraphExec_t exec;
    int launches_per_step;
    int atom_offset;
    // fragment-conditioned sampling (kpd_sampler_enable_inpainting): 0 = plain loop, else resamplings per step
    int resamplings;
    InpaintParams frag;       // host copy with the create-time coef2; every run uploads it with the active coef2
    InpaintParams* frag_dev;
    // partial noising (kpd_sampler_set_start): x_start == NULL = the plain start from pure noise at step T
    const float *x_start, *h_start;
    int start_step;
    float start_alpha, start_sigma;
    // trajectory recording (kpd_sampler_enable_recording): rec_dev == NULL = no record_frame launch in the step
    RecordParams rec;         // host copy; x_frames == NULL records nothing.  Every run uploads it
    RecordParams* rec_dev;
    int rec_frames, rec_rows;
    // DPM-Solver++(2M) (kpd_sampler_enable_multistep): ms_dev == NULL = the plain step kernel
    MultistepParams ms;       // host copy; every run uploads it
    MultistepParams* ms_dev;
    int ms_rows;
};

static int64_t model_ws_bytes(const kpd_sampler_config* cfg, const void* model, const kpd_batch* b, int cap_ll,
                              int cap_kl, int cap_kk) {
    return cfg->arch == 0 ? kpd_egnn_workspace_bytes(static_cast<const kpd_egnn_model*>(model), b, cap_ll, cap_kl, cap_kk)
                          : kpd_gvp_workspace_bytes(static_cast<const kpd_gvp_model*>(model), b, cap_ll, cap_kl, cap_kk);
}

static int carve_sampler(kpd_sampler* s, void* ws, int cap_ll, int cap_kl, int64_t* bytes) {
    const kpd_batch& b = s->batch;
    Carver c(ws);
    const int F = s->cfg.atom_nf;
    s->ll.n_dst = b.n_lig; s->ll.cap = cap_ll;
    s->ll.rowptr = c.take<int>(b.n_lig + 1); s->ll.src = c.take<int>(cap_ll + 1); s->ll.dst = c.take<int>(cap_ll + 1);
    s->kl.n_dst = b.n_lig; s->kl.cap = cap_kl;
    s->kl.rowptr = c.take<int>(b.n_lig + 1); s->kl.src = c.take<int>(cap_kl + 1); s->kl.dst = c.take<int>(cap_kl + 1);
    s->lk.n_dst = b.n_kp; s->lk.cap = cap_kl;
    s->lk.rowptr = c.take<int>(b.n_kp + 1); s->lk.src = c.take<int>(cap_kl + 1); s->lk.dst = c.take<int>(cap_kl + 1);
    s->counter = c.take<int>(4);
    s->step = s->counter + 1;
    s->x_lig = c.take<float>((int64_t)b.n_lig * 3);
    s->h_lig = c.take<float>((int64_t)b.n_lig * F);
    s->x_kp = c.take<float>((int64_t)b.n_kp * 3);
    s->h_kp = c.take<float>((int64_t)b.n_kp * s->kp_width);
    s->v_kp = c.take<float>((int64_t)b.n_kp * (s->v_width > 0 ? s->v_width : 1));
    s->eps_h = c.take<float>((int64_t)b.n_lig * F);
    s->eps_x = c.take<float>((int64_t)b.n_lig * 3);
    int rec_nf = 0, hid = 0;
    if (s->cfg.arch == 0) kpd_egnn_dims(static_cast<const kpd_egnn_model*>(s->model), &rec_nf, &hid);
    s->kp_enc = c.take<float>((int64_t)b.n_kp * (hid > 0 ? hid : 1));
    s->init_kp_com = c.take<float>((int64_t)b.B * 3);
    s->init_lig_pos = c.take<float>((int64_t)b.B * 3);
    s->t_cur = c.take<float>(4);
    s->coef_run = c.take<float>((int64_t)s->cfg.T * 4);
    s->rp = c.take<RunParams>(1);
    s->edge_accum = c.take<long long>(4);
    s->graph_ws = c.take<char>(kpd_graph_workspace_bytes(&b));
    s->model_ws = c.take<char>(model_ws_bytes(&s->cfg, s->model, &b, cap_ll, cap_kl, s->kk.cap));
    if (bytes) *bytes = c.bytes();
    return 0;
}

static int fill_dims(kpd_sampler* s) {
    if (s->cfg.arch == 0) {
        int rec_nf = 0, hid = 0;
        KPD_TRY(kpd_egnn_dims(static_cast<const kpd_egnn_model*>(s->model), &rec_nf, &hid));
        s->kp_width = rec_nf; s->v_width = 0;
    } else {
        int c = 0, v = 0;
        KPD_TRY(kpd_gvp_dims(static_cast<const kpd_gvp_model*>(s->model), &c, &v));
        s->kp_width = c; s->v_width = v * 3;
    }
    return 0;
}

extern "C" int64_t kpd_sampler_workspace_bytes(const kpd_sampler_config* cfg, const void* model, const kpd_batch* batch,
                                               int32_t cap_ll, int32_t cap_kl, int32_t cap_kk) {
    kpd_sampler s;
    memset(&s, 0, sizeof(s));
    s.cfg = *cfg; s.model = model; s.batch = *batch; s.kk.cap = cap_kk;
    if (fill_dims(&s) != 0) return -1;
    int64_t bytes = 0;
    carve_sampler(&s, nullptr, cap_ll, cap_kl, &bytes);
    return bytes;
}

// graph build + denoiser on the current state
static int enqueue_denoiser(kpd_sampler* s, cudaStream_t st) {
    KPD_TRY(build_graph_impl(&s->batch, s->x_lig, s->x_kp, &s->gp, &s->ll, &s->kl, s->has_lk ? &s->lk : nullptr,
                             nullptr, nullptr, s->graph_ws, s->edge_accum, st));
    if (s->cfg.arch == 0)
        return kpd_egnn_forward(static_cast<const kpd_egnn_model*>(s->model), &s->batch, s->h_lig, s->x_lig, s->h_kp,
                                s->x_kp, s->kp_enc, s->t_cur, 0, &s->ll, &s->kl, s->has_lk ? &s->lk : nullptr,
                                s->has_lk ? &s->kk : nullptr, s->eps_h, s->eps_x, s->model_ws, st);
    return kpd_gvp_forward(static_cast<const kpd_gvp_model*>(s->model), &s->batch, s->h_lig, s->x_lig, s->h_kp, s->x_kp,
                           s->v_kp, s->t_cur, 0, &s->ll, &s->kl, s->has_lk ? &s->lk : nullptr,
                           s->has_lk ? &s->kk : nullptr, s->eps_h, s->eps_x, s->model_ws, st);
}

// the frame of a recording sampler: the state after the prologue and the first denoiser pass's eps
static int enqueue_record(kpd_sampler* s, cudaStream_t st) {
    if (!s->rec_dev) return 0;
    return launch_record_frame(&s->batch, s->x_lig, s->h_lig, s->x_kp, s->eps_x, s->eps_h, s->cfg.atom_nf, s->step,
                               s->rp, s->rec_dev, s->init_kp_com, s->cfg.lig_feat_norm_constant, st);
}

static int enqueue_step(kpd_sampler* s, cudaStream_t st) {
    KPD_TRY(launch_step_prologue(s->counter, s->step, s->t_cur, s->coef_run, st));
    KPD_TRY(enqueue_denoiser(s, st));
    KPD_TRY(enqueue_record(s, st));
    KPD_TRY(launch_ddpm_step(&s->batch, s->x_lig, s->h_lig, s->x_kp, s->eps_x, s->eps_h, s->cfg.atom_nf, s->coef_run,
                             s->step, nullptr, nullptr, 0, s->rp, st, s->ms_dev));
    return 0;
}

// one reverse step of the inpainting loop: prologue, then r x (graph build, denoiser, inpaint step[, re-noise])
static int enqueue_inpaint_step(kpd_sampler* s, cudaStream_t st) {
    const int r = s->resamplings, F = s->cfg.atom_nf;
    KPD_TRY(launch_step_prologue(s->counter, s->step, s->t_cur, s->coef_run, st));
    for (int u = 0; u < r; ++u) {
        KPD_TRY(enqueue_denoiser(s, st));
        if (u == 0) KPD_TRY(enqueue_record(s, st));
        KPD_TRY(launch_ddpm_inpaint_step(&s->batch, s->x_lig, s->h_lig, s->x_kp, s->eps_x, s->eps_h, F, s->coef_run,
                                         s->step, u, r, InpaintParams{}, s->frag_dev, s->init_kp_com,
                                         s->cfg.lig_feat_norm_constant, nullptr, 0, s->rp, st));
        if (u < r - 1)
            KPD_TRY(launch_renoise(&s->batch, s->x_lig, s->h_lig, s->x_kp, F, s->step, u, r, nullptr, s->frag_dev,
                                   nullptr, 0, s->rp, st));
    }
    return 0;
}

extern "C" int kpd_sampler_create(const kpd_sampler_config* cfg, const void* model, const kpd_batch* batch,
                                  const kpd_graph_params* gp, const kpd_csr* kk, int32_t has_lk, const float* coef,
                                  int32_t cap_ll, int32_t cap_kl, void* workspace, int64_t workspace_bytes,
                                  kpd_sampler** out) {
    KPD_REQUIRE(cfg && model && batch && gp && coef && workspace && out, "kpd_sampler_create: null argument");
    KPD_REQUIRE(cfg->arch == 0 || cfg->arch == 1, "kpd_sampler_create: arch must be 0 (egnn) or 1 (gvp)");
    KPD_REQUIRE(cfg->T >= 1 && cfg->steps_per_graph >= 1, "kpd_sampler_create: bad T / steps_per_graph");
    KPD_REQUIRE(!has_lk || kk, "kpd_sampler_create: keypoint updates need the kk graph");
    auto* s = new kpd_sampler();
    memset(s, 0, sizeof(*s));
    s->cfg = *cfg; s->model = model; s->batch = *batch; s->gp = *gp; s->coef = coef; s->has_lk = has_lk;
    if (kk) s->kk = *kk;
    if (fill_dims(s) != 0) { delete s; return -1; }
    int64_t need = 0;
    carve_sampler(s, workspace, cap_ll, cap_kl, &need);
    if (need > workspace_bytes) { delete s; KPD_REQUIRE(false, "kpd_sampler_create: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)need); }
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_out, cudaEventDisableTiming);
    if (e != cudaSuccess) { delete s; KPD_REQUIRE(false, "kpd_sampler_create: %s", cudaGetErrorString(e)); }
    *out = s;
    return 0;
}

extern "C" void kpd_sampler_destroy(kpd_sampler* s) {
    if (!s) return;
    if (s->exec) cudaGraphExecDestroy(s->exec);
    if (s->frag_dev) cudaFree(s->frag_dev);
    if (s->rec_dev) cudaFree(s->rec_dev);
    if (s->ms_dev) cudaFree(s->ms_dev);
    if (s->graph) cudaGraphDestroy(s->graph);
    if (s->ev_in) cudaEventDestroy(s->ev_in);
    if (s->ev_out) cudaEventDestroy(s->ev_out);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

// mean edges per reverse step of the last run: out = {E_ll, E_kl (= E_lk), E_kk, steps}.  Synchronises.
extern "C" int kpd_sampler_edge_stats(kpd_sampler* s, double* out) {
    KPD_REQUIRE(s && out, "kpd_sampler_edge_stats: null argument");
    long long h[4] = {0, 0, 0, 0};
    int e_kk = 0;
    cudaError_t e = cudaStreamSynchronize(s->stream);
    if (e == cudaSuccess) e = cudaMemcpy(h, s->edge_accum, sizeof(h), cudaMemcpyDeviceToHost);
    // the kk edge count lives on the device like every other (rowptr[n_dst]); cap is only the capacity of the arrays
    if (e == cudaSuccess && s->has_lk) e = cudaMemcpy(&e_kk, s->kk.rowptr + s->kk.n_dst, sizeof(int), cudaMemcpyDeviceToHost);
    KPD_REQUIRE(e == cudaSuccess, "kpd_sampler_edge_stats: %s", cudaGetErrorString(e));
    const double n = h[2] > 0 ? (double)h[2] : 1.0;
    out[0] = h[0] / n; out[1] = h[1] / n; out[2] = s->has_lk ? (double)e_kk : 0.0; out[3] = (double)h[2];
    return 0;
}

extern "C" int32_t kpd_sampler_launches_per_step(const kpd_sampler* s) { return s ? s->launches_per_step : 0; }

// A batch may be sampled as several sub-batches on their own streams (their kernels fill each other's idle SMs); with
// the sub-batch's first global ligand-atom index as offset the generated noise does not depend on the split.
extern "C" int kpd_sampler_set_atom_offset(kpd_sampler* s, int32_t first_atom) {
    KPD_REQUIRE(s && first_atom >= 0, "kpd_sampler_set_atom_offset: bad argument");
    s->atom_offset = first_atom;
    return 0;
}

extern "C" int kpd_sampler_enable_inpainting(kpd_sampler* s, int32_t resamplings, const float* coef2) {
    KPD_REQUIRE(s && coef2 && resamplings >= 1, "kpd_sampler_enable_inpainting: bad argument");
    KPD_REQUIRE(!s->exec && !s->resamplings, "kpd_sampler_enable_inpainting: the sampler has already run or is inpainting");
    KPD_REQUIRE(!s->ms_dev, "kpd_sampler_enable_inpainting: a multistep sampler cannot inpaint");
    KPD_REQUIRE(sizeof(float) * 3 * (size_t)s->batch.max_lig <= 48 * 1024,
                "kpd_sampler_enable_inpainting: %d atoms in one complex exceed the supported 4096", s->batch.max_lig);
    const cudaError_t e = cudaMalloc(&s->frag_dev, sizeof(InpaintParams));
    KPD_REQUIRE(e == cudaSuccess, "kpd_sampler_enable_inpainting: %s", cudaGetErrorString(e));
    s->resamplings = resamplings;
    s->frag = InpaintParams{nullptr, nullptr, nullptr, coef2};
    return 0;
}

extern "C" int kpd_sampler_set_fragment(kpd_sampler* s, const uint8_t* fixed_mask, const float* x_fix, const float* h_fix) {
    KPD_REQUIRE(s && s->resamplings, "kpd_sampler_set_fragment: not an inpainting sampler");
    KPD_REQUIRE(!fixed_mask || (x_fix && h_fix), "kpd_sampler_set_fragment: a fixed mask needs x_fix and h_fix");
    s->frag.mask = fixed_mask; s->frag.x_fix = x_fix; s->frag.h_fix = h_fix;
    return 0;
}

extern "C" int kpd_sampler_set_start(kpd_sampler* s, int32_t start_step, const float* x_start, const float* h_start,
                                     float alpha, float sigma) {
    KPD_REQUIRE(s, "kpd_sampler_set_start: null sampler");
    KPD_REQUIRE(!x_start || (h_start && start_step >= 0 && start_step <= s->cfg.T),
                "kpd_sampler_set_start: a start ligand needs h_start and a start step in [0, T]");
    s->x_start = x_start; s->h_start = x_start ? h_start : nullptr;
    s->start_step = x_start ? start_step : 0;
    s->start_alpha = alpha; s->start_sigma = sigma;
    return 0;
}

extern "C" int kpd_sampler_set_schedule(kpd_sampler* s, int32_t n_rows, const float* coef, const float* coef2) {
    KPD_REQUIRE(s, "kpd_sampler_set_schedule: null sampler");
    if (!coef) {
        s->sched_coef = s->sched_coef2 = nullptr;
        s->sched_rows = 0;
        return 0;
    }
    KPD_REQUIRE(n_rows >= 1 && n_rows <= s->cfg.T, "kpd_sampler_set_schedule: %d rows outside [1, T = %d]", n_rows,
                s->cfg.T);
    KPD_REQUIRE(!s->resamplings || coef2, "kpd_sampler_set_schedule: an inpainting sampler needs coef2");
    s->sched_coef = coef; s->sched_coef2 = coef2; s->sched_rows = n_rows;
    return 0;
}

extern "C" int kpd_sampler_enable_recording(kpd_sampler* s) {
    KPD_REQUIRE(s, "kpd_sampler_enable_recording: null sampler");
    KPD_REQUIRE(!s->exec && !s->rec_dev, "kpd_sampler_enable_recording: the sampler has already run or is recording");
    const cudaError_t e = cudaMalloc(&s->rec_dev, sizeof(RecordParams));
    KPD_REQUIRE(e == cudaSuccess, "kpd_sampler_enable_recording: %s", cudaGetErrorString(e));
    s->rec = RecordParams{1, nullptr, nullptr, nullptr, nullptr, nullptr};
    return 0;
}

extern "C" int kpd_sampler_set_recording(kpd_sampler* s, int32_t every, int32_t n_frames, float* x_frames,
                                         float* h_frames, float* x_pred, float* h_pred, int32_t n_pred_rows,
                                         const float* pred_coef) {
    KPD_REQUIRE(s && s->rec_dev, "kpd_sampler_set_recording: not a recording sampler");
    if (!x_frames) {
        s->rec = RecordParams{1, nullptr, nullptr, nullptr, nullptr, nullptr};
        s->rec_frames = s->rec_rows = 0;
        return 0;
    }
    KPD_REQUIRE(every >= 1 && n_frames >= 1 && h_frames && pred_coef && n_pred_rows >= 1,
                "kpd_sampler_set_recording: bad argument");
    KPD_REQUIRE(n_frames == 1 || (x_pred && h_pred), "kpd_sampler_set_recording: prediction frames need buffers");
    s->rec = RecordParams{every, x_frames, h_frames, x_pred, h_pred, pred_coef};
    s->rec_frames = n_frames;
    s->rec_rows = n_pred_rows;
    return 0;
}

extern "C" int kpd_sampler_enable_multistep(kpd_sampler* s) {
    KPD_REQUIRE(s, "kpd_sampler_enable_multistep: null sampler");
    KPD_REQUIRE(!s->exec && !s->ms_dev, "kpd_sampler_enable_multistep: the sampler has already run or is multistep");
    KPD_REQUIRE(!s->resamplings, "kpd_sampler_enable_multistep: an inpainting sampler cannot run multistep steps");
    const cudaError_t e = cudaMalloc(&s->ms_dev, sizeof(MultistepParams));
    KPD_REQUIRE(e == cudaSuccess, "kpd_sampler_enable_multistep: %s", cudaGetErrorString(e));
    s->ms = MultistepParams{nullptr, nullptr, nullptr};
    return 0;
}

extern "C" int kpd_sampler_set_multistep(kpd_sampler* s, int32_t n_rows, const float* ms_coef, float* hist_x,
                                         float* hist_h) {
    KPD_REQUIRE(s && s->ms_dev, "kpd_sampler_set_multistep: not a multistep sampler");
    KPD_REQUIRE(ms_coef && hist_x && hist_h && n_rows >= 1, "kpd_sampler_set_multistep: bad argument");
    s->ms = MultistepParams{ms_coef, hist_x, hist_h};
    s->ms_rows = n_rows;
    return 0;
}

static int enqueue_any_step(kpd_sampler* s, cudaStream_t st) {
    return s->resamplings ? enqueue_inpaint_step(s, st) : enqueue_step(s, st);
}

static int capture(kpd_sampler* s) {
    cudaError_t e = cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal);
    KPD_REQUIRE(e == cudaSuccess, "sampler: begin capture: %s", cudaGetErrorString(e));
    int rc = 0;
    for (int i = 0; i < s->cfg.steps_per_graph && rc == 0; ++i) rc = enqueue_any_step(s, s->stream);
    e = cudaStreamEndCapture(s->stream, &s->graph);
    if (rc != 0) return rc;
    KPD_REQUIRE(e == cudaSuccess, "sampler: end capture: %s", cudaGetErrorString(e));
    // per-node priorities: the denoisers mark their critical-path kernels (kpd_gvp_forward) and those must be dispatched
    // ahead of already-queued CTAs of lower-priority kernels, whatever the priority of the launching stream
    e = cudaGraphInstantiateWithFlags(&s->exec, s->graph, cudaGraphInstantiateFlagUseNodePriority);
    KPD_REQUIRE(e == cudaSuccess, "sampler: graph instantiate: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int kpd_sampler_run(kpd_sampler* s, float* x_kp, const float* h_kp, const float* v_kp,
                               const float* init_lig_pos, float* x_lig, float* h_lig, const float* noise,
                               uint64_t seed, int32_t n_steps, void* stream) {
    KPD_REQUIRE(s && x_kp && h_kp && init_lig_pos && x_lig && h_lig, "kpd_sampler_run: null argument");
    KPD_REQUIRE(s->cfg.arch == 0 || v_kp, "kpd_sampler_run: the GVP denoiser needs keypoint vectors v_kp");
    // the first executed reverse step is row t0 - 1 of the active schedule: t0 = its row count from pure noise, the
    // start step from a start ligand
    const int rows = s->sched_coef ? s->sched_rows : s->cfg.T;
    const float* coef = s->sched_coef ? s->sched_coef : s->coef;
    const int t0 = s->x_start ? s->start_step : rows;
    KPD_REQUIRE(t0 <= rows, "kpd_sampler_run: start step %d beyond the %d rows of the schedule", t0, rows);
    KPD_REQUIRE(!s->resamplings || !s->sched_coef || s->sched_coef2, "kpd_sampler_run: the schedule has no coef2");
    KPD_REQUIRE(n_steps >= 0 && n_steps <= t0, "kpd_sampler_run: n_steps out of range");
    // what keeps record_frame_kernel inside its buffers: frame j <= (n_steps-1) / every, prediction row s < rows
    KPD_REQUIRE(!s->rec.x_frames || s->rec_frames == (n_steps + s->rec.every - 1) / s->rec.every + 1,
                "kpd_sampler_run: %d frames recorded every %d steps need %d buffers, got %d", n_steps, s->rec.every,
                (n_steps + s->rec.every - 1) / s->rec.every + 1, s->rec_frames);
    KPD_REQUIRE(!s->rec.x_frames || s->rec_rows == rows,
                "kpd_sampler_run: %d prediction rows for a schedule of %d rows", s->rec_rows, rows);
    // what keeps the multistep step kernel inside its rows: row s < rows of the active schedule
    KPD_REQUIRE(!s->ms_dev || s->ms.ms_coef, "kpd_sampler_run: a multistep sampler needs kpd_sampler_set_multistep");
    KPD_REQUIRE(!s->ms_dev || s->ms_rows == rows, "kpd_sampler_run: %d multistep rows for a schedule of %d rows",
                s->ms_rows, rows);
    const kpd_batch& b = s->batch;
    const int F = s->cfg.atom_nf;
    cudaStream_t user = static_cast<cudaStream_t>(stream), st = s->stream;
    cudaError_t e;
#define CU(x) do { e = (x); KPD_REQUIRE(e == cudaSuccess, "kpd_sampler_run: %s: %s", #x, cudaGetErrorString(e)); } while (0)
    CU(cudaEventRecord(s->ev_in, user));
    CU(cudaStreamWaitEvent(st, s->ev_in, 0));
    CU(cudaMemcpyAsync(s->x_kp, x_kp, sizeof(float) * 3 * b.n_kp, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(s->h_kp, h_kp, sizeof(float) * (size_t)s->kp_width * b.n_kp, cudaMemcpyDeviceToDevice, st));
    if (s->v_width) CU(cudaMemcpyAsync(s->v_kp, v_kp, sizeof(float) * (size_t)s->v_width * b.n_kp, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(s->init_lig_pos, init_lig_pos, sizeof(float) * 3 * b.B, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(s->coef_run, coef, sizeof(float) * 4 * (size_t)rows, cudaMemcpyDeviceToDevice, st));
    RunParams rp;
    rp.noise = noise; rp.seed = seed; rp.T = t0; rp.atom_offset = s->atom_offset;
    int counter0[4] = {t0, t0, 0, 0};
    // small pageable H2D copies: staged by the runtime before the call returns
    CU(cudaMemcpyAsync(s->rp, &rp, sizeof(rp), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(s->counter, counter0, sizeof(counter0), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(s->edge_accum, 0, 4 * sizeof(long long), st));
    if (s->resamplings) {
        InpaintParams frag = s->frag;
        if (s->sched_coef) frag.coef2 = s->sched_coef2;
        CU(cudaMemcpyAsync(s->frag_dev, &frag, sizeof(InpaintParams), cudaMemcpyHostToDevice, st));
    }
    if (s->rec_dev) CU(cudaMemcpyAsync(s->rec_dev, &s->rec, sizeof(RecordParams), cudaMemcpyHostToDevice, st));
    if (s->ms_dev) CU(cudaMemcpyAsync(s->ms_dev, &s->ms, sizeof(MultistepParams), cudaMemcpyHostToDevice, st));

    // frame setup (ligand_diffuser.py:348-370)
    KPD_TRY(launch_com(&b, s->x_lig, s->x_kp, 1, 0, s->init_kp_com, st));                // init_kp_com (:348)
    if (s->x_start) {       // start ligand noised to t0 in the frame of its own mean (partial_noise.cu)
        KPD_TRY(launch_partial_noise(&b, s->x_start, s->h_start, s->x_lig, s->h_lig, s->x_kp, F, s->start_alpha,
                                     s->start_sigma, s->cfg.lig_feat_norm_constant, nullptr, seed, s->rp, st));
    } else {
        KPD_TRY(launch_shift(s->x_kp, b.kp_batch, b.n_kp, s->init_lig_pos, -1.0f, st));  // :363
        KPD_TRY(launch_randn_init(s->x_lig, s->h_lig, b.n_lig, F, seed, s->rp, st));     // :366-367
        KPD_TRY(launch_com(&b, s->x_lig, s->x_kp, 0, 1, nullptr, st));                   // :370
    }
    if (s->cfg.arch == 0)   // the EGNN keypoint encoder does not depend on t: hoisted out of the loop
        KPD_TRY(kpd_egnn_encode_kp(static_cast<const kpd_egnn_model*>(s->model), s->h_kp, b.n_kp, s->kp_enc, s->model_ws, st));

    int done = 0;
    if (s->cfg.use_cuda_graph) {
        if (!s->exec && n_steps >= s->cfg.steps_per_graph) {
            const long long l0 = launch_count();
            KPD_TRY(capture(s));
            s->launches_per_step = (int)((launch_count() - l0) / s->cfg.steps_per_graph);
        }
        while (s->exec && n_steps - done >= s->cfg.steps_per_graph) {
            CU(cudaGraphLaunch(s->exec, st));
            done += s->cfg.steps_per_graph;
        }
    }
    for (; done < n_steps; ++done) {
        const long long l0 = launch_count();
        KPD_TRY(enqueue_any_step(s, st));
        s->launches_per_step = (int)(launch_count() - l0);
    }
    // frame restore (:438-447)
    KPD_TRY(launch_com(&b, s->x_lig, s->x_kp, 1, 1, nullptr, st));
    KPD_TRY(launch_shift(s->x_lig, b.lig_batch, b.n_lig, s->init_kp_com, 1.0f, st));
    KPD_TRY(launch_shift(s->x_kp, b.kp_batch, b.n_kp, s->init_kp_com, 1.0f, st));
    if (s->cfg.lig_feat_norm_constant != 1.0f) KPD_TRY(launch_scale(s->h_lig, b.n_lig * F, s->cfg.lig_feat_norm_constant, st));
    CU(cudaMemcpyAsync(x_lig, s->x_lig, sizeof(float) * 3 * b.n_lig, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(h_lig, s->h_lig, sizeof(float) * (size_t)F * b.n_lig, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(x_kp, s->x_kp, sizeof(float) * 3 * b.n_kp, cudaMemcpyDeviceToDevice, st));
    if (s->rec.x_frames) {  // the last state frame is the output
        const size_t last = (size_t)(s->rec_frames - 1) * b.n_lig;
        CU(cudaMemcpyAsync(s->rec.x_frames + last * 3, s->x_lig, sizeof(float) * 3 * b.n_lig, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(s->rec.h_frames + last * F, s->h_lig, sizeof(float) * (size_t)F * b.n_lig,
                           cudaMemcpyDeviceToDevice, st));
    }
    CU(cudaEventRecord(s->ev_out, st));
    CU(cudaStreamWaitEvent(user, s->ev_out, 0));
#undef CU
    return 0;
}
