/*
 * kpdiff_b200 -- C ABI of the B200-native sampling hot path of keypoint-diffusion.
 *
 * The reference (Dunni3/keypoint-diffusion) is pure Python and has no FFI; its boundary for
 * this path is the Python module API (SURVEY.md section 8b).  This header is what a binding
 * for that path calls underneath the drop-in Python classes in keypoint_diffusion_b200/:
 * every entry point below names the reference interface it replaces (file:line relative to
 * the reference tree).  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the parameter is documented as host;
 *   - tensors are contiguous fp32 / int32, caller-owned (allocate with torch or cudaMalloc);
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it, never
 *     synchronises or allocates (so every call is CUDA-graph capturable) unless stated;
 *   - return value 0 = ok; otherwise kpd_last_error() describes the failure
 *     (the Python host turns it into RuntimeError);
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef KPDIFF_B200_H
#define KPDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KPD_TILE_EDGES 64      /* edges (or nodes) per CTA tile in the fused kernels          */
#define KPD_MAX_KNN 100        /* torch_cluster's own k limit                                  */
#define KPD_MAX_HIDDEN 260     /* EGNN hidden_nf+1 and GVP scalar width supported by the tiles */

const char* kpd_last_error(void);
int kpd_version(void);
/* kernels this library has launched in this process (captured launches count once) */
int64_t kpd_launch_count(void);
/* Optional CUDA-event timing of one kernel family for bench.py's roofline leg.  kernel_id:
 * 1 egnn_edge, 2 gvp_edge, 3 graph build, 4 ddpm_step, 5 gvp_node, 6 gvp_head, 7 egnn node
 * stage, 8 egnn per-node pre-GEMM; 0 disables.  Inactive during stream capture.
 * kpd_profile_collect synchronises on the recorded events and resets the record list. */
int kpd_profile_enable(int32_t kernel_id, int32_t max_records);
int kpd_profile_collect(double* total_ms, int32_t* count);

/* ------------------------------------------------------------------------------------------
 * Batch layout.  Replaces the DGL batched heterograph bookkeeping the path reads:
 * g.batch_size / g.batch_num_nodes(ntype) (utils.py:81-90) and get_batch_idxs (utils.py:158-170).
 * Nodes of one complex are contiguous; *_ptr are exclusive prefix sums of nodes per complex.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t B;                 /* complexes in the batch                                       */
    int32_t n_lig, n_kp;       /* total ligand atoms / keypoints                               */
    int32_t max_lig, max_kp;   /* largest complex (sizes shared memory)                        */
    const int32_t* lig_ptr;    /* [B+1]                                                        */
    const int32_t* kp_ptr;     /* [B+1]                                                        */
    const int32_t* lig_batch;  /* [n_lig] complex index per ligand atom                        */
    const int32_t* kp_batch;   /* [n_kp]                                                       */
} kpd_batch;

/* dst-sorted CSR + COO of one edge type.  n_edges lives on the device: rowptr[n_dst]. */
typedef struct {
    int32_t n_dst;             /* number of destination nodes                                  */
    int32_t cap;               /* capacity of src/dst in edges                                 */
    int32_t* rowptr;           /* [n_dst+1]                                                    */
    int32_t* src;              /* [cap] global index in the source node type                   */
    int32_t* dst;              /* [cap] global index in the destination node type              */
} kpd_csr;

/* ------------------------------------------------------------------------------------------
 * (a) Per-step graph construction.  Replaces LigRecDynamics.add_lig_edges /
 * remove_lig_edges (models/dynamics.py:387-442) and LigRecDynamicsGVP.add_lig_edges
 * (models/dynamics_gvp.py:201-255), i.e. torch_cluster.radius_graph / knn_graph / knn / radius
 * + DGL add_edges/remove_edges + utils.get_edges_per_batch (utils.py:92-98).
 * Emits dst-sorted CSR for ll (lig->lig), kl (kp->lig) and lk (lig->kp).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t ll_k;              /* >0: knn_graph with ll_k neighbours; 0: radius graph           */
    int32_t ll_cap;            /* max_num_neighbors of radius_graph (200 in the reference)      */
    int32_t kl_k;              /* >0: knn(x=lig,y=kp,k); 0: radius(x=lig,y=kp)                  */
    int32_t kl_cap;            /* max_num_neighbors of radius (100 in the reference)            */
    double  ll_r;              /* radius (graph_cutoffs['ll']); r*r is formed in double and
                                  rounded to fp32 once, as torch_cluster does                  */
    double  kl_r;              /* radius (graph_cutoffs['kl'])                                  */
} kpd_graph_params;

/* bytes of scratch kpd_build_graph needs for this batch (host computation, no device work) */
int64_t kpd_graph_workspace_bytes(const kpd_batch* batch);

/* Edge capacities are host arithmetic on the per-complex node counts (done by the caller):
 *   cap_ll = sum_b n_l * min(n_l - 1, ll_k > 0 ? ll_k : ll_cap)
 *   cap_kl = sum_b n_k * min(n_l,     kl_k > 0 ? kl_k : kl_cap)        (lk has the same capacity)
 * counts_ll / counts_kl (optional, [B]) receive the per-complex edge counts
 * (= utils.get_edges_per_batch). */
int kpd_build_graph(const kpd_batch* batch, const float* x_lig, const float* x_kp,
                    const kpd_graph_params* p, kpd_csr* ll, kpd_csr* kl, kpd_csr* lk,
                    int32_t* counts_ll /*[B] or NULL*/, int32_t* counts_kl /*[B] or NULL*/,
                    void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense row op used for the node-level linears ((d) in the north star):
 *   Y[m, 0:N] = act( X[m, 0:K] @ WT[0:K, 0:N] + bias ) (+ R[m, 0:N])
 * WT is K-major ([K][ldw], i.e. the transpose of nn.Linear.weight).  act: 0 none, 1 SiLU.
 * Replaces the nn.Linear / SiLU calls at models/dynamics.py:355-356, :202-204, :380.
 * ------------------------------------------------------------------------------------------ */
int kpd_linear(const float* X, int32_t ldx, const float* WT, int32_t ldw, const float* bias,
               const float* R, int32_t ldr, float* Y, int32_t ldy, int32_t M, int32_t K, int32_t N,
               int32_t act, void* stream);

/* Same operation on the 5th-generation tensor cores (tcgen05.mma, fp32 accumulation in TMEM): W_packed from
 * pack.pack_tc_weight (k-step slabs streamed with cp.async.bulk); X is converted while it is staged.
 *   nsplit = 1: bf16 operands (the "bf16 GEMM mode");
 *   nsplit = 2: bf16 (hi, lo) operand pairs, all four products -> fp32-grade results ("bf16x3", the parity mode;
 *               W_packed from pack_tc_weight(w, split=True)).
 * X rows must be 16-byte aligned. */
int kpd_tc_linear(const float* X, int32_t ldx, const void* W_packed, const float* bias, const float* R,
                  int32_t ldr, float* Y, int32_t ldy, int32_t M, int32_t K, int32_t N, int32_t act,
                  int32_t nsplit, void* stream);

/* ------------------------------------------------------------------------------------------
 * (b)+(d) EGNN denoiser.  Replaces LigRecDynamics.forward (models/dynamics.py:342-385),
 * LigRecEGNN.forward (:266-294) and LigRecConv.forward/message (:89-217).
 * The model is an opaque handle holding packed device weights (see kpd_egnn_create).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t atom_nf, rec_nf;   /* ligand / keypoint input feature widths                        */
    int32_t hidden_nf;         /* H = hidden_nf + 1 is the conv width                           */
    int32_t n_layers;
    int32_t use_tanh;          /* models/dynamics.py:117-118                                    */
    int32_t update_kp_feat;    /* 4 edge types + kp updates when 1                              */
    int32_t norm;              /* LayerNorm(H) after the node MLP                               */
    int32_t has_rec_encoder;   /* 0 when rec_nf == hidden_nf (nn.Identity, :333-334)            */
    float   coords_range;      /* 10                                                            */
    float   message_norm;      /* constant z, or 0 -> mean in-degree + 1 (:281-285)             */
    int32_t z_effective;       /* 0 = as executed by the reference (division is a no-op, see
                                  DESIGN.md N11); 1 = divide h_neigh/x_neigh by z              */
} kpd_egnn_config;

typedef struct kpd_egnn_model kpd_egnn_model;

/* Packed-weight blob layout is produced by the Python host (keypoint_diffusion_b200/pack.py)
 * from the reference state_dict; `blob` is a device pointer that must outlive the model, and
 * `offsets` is a HOST array of float offsets in the order kpd_egnn_create reads them (csrc/egnn.cu; written by
 * keypoint_diffusion_b200/pack.py: pack_egnn). */
int kpd_egnn_create(const kpd_egnn_config* cfg, const float* blob, const int64_t* offsets,
                    int32_t n_offsets, kpd_egnn_model** out);
void kpd_egnn_destroy(kpd_egnn_model* m);
/* Tensor-core modes of the EGNN: the per-node first-layer products and the node MLPs run through
 * kpd_tc_linear(nsplit = 2), the edge stage through the warp-specialised kernel of csrc/egnn_ws.inl.
 *   nsplit = 2: "bf16x3", split (hi, lo) bf16 operands, all four products, fp32 accumulation in TMEM -- inside the
 *               1e-4 parity bar -> mode 2;
 *   nsplit = 1: "bf16", plain bf16 operands in the edge kernel (one M = 64 MMA per k-step, one-MUFU activations;
 *               within 3e-2 of the output scale) -> mode 1, which needs the nsplit = 2 pack as well (node GEMMs).
 * tc_blob / byte_offsets from pack.pack_egnn_tc(split = nsplit == 2); both packs stay attached side by side.
 * mode: 0 = fp32 SIMT (default), 1 = bf16, 2 = bf16x3. */
int kpd_egnn_attach_tc(kpd_egnn_model* m, const void* tc_blob, const int64_t* byte_offsets, int32_t n,
                       int32_t nsplit);
int kpd_egnn_set_mode(kpd_egnn_model* m, int32_t mode);
int kpd_egnn_dims(const kpd_egnn_model* m, int* rec_nf, int* hidden_nf);
int64_t kpd_egnn_workspace_bytes(const kpd_egnn_model* m, const kpd_batch* batch,
                                 int32_t cap_ll, int32_t cap_kl, int32_t cap_kk);

/* One denoiser evaluation.  t_ptr: device pointer to ONE float (all complexes share t inside
 * the sampling loop, ligand_diffuser.py:405-408) or, if t_per_complex != 0, to [B] floats.
 * kp_feat_enc: optional precomputed encoder output for the keypoints [n_kp, hidden_nf] (the
 * encoder does not depend on t, so the sampler hoists it out of the loop); NULL = compute.
 * Graphs must have been built by kpd_build_graph for the same x. Outputs eps_h [n_lig, atom_nf],
 * eps_x [n_lig, 3]. */
int kpd_egnn_forward(const kpd_egnn_model* m, const kpd_batch* batch,
                     const float* h_lig, const float* x_lig, const float* h_kp, const float* x_kp,
                     const float* kp_feat_enc, const float* t_ptr, int32_t t_per_complex,
                     const kpd_csr* ll, const kpd_csr* kl, const kpd_csr* lk, const kpd_csr* kk,
                     float* eps_h, float* eps_x, void* workspace, void* stream);

/* keypoint encoder only (models/dynamics.py:356); out [n_kp, hidden_nf] */
int kpd_egnn_encode_kp(const kpd_egnn_model* m, const float* h_kp, int32_t n_kp, float* out,
                       void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * (c) GVP denoiser.  Replaces LigRecDynamicsGVP.forward (models/dynamics_gvp.py:149-199),
 * LigRecGVP.forward / NoisePredictionBlock (:38-101), GVPMultiEdgeConv.forward/message
 * (models/gvp.py:459-550), GVP.forward (:89-116), GVPLayerNorm (:152-166), _rbf (:26-41).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t n_lig_scalars, n_kp_scalars;
    int32_t vector_size;       /* V (<=16)                                                      */
    int32_t n_convs;
    int32_t n_hidden_scalars;  /* S (<=256, multiple of 4)                                      */
    int32_t n_message_gvps, n_update_gvps, n_noise_gvps;
    int32_t update_kp;
    int32_t norm_mode;         /* 0: divide by message_norm; 1: 'mean' per edge type;
                                  2: message_norm == 0 -> mean in-degree + 1 per complex       */
    float   message_norm;
    float   rbf_dmax;          /* 15 */
    int32_t rbf_dim;           /* 16 */
} kpd_gvp_config;

typedef struct kpd_gvp_model kpd_gvp_model;

int kpd_gvp_create(const kpd_gvp_config* cfg, const float* blob, const int64_t* offsets,
                   int32_t n_offsets, kpd_gvp_model** out);
void kpd_gvp_destroy(kpd_gvp_model* m);
int kpd_gvp_dims(const kpd_gvp_model* m, int* n_kp_scalars, int* vector_size);
/* Tensor-core modes: the scalar Linear of every GVP and its gates run as tcgen05.mma with fp32 accumulation in
 * TMEM (csrc/gvp_ws.inl).  tc_blob holds, for every GVP in creation order, THREE entries (pack.pack_gvp_tc): the packed
 * to_feats_out weight (k-step slabs), the gates weight, and the image of its small fp32 weights (Wh, Wu, biases);
 * byte_offsets has three entries per GVP.
 *   nsplit = 1: bf16 operands                        -> mode 1, the "bf16 GEMM mode" the north star reports
 *               separately (outputs within ~2e-3 of fp32);
 *   nsplit = 2: split bf16 operands, x = hi + lo with hi = bf16(x), lo = bf16(x - hi) -> mode 2, "bf16x3": fp32-grade
 *               operands, meets the 1e-4 parity bar on the tensor cores.  The edge kernel keeps hi and lo PLANES of a
 *               128-row tile and issues THREE MMAs per k-step (hi*hi + lo*hi + hi*lo); the node / head kernels stack the
 *               hi and lo rows of 64 tile rows into one 128-row operand and issue TWO (x W_hi, x W_lo: all four
 *               products).  When the edge tile of hi / lo planes does not fit in 227 KB of shared memory, the
 *               edge kernel uses the stacked layout too; of the accepted configurations only n_hidden_scalars = 256,
 *               vector_size = 16, rbf_dim = 32 (a 305-column first message GVP input) is that wide.
 * mode: 0 = fp32 SIMT (reference arithmetic), 1 = bf16, 2 = bf16x3. */
int kpd_gvp_attach_tc(kpd_gvp_model* m, const void* tc_blob, const int64_t* byte_offsets, int32_t n,
                      int32_t nsplit);
int kpd_gvp_set_mode(kpd_gvp_model* m, int32_t mode);
int64_t kpd_gvp_workspace_bytes(const kpd_gvp_model* m, const kpd_batch* batch,
                                int32_t cap_ll, int32_t cap_kl, int32_t cap_kk);

/* Stream semantics: the call is ordered on `stream` like any kernel launch (everything it does starts after prior work
 * on `stream` and is complete before later work on `stream`), and it may be captured into a CUDA graph.  In the
 * tensor-core modes the convs are issued as a dependency graph over auxiliary streams owned by the model (forked from
 * and joined back to `stream` by events inside the call; KPD_GVP_SERIAL=1 at model creation keeps everything on
 * `stream`).  A graph captured from it should be instantiated with cudaGraphInstantiateFlagUseNodePriority (the
 * node kernels carry a launch priority).  One call at a time per model handle from the host's point of view (the
 * model owns the events); concurrent execution of several captured graphs of the same model is fine. */
int kpd_gvp_forward(const kpd_gvp_model* m, const kpd_batch* batch,
                    const float* h_lig, const float* x_lig, const float* h_kp, const float* x_kp,
                    const float* v_kp, const float* t_ptr, int32_t t_per_complex,
                    const kpd_csr* ll, const kpd_csr* kl, const kpd_csr* lk, const kpd_csr* kk,
                    float* eps_h, float* eps_x, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * (e) Reverse-diffusion step.  Replaces KeypointDiffusion.sample_p_zs_given_zt after the
 * denoiser call (models/ligand_diffuser.py:515-536) and remove_com (:185-203).
 *   coef: [T,4] rows (alpha_t|s, var_terms, sigma, t) precomputed on the host from
 *         gamma (ligand_diffuser.py:232-252, :505-527); step_ptr: device int32 = current s.
 *   noise_x/noise_h: injected N(0,1) draws for this step, or NULL -> in-kernel Philox4x32-10
 *         keyed by (seed, s, atom, channel).
 * Updates x_lig, h_lig, x_kp in place.
 * ------------------------------------------------------------------------------------------ */
int kpd_ddpm_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp,
                  const float* eps_x, const float* eps_h, int32_t atom_nf,
                  const float* coef, const int32_t* step_ptr,
                  const float* noise_x, const float* noise_h, uint64_t seed, void* stream);

/* ------------------------------------------------------------------------------------------
 * (e) multistep: one DPM-Solver++(2M) reverse step (an extension beyond the reference, DESIGN.md
 * section 6.5), what a multistep sampler's captured step runs.  Row s of coef is a DDIM eta = 0 row
 * (schedule.coefficient_rows(..., eta=0)), row s of ms_coef [rows,4] = (c, alpha_t, sigma_t, 0)
 * (schedule.multistep_rows over the same grid):
 *   z'  = z/alpha_t|s - var_terms*eps + sigma*noise          (kpd_ddpm_step, draws included)
 *   x^  = (z - sigma_t eps) / alpha_t                        positions and features
 *   z_s = z' + c (x^ - hist)  unless s == first_row;  hist = x^
 *   then the ligand COM is removed from ligand and keypoints, and from the positions of hist.
 * first_row: the row a run executes first; that step does not read hist (it may hold anything).
 * hist_x [n_lig,3] / hist_h [n_lig,atom_nf]: caller-owned history, updated in place.
 * ------------------------------------------------------------------------------------------ */
int kpd_ddpm_multistep_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp,
                            const float* eps_x, const float* eps_h, int32_t atom_nf,
                            const float* coef, const float* ms_coef, const int32_t* step_ptr,
                            int32_t first_row, float* hist_x, float* hist_h,
                            const float* noise_x, const float* noise_h, uint64_t seed, void* stream);

/* ------------------------------------------------------------------------------------------
 * (e') Fragment-conditioned reverse step (inpainting with RePaint-style resampling; an extension
 * beyond the reference, DESIGN.md section 6.1).  Pass u of step s (t = s+1):
 *   z_unk = x/alpha_t|s - var_terms*eps + sigma*noise             (what kpd_ddpm_step computes)
 *   z_kn  = alpha_s*(x_fix - init_kp_com + kp_com) + sigma_s*e    positions of the fixed atoms
 *           alpha_s*h_fix/lig_feat_norm_constant + sigma_s*e      their features
 *   dx    = mean over fixed atoms of (z_unk_x - z_kn_x), added to z_kn_x and the complex's keypoints
 *   x, h  = fixed ? z_kn : z_unk; then the ligand COM is removed from ligand and keypoints.
 * kp_com is the complex's keypoint mean before the step; init_kp_com [B,3] the keypoint mean of
 * the frame x_fix is given in.  A complex without a fixed atom gets exactly kpd_ddpm_step.
 *   coef2: [T,4] rows (alpha_s, sigma_s, alpha_t|s, sigma_t|s) (schedule.inpaint_table);
 *   fixed_mask: uint8 [n_lig] (nonzero = fixed) or NULL; x_fix [n_lig,3], h_fix [n_lig,atom_nf];
 *   noise: NULL -> Philox keyed by (seed, s, atom, channel, word) with word 3u (posterior) and
 *          3u+1 (known part); or injected [2][n_lig*(3+atom_nf)]: posterior then known-part draws,
 *          each x channels [n_lig,3] first, then features [n_lig,atom_nf].
 * Updates x_lig, h_lig, x_kp in place.
 * ------------------------------------------------------------------------------------------ */
int kpd_ddpm_inpaint_step(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp,
                          const float* eps_x, const float* eps_h, int32_t atom_nf,
                          const float* coef, const float* coef2, const int32_t* step_ptr, int32_t u,
                          const uint8_t* fixed_mask, const float* x_fix, const float* h_fix,
                          const float* init_kp_com, float lig_feat_norm_constant,
                          const float* noise, uint64_t seed, void* stream);
/* Re-noise between resampling passes: z_t = alpha_t|s*z_s + sigma_t|s*e for positions and features
 * (Philox word 3u+2, or injected noise [n_lig*(3+atom_nf)], x first), then the ligand COM is removed
 * from ligand and keypoints. */
int kpd_renoise(const kpd_batch* batch, float* x_lig, float* h_lig, float* x_kp, int32_t atom_nf,
                const float* coef2, const int32_t* step_ptr, int32_t u, const float* noise, uint64_t seed,
                void* stream);

/* ------------------------------------------------------------------------------------------
 * (e'') Start of a run from a given ligand (ligand optimisation by partial noising, SDEdit-style;
 * an extension beyond the reference, DESIGN.md section 6.2).  One CTA per complex:
 *   c_b  = mean of x_start over the complex's atoms; x_kp -= c_b
 *   z_x  = alpha*(x_start - c_b) + sigma*e_x,  z_h = alpha*h_start/lig_feat_norm_constant + sigma*e_h
 *   then the ligand COM is removed from ligand and keypoints.
 * alpha / sigma = alpha_t0 / sigma_t0 (schedule.start_coefficients).  noise: NULL -> the Philox draw of
 * kpd_randn_init (seed, step = -1, atom, channel), or injected [n_lig*(3+atom_nf)], x channels first.
 * Writes x_lig [n_lig,3], h_lig [n_lig,atom_nf]; updates x_kp in place.
 * ------------------------------------------------------------------------------------------ */
int kpd_partial_noise(const kpd_batch* batch, const float* x_start, const float* h_start, float* x_lig,
                      float* h_lig, float* x_kp, int32_t atom_nf, float alpha, float sigma,
                      float lig_feat_norm_constant, const float* noise, uint64_t seed, void* stream);

/* remove_com (ligand_diffuser.py:185-203): which = 0 ligand COM, 1 keypoint COM; shifts both
 * node types.  If com_out != NULL the [B,3] means are also written there. */
int kpd_remove_com(const kpd_batch* batch, float* x_lig, float* x_kp, int32_t which,
                   float* com_out, void* stream);
/* x[node] += sign * v[batch[node]]  (frame shifts at ligand_diffuser.py:363, :443-444) */
int kpd_shift_by_complex(float* x, const int32_t* node_batch, int32_t n, const float* v, float sign,
                         void* stream);
/* standard-normal fill with the same Philox stream as kpd_ddpm_step uses for step = -1
 * (initial x_0 / h_0, ligand_diffuser.py:366-367) */
int kpd_randn_init(float* x_lig, float* h_lig, int32_t n_lig, int32_t atom_nf, uint64_t seed,
                   void* stream);

/* ------------------------------------------------------------------------------------------
 * The whole loop.  Replaces the body of KeypointDiffusion.sample_from_encoded_receptors
 * (models/ligand_diffuser.py:342-447, visualize=False): frame setup, T reverse steps (graph
 * build + denoiser + posterior step each), frame restore.  The per-step kernel sequence is
 * captured once into a CUDA graph of `steps_per_graph` steps and replayed.  With a start ligand
 * (kpd_sampler_set_start) the frame setup is kpd_partial_noise and the loop runs t0 steps from
 * step t0 - 1 down, through the same captured graphs.
 * ------------------------------------------------------------------------------------------ */
typedef struct kpd_sampler kpd_sampler;

typedef struct {
    int32_t arch;              /* 0 = egnn, 1 = gvp                                             */
    int32_t T;                 /* n_timesteps                                                   */
    int32_t atom_nf;
    int32_t steps_per_graph;   /* reverse steps captured per CUDA graph (>=1; T = whole loop)   */
    int32_t use_cuda_graph;    /* 0 = plain stream launches (debug / ncu)                       */
    float   lig_feat_norm_constant;
} kpd_sampler_config;

/* model: kpd_egnn_model* or kpd_gvp_model*.  kk is the static keypoint graph.  All buffers
 * (state, workspace) are caller-owned; the sampler only keeps pointers.  coef (schedule.coefficient_table)
 * is the default schedule of kpd_sampler_set_schedule. */
int kpd_sampler_create(const kpd_sampler_config* cfg, const void* model, const kpd_batch* batch,
                       const kpd_graph_params* gp, const kpd_csr* kk, int32_t has_lk,
                       const float* coef /*[T,4] device*/, int32_t cap_ll, int32_t cap_kl,
                       void* workspace, int64_t workspace_bytes, kpd_sampler** out);
int64_t kpd_sampler_workspace_bytes(const kpd_sampler_config* cfg, const void* model,
                                    const kpd_batch* batch, int32_t cap_ll, int32_t cap_kl,
                                    int32_t cap_kk);
void kpd_sampler_destroy(kpd_sampler* s);

/* Runs the loop.  x_kp/h_kp/v_kp: encoded keypoints (x_kp is modified in place and restored
 * to the input frame); init_lig_pos [B,3] (not read in a run from a start ligand, but still
 * required); x_lig/h_lig: outputs [n_lig,3]/[n_lig,atom_nf].
 * noise: NULL (Philox, `seed`) or device fp32 [(t0+1), n_lig, 3+atom_nf] with slot 0 = initial
 * draw and slot 1+k = the k-th executed step (s = t0-1-k), x channels first; t0 = T, or the
 * start step of kpd_sampler_set_start.  An inpainting sampler takes 1 + t0*(3r-1) slots.
 * n_steps: reverse steps to run, at most t0 (t0 for a full sample; fewer only for testing).
 * Graph replays cover floor(n_steps / steps_per_graph) * steps_per_graph steps; the rest run
 * as stream launches. */
int kpd_sampler_run(kpd_sampler* s, float* x_kp, const float* h_kp, const float* v_kp,
                    const float* init_lig_pos, float* x_lig, float* h_lig, const float* noise,
                    uint64_t seed, int32_t n_steps, void* stream);
/* mean edges per reverse step of the last run: out[4] = {E_ll, E_kl (= E_lk), E_kk, steps}; syncs */
int kpd_sampler_edge_stats(kpd_sampler* s, double* out);
/* kernels launched per reverse step by the captured sequence (for bench.py's gpu_launches) */
int32_t kpd_sampler_launches_per_step(const kpd_sampler* s);
/* Offset added to the ligand-atom index of the noise counter (seed, step, atom, channel): lets a caller sample one batch
 * as several sub-batches (own samplers, own streams) and draw exactly the noise of the undivided batch. */
int kpd_sampler_set_atom_offset(kpd_sampler* s, int32_t first_atom);
/* Turns a freshly created sampler (not yet run) into an inpainting sampler: every reverse step runs
 * `resamplings` passes of graph build + denoiser + kpd_ddpm_inpaint_step, with kpd_renoise between
 * passes; launches_per_step counts all of them.  coef2: [T,4] device table (schedule.inpaint_table),
 * must outlive the sampler.  Allocates a few bytes of device memory (synchronous).  Pick
 * steps_per_graph ~ (plain value) / resamplings so that a captured graph stays as large as a plain one.
 * With injected noise, kpd_sampler_run takes [1 + T*(3*resamplings - 1), n_lig, 3+atom_nf]: slot 0 =
 * initial draw, then per executed step and pass u the posterior, known-part and (u < resamplings-1)
 * re-noise draws. */
int kpd_sampler_enable_inpainting(kpd_sampler* s, int32_t resamplings, const float* coef2);
/* The fragment of the next runs of an inpainting sampler: fixed_mask uint8 [n_lig] (NULL = no fixed
 * atom), x_fix [n_lig,3] in the frame of the x_kp passed to kpd_sampler_run, h_fix [n_lig,atom_nf] in
 * the returned feature space.  Only pointers are kept; each run uploads them to device memory, so a
 * captured sampler follows new buffers without capturing again. */
int kpd_sampler_set_fragment(kpd_sampler* s, const uint8_t* fixed_mask, const float* x_fix, const float* h_fix);
/* The start of the next runs (ligand optimisation by partial noising, DESIGN.md section 6.2):
 * x_start [n_lig,3] in the frame of the x_kp passed to kpd_sampler_run, h_start [n_lig,atom_nf] in
 * the returned feature space, noised to step start_step (in [0, T]) with alpha / sigma =
 * alpha_t0 / sigma_t0 (HOST floats, schedule.start_coefficients) by kpd_partial_noise; the runs
 * then execute reverse steps start_step-1 .. 0.  x_start = NULL restores the plain start from
 * pure noise at step T.  Works for plain and inpainting samplers.  Only pointers are kept and each
 * run reads them, so a captured sampler follows new buffers and any start_step without capturing
 * again. */
int kpd_sampler_set_start(kpd_sampler* s, int32_t start_step, const float* x_start, const float* h_start,
                          float alpha, float sigma);
/* The coefficient rows of the next runs (fewer-step sampling, DESIGN.md section 6.3): coef [n_rows,4] device rows
 * (schedule.coefficient_rows over a step grid; row k is the reverse step tau_{k+1} -> tau_k) and, for an inpainting
 * sampler (required there), coef2 [n_rows,4] (schedule.inpaint_rows over the same grid); 1 <= n_rows <= T.  A run
 * then starts at row n_rows - 1, or at the start_step of kpd_sampler_set_start, which counts rows of this schedule
 * and must be <= n_rows (checked by kpd_sampler_run); injected noise has the slots of a run of that many steps, and
 * the Philox draws of row k are keyed by k.  coef = NULL restores the tables given at create time (T rows).  Only
 * pointers are kept: every run copies the active rows into the sampler's own table (cudaMemcpyAsync on its stream),
 * so a captured sampler serves any schedule without capturing again; the buffers must stay valid while runs use
 * them. */
int kpd_sampler_set_schedule(kpd_sampler* s, int32_t n_rows, const float* coef, const float* coef2);
/* Turns a freshly created sampler (not yet run) into a recording one (trajectories, DESIGN.md section 6.4): every
 * captured step gets one more launch, record_frame_kernel, after its first denoiser pass; launches_per_step counts it.
 * Allocates a few bytes of device memory (synchronous).  A sampler that never calls this captures what it did before. */
int kpd_sampler_enable_recording(kpd_sampler* s);
/* The frames of the next runs of a recording sampler.  A run of n_steps executed steps i = 0 .. n_steps-1 with stride
 * every >= 1 writes m = ceil(n_steps / every) frames, frame j = the state just before step i = j * every (after its
 * prologue), and copies the run's outputs into frame m:
 *   x_frames [m+1, n_lig, 3], h_frames [m+1, n_lig, atom_nf]: positions (x - kp mean) + initial kp mean, features
 *     h * lig_feat_norm_constant -- the frame and feature space the outputs are returned in;
 *   x_pred [m, n_lig, 3], h_pred [m, n_lig, atom_nf]: the clean-ligand estimate (z - sigma_t eps) / alpha_t of frame j
 *     from that step's first denoiser pass, in the same frame (unused, may be NULL, when n_frames == 1);
 *   pred_coef [n_pred_rows, 2] device: (alpha_t, sigma_t) of the level each row of the active schedule starts from
 *     (schedule.prediction_rows over its grid).
 * kpd_sampler_run checks n_frames == ceil(n_steps / every) + 1 and n_pred_rows == the active schedule's rows.
 * x_frames = NULL records nothing.  Only pointers are kept and each run uploads them, so a captured sampler follows new
 * buffers and strides without capturing again. */
int kpd_sampler_set_recording(kpd_sampler* s, int32_t every, int32_t n_frames, float* x_frames, float* h_frames,
                              float* x_pred, float* h_pred, int32_t n_pred_rows, const float* pred_coef);

/* Turns a freshly created sampler (not yet run, not inpainting) into a multistep one (DPM-Solver++(2M), DESIGN.md
 * section 6.5): its captured step launches the multistep instantiation of the step kernel instead of the plain one, so
 * launches_per_step does not change.  Allocates a few bytes of device memory (synchronous).  A sampler that never calls
 * this captures what it did before. */
int kpd_sampler_enable_multistep(kpd_sampler* s);
/* The multistep rows and history of the next runs: ms_coef [n_rows,4] device rows (schedule.multistep_rows over the
 * grid of the active schedule, whose coef rows must be DDIM eta = 0 rows), hist_x [n_lig,3] and hist_h [n_lig,atom_nf]
 * caller-owned scratch (need no initialisation: the first executed row writes them before any read).
 * kpd_sampler_run checks n_rows == the active schedule's rows.  Only pointers are kept and each run uploads them, so a
 * captured sampler follows new rows and buffers without capturing again. */
int kpd_sampler_set_multistep(kpd_sampler* s, int32_t n_rows, const float* ms_coef, float* hist_x, float* hist_h);

/* Output decode, the step right behind the path (reference test.py:199-203: torch.argmax(lig_feat, dim=1) on the
 * host, then dataset.lig_atom_idx_to_element): atom_type[i] = argmax_c h_lig[i, c], lowest index on ties. */
int kpd_decode_atom_types(const float* h_lig, int32_t n_lig, int32_t atom_nf, int32_t* atom_type, void* stream);

/* ------------------------------------------------------------------------------------------
 * Diagnostics (tools/tc_phase_times.py, tools/eg_phase_times.py, tools/ws_trace.py): in-kernel phase timers of the
 * warp-specialised kernels, in SM cycles summed over CTAs; each call synchronises the device, copies the counters
 * out and resets them.  kpd_debug_ws_trace returns the (tag, warp, clock) event list of one CTA and is empty unless
 * the library was built with `make TRACE=1`.
 * ------------------------------------------------------------------------------------------ */
int kpd_debug_ws_times(unsigned long long* out64);
int kpd_debug_eg_times(unsigned long long* out16);
int kpd_debug_ws_trace(unsigned long long* out, int32_t cap, int32_t* count);
/* Launch timeline of the GVP convs (library built with -DKPD_TIMELINE, else returns 0 slots): out = [256][3] =
 * (first CTA start ns, last CTA end ns, working CTAs) per slot 8 * conv + edge type (or 4 + node type). */
int kpd_debug_timeline(unsigned long long* out, int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* KPDIFF_B200_H */
