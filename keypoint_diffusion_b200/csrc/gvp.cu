// (c) GVP denoiser on flat tensors + dst-sorted CSR.
//
// Replaces LigRecDynamicsGVP.forward (models/dynamics_gvp.py:149-199), LigRecGVP.forward and
// NoisePredictionBlock (:38-101), GVPMultiEdgeConv.forward/message (models/gvp.py:459-550),
// GVP.forward (:89-116), GVPLayerNorm (:152-166), _rbf (:26-41), _norm_no_nan (:12-19).
//
// One device routine, gvp_tile(), applies a GVP to a tile of 64 rows held in shared memory
// (scalars [64 x (fin+h)], vectors [64 x v x 3]); it is the body of
//   gvp_edge_kernel  -- gather (s_src, v_src, unit x_diff, rbf(d)) per edge, chain the message
//                       GVPs in shared memory, deterministic segmented reduction by destination
//                       (no per-edge message ever reaches HBM);
//   gvp_node_kernel  -- recombine messages, /norm, residual, GVPLayerNorm, update GVPs,
//                       residual, GVPLayerNorm (gvp.py:501-536);
//   gvp_head_kernel  -- NoisePredictionBlock: noise GVPs + Linear(64 -> atom_nf).
// The scalar contraction [64 x (fin+h)] @ WfT is the shared tile GEMM of common.cuh.
//
// Offsets array (float offsets into the packed blob), in this order:
//   globals [8]:  lig_enc.WT, b, ln.w, ln.b, kp_enc.WT, b, ln.w, ln.b
//   per conv l:   for et in etypes(l):  n_message_gvps x (Wh, Wu, WfT, bf, WgT, bg)
//                 for nt in dst(l):     n_update_gvps  x (Wh, Wu, WfT, bf, WgT, bg),
//                                       msg_ln.w, msg_ln.b, upd_ln.w, upd_ln.b
//   head:         n_noise_gvps x (Wh, Wu, WfT, bf, WgT, bg), WoT, bo
//   etypes(l) = (ll, kl, lk, kk) if update_kp and l != n_convs-1 else (ll, kl)
#include "common.cuh"
#include "tc.cuh"
#include "ws_common.cuh"
#include <string.h>
#include <vector>

namespace kpd {

constexpr int VMAX = 17;   // vector channels held per row (vector_size + 1 for x_diff)
constexpr int MAXG = 4;    // GVPs chained per kernel

struct GvpW {
    const float* Wh;    // [vin][hd]
    const float* Wu;    // [hd][vout]
    const float* WfT;   // [fin+hd][ldf]
    const float* bf;    // [ldf]
    const float* WgT;   // [fout][vout]
    const float* bg;    // [vout]
    const uint4* WfP;   // bf16 mode: to_feats_out weight as tcgen05 k-step slabs (pack_tc_weight)
    const uint4* WgP;   // bf16 mode: gates weight, rows padded to 16
    const uint4* WfP2;  // bf16x3 mode: the same two weights as interleaved (hi, lo) k-step slabs
    const uint4* WgP2;  //   gates weight as mma.sync B fragments (pack.pack_gates_frag) ...
    const uint4* WgP2c; //   ... followed by the same weight as (hi, lo) tcgen05 k-step slabs (the KS edge kernel)
    const float* wsmP;  // tensor-core modes: shared-memory image of Wh, Wu, bf, bg (pack.pack_gvp_small)
    const float* wsmP2;
    int vin, vout, hd, fin, fout, ldf, sigmoid_gate;
    int xfirst;         // input vector channel 0 is the edge's unit x_diff (message GVP 0)
};

// GVP.forward (models/gvp.py:89-116) on a shared-memory tile of TE rows.
//   S: [TE][lds], input scalars in cols [0,fin); V: [TE][VMAX][3] input vectors (vin used).
//   On return S cols [0,fout) hold feats_out and V rows [0,vout) hold the gated vectors.
template <int RM>
__device__ void gvp_tile(const GvpW& g, float* S, int lds, float* V, float* Vh, float* Bs) {
    constexpr int TR = 16 * RM;   // rows of this tile
    const int tid = threadIdx.x;
    // Vh = einsum('b v c, v h -> b h c'); sh = sqrt(clamp(sum_c Vh^2, 1e-8))  (:96, :99)
    for (int idx = tid; idx < TR * g.hd; idx += NT) {
        const int r = idx / g.hd, hh = idx - r * g.hd;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        const float* v = V + r * (VMAX * 3);
        for (int k = 0; k < g.vin; ++k) {
            const float w = g.Wh[k * g.hd + hh];
            a0 = fmaf(v[3 * k], w, a0); a1 = fmaf(v[3 * k + 1], w, a1); a2 = fmaf(v[3 * k + 2], w, a2);
        }
        float* o = Vh + r * (VMAX * 3) + 3 * hh;
        o[0] = a0; o[1] = a1; o[2] = a2;
        S[r * lds + g.fin + hh] = sqrtf(fmaxf(a0 * a0 + a1 * a1 + a2 * a2, 1e-8f));
    }
    __syncthreads();
    // Vu = einsum('b h c, h u -> b u c')  (:97) -> V (the input vectors are dead now)
    for (int idx = tid; idx < TR * g.vout; idx += NT) {
        const int r = idx / g.vout, u = idx - r * g.vout;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        const float* vh = Vh + r * (VMAX * 3);
        for (int k = 0; k < g.hd; ++k) {
            const float w = g.Wu[k * g.vout + u];
            a0 = fmaf(vh[3 * k], w, a0); a1 = fmaf(vh[3 * k + 1], w, a1); a2 = fmaf(vh[3 * k + 2], w, a2);
        }
        float* o = V + r * (VMAX * 3) + 3 * u;
        o[0] = a0; o[1] = a1; o[2] = a2;
    }
    // feats_out = SiLU(Linear(cat(feats, sh)))  (:101-103)
    float acc[RM][16];
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[i][j] = 0.f;
    const int nmain = (g.fout + 3) & ~3;
    tile_gemm<RM>(S, lds, g.WfT, g.ldf, g.fin + g.hd, nmain, Bs, acc);
    {
        const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
        for (int i = 0; i < RM; ++i) {
            const int r = ty * (RM) + i;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int col = 4 * tx + 64 * j;
                if (col < nmain) {
                    float4 o;
                    o.x = silu_f(acc[i][4 * j + 0] + g.bf[col + 0]);
                    o.y = silu_f(acc[i][4 * j + 1] + g.bf[col + 1]);
                    o.z = silu_f(acc[i][4 * j + 2] + g.bf[col + 2]);
                    o.w = silu_f(acc[i][4 * j + 3] + g.bf[col + 3]);
                    *reinterpret_cast<float4*>(S + r * lds + col) = o;
                }
            }
        }
    }
    __syncthreads();
    // gating = Linear(feats_out); vectors_out = act(gating) * Vu  (:105-111)
    for (int idx = tid; idx < TR * g.vout; idx += NT) {
        const int r = idx / g.vout, u = idx - r * g.vout;
        float a = g.bg[u];
        const float* s = S + r * lds;
        for (int k = 0; k < g.fout; ++k) a = fmaf(s[k], g.WgT[k * g.vout + u], a);
        if (g.sigmoid_gate) a = sigmoid_f(a);
        float* o = V + r * (VMAX * 3) + 3 * u;
        o[0] *= a; o[1] *= a; o[2] *= a;
    }
    __syncthreads();
}

// scalar LayerNorm over S cols [0,Sdim) (one warp per row) + GVP vector norm (gvp.py:159-166)
template <int RM>
__device__ void gvp_layernorm_tile(float* S, int lds, int Sdim, float* V, int nv, const float* w, const float* b) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int rr = 0; rr < 2 * RM; ++rr) {
        const int r = warp * (2 * RM) + rr;
        float* x = S + r * lds;
        float s = 0.f;
        for (int c = lane; c < Sdim; c += 32) s += x[c];
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = s / (float)Sdim;
        float v = 0.f;
        for (int c = lane; c < Sdim; c += 32) { const float d = x[c] - mean; v += d * d; }
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        const float rstd = 1.0f / sqrtf(v / (float)Sdim + 1e-5f);
        for (int c = lane; c < Sdim; c += 32) x[c] = (x[c] - mean) * rstd * w[c] + b[c];
        // vn = sqrt(mean_v clamp(|v|^2, 1e-8) + eps) + eps
        float* vv = V + r * (VMAX * 3);
        float q = 0.f;
        for (int k = lane; k < nv; k += 32)
            q += fmaxf(vv[3 * k] * vv[3 * k] + vv[3 * k + 1] * vv[3 * k + 1] + vv[3 * k + 2] * vv[3 * k + 2], 1e-8f);
#pragma unroll
        for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float vn = sqrtf(q / (float)nv + 1e-5f) + 1e-5f;
        for (int k = lane; k < 3 * nv; k += 32) vv[k] = vv[k] / vn;
    }
    __syncthreads();
}

struct GvpSmem {
    float *S, *Bs, *V, *Vh;
    int* src_s; int* dst_s;
};

template <int RM>
__device__ __forceinline__ GvpSmem gvp_carve_smem(float* smem, int lds) {
    constexpr int TR = 16 * RM;
    GvpSmem m;
    m.S = smem;
    m.Bs = m.S + TR * lds;
    m.V = m.Bs + BS_FLOATS;
    m.Vh = m.V + TR * VMAX * 3;
    m.src_s = reinterpret_cast<int*>(m.Vh + TR * VMAX * 3);
    m.dst_s = m.src_s + TR;
    return m;
}

static size_t gvp_smem_bytes(int lds, int rows) {
    return sizeof(float) * ((size_t)rows * lds + BS_FLOATS + 2 * rows * VMAX * 3) + sizeof(int) * 2 * rows;
}

constexpr int RM_EDGE = TE / 16;   // 64-edge tiles (seg_gather's tile size)
constexpr int RM_NODE = 2;         // 32-node tiles: node counts are small, more CTAs fill the GPU
constexpr int TN = 16 * RM_NODE;

struct GvpEtypeArgs {
    const int* rowptr; const int* src; const int* dst; int n_dst; int cap;
    const float* s_src; const float* v_src; const float* xs; const float* xd;
    const __nv_bfloat16* s_hi; const __nv_bfloat16* s_lo;   // tensor-core modes: bf16 planes of s_src
    GvpW msg[MAXG];
    float* sm; float* vm; float* part;
};

// launch timeline (only with -DKPD_TIMELINE): per slot the start of CTA 0 of the LAST launch, the latest CTA end
// (globaltimer, ns) and the number of working CTAs summed over launches; slot = 8 * conv + edge type (or 4 + node type); see kpd_debug_timeline
#ifdef KPD_TIMELINE
__device__ unsigned long long g_tl[3 * 256];
__device__ __forceinline__ unsigned long long tl_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define TL_BEGIN(slot) do { if (threadIdx.x == 0 && (slot) >= 0) { if (blockIdx.x == 0) g_tl[3 * (slot)] = tl_now(); atomicAdd(&g_tl[3 * (slot) + 2], 1ull); } } while (0)
#define TL_END(slot) do { if (threadIdx.x == 0 && (slot) >= 0) atomicMax(&g_tl[3 * (slot) + 1], tl_now()); } while (0)
#else
#define TL_BEGIN(slot) do { } while (0)
#define TL_END(slot) do { } while (0)
#endif

struct GvpEdgeLaunch {
    GvpEtypeArgs e[4];
    int tl_slot;
    int Sdim, Vdim, n_msg, lds, pw, rbf_dim, kch;
    float rbf_step, rbf_sigma;
};

__global__ void __launch_bounds__(NT, 1) gvp_edge_kernel(const GvpEdgeLaunch L) {
    const GvpEtypeArgs& a = L.e[blockIdx.y];
    const int E = a.rowptr[a.n_dst];
    const int tile_begin = blockIdx.x * TE;
    if (tile_begin >= E) return;
    const int n = min(TE, E - tile_begin);
    extern __shared__ __align__(16) float smem[];
    GvpSmem m = gvp_carve_smem<RM_EDGE>(smem, L.lds);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Sd = L.Sdim, Vd = L.Vdim, lds = L.lds;

    zero_stage(m.Bs);
    if (tid < TE) {
        const int e = tile_begin + min(tid, n - 1);
        const int s = a.src[e], d = a.dst[e];
        m.src_s[tid] = s;
        m.dst_s[tid] = d;
        // gvp.py:474-480: x_diff, dij = sqrt(clamp(|x_diff|^2,1e-8)) + 1e-8, unit vector, rbf(dij)
        const float dx = a.xs[3 * s] - a.xd[3 * d], dy = a.xs[3 * s + 1] - a.xd[3 * d + 1],
                    dz = a.xs[3 * s + 2] - a.xd[3 * d + 2];
        const float dij = sqrtf(fmaxf(dx * dx + dy * dy + dz * dz, 1e-8f)) + 1e-8f;
        float* v0 = m.V + tid * (VMAX * 3);
        v0[0] = dx / dij; v0[1] = dy / dij; v0[2] = dz / dij;
        float* srow = m.S + tid * lds + Sd;
        for (int k = 0; k < L.rbf_dim; ++k) {
            const float z = (dij - (float)k * L.rbf_step) / L.rbf_sigma;
            srow[k] = expf(-(z * z));
        }
    }
    __syncthreads();
    // gather s_src (float4 rows) and v_src
    for (int rr = 0; rr < TE / 8; ++rr) {
        const int r = warp * (TE / 8) + rr;
        const float* sp = a.s_src + (size_t)m.src_s[r] * Sd;
        for (int f = lane; f < (Sd >> 2); f += 32)
            *reinterpret_cast<float4*>(m.S + r * lds + 4 * f) = *reinterpret_cast<const float4*>(sp + 4 * f);
        const float* vp = a.v_src + (size_t)m.src_s[r] * (Vd * 3);
        for (int k = lane; k < Vd * 3; k += 32) m.V[r * (VMAX * 3) + 3 + k] = vp[k];
    }
    __syncthreads();
    for (int i = 0; i < L.n_msg; ++i) gvp_tile<RM_EDGE>(a.msg[i], m.S, lds, m.V, m.Vh, m.Bs);

    SegOut o;
    o.part0 = a.part + ((size_t)blockIdx.x * 2 + 0) * L.pw;
    o.part1 = a.part + ((size_t)blockIdx.x * 2 + 1) * L.pw;
    o.out = a.sm; o.ld_out = Sd;
    for (int col = tid; col < Sd; col += NT)
        seg_reduce_column(m.S, lds, col, n, m.dst_s, a.rowptr, tile_begin, o, col);
    if (tid < Vd * 3) {
        SegOut ov = o;
        ov.out = a.vm; ov.ld_out = Vd * 3;
        ov.part0 += Sd; ov.part1 += Sd;
        seg_reduce_column(m.V, VMAX * 3, tid, n, m.dst_s, a.rowptr, tile_begin, ov, tid);
    }
}

struct GvpNodeArgs {
    int n, Sdim, Vdim, lds, pw, n_upd, n_et, kch, edge_tile;
    float* s; float* v;                        // node features (fp32 SIMT kernel: updated in place)
    __nv_bfloat16* s_hi; __nv_bfloat16* s_lo;  // tensor-core modes: bf16 planes of s (what the edge kernels gather)
    // tensor-core modes: the updated features go to a SECOND buffer set (== the inputs when the caller runs the layers
    // serially), so that edge kernels still reading the old features may overlap this kernel (kpd_gvp_forward)
    float* s_out; float* v_out; __nv_bfloat16* s_hi_out; __nv_bfloat16* s_lo_out;
    const int* rowptr[2]; const float* sm[2]; const float* vm[2]; const float* part[2];
    int norm_mode; float norm_const;           // 0 const, 1 per-etype mean, 2 mean in-degree + 1
    const int* node_batch; const int* ptr;
    GvpW upd[MAXG];
    const float *mln_w, *mln_b, *uln_w, *uln_b;
};

struct GvpNodeLaunch { GvpNodeArgs nt[2]; int tl_slot; };

__global__ void __launch_bounds__(NT, 1) gvp_node_kernel(const GvpNodeLaunch L) {
    const GvpNodeArgs& a = L.nt[blockIdx.y];
    extern __shared__ __align__(16) float smem[];
    GvpSmem m = gvp_carve_smem<RM_NODE>(smem, a.lds);
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * TN;
    if (n0 >= a.n) return;
    const int n = min(TN, a.n - n0);
    const int Sd = a.Sdim, Vd = a.Vdim, lds = a.lds, W = Sd + 3 * Vd;
    zero_stage(m.Bs);
    // features + aggregated messages / norm  (gvp.py:501-520)
    for (int idx = tid; idx < TN * W; idx += NT) {
        const int r = idx / W, c = idx - r * W;
        const int nd = n0 + min(r, n - 1);
        float msg = 0.f;
        for (int e = 0; e < a.n_et; ++e) {
            const int r0 = a.rowptr[e][nd], r1 = a.rowptr[e][nd + 1];
            float g = c < Sd ? seg_gather(a.sm[e], Sd, a.part[e], a.pw, r0, r1, nd, c, a.edge_tile)
                             : seg_gather(a.vm[e], 3 * Vd, a.part[e] + Sd, a.pw, r0, r1, nd, c - Sd, a.edge_tile);
            if (a.norm_mode == 1) g = g / (float)max(r1 - r0, 1);      // fn.mean per edge type
            msg += g;
        }
        float nv = a.norm_const;
        if (a.norm_mode == 1) nv = 1.0f;
        else if (a.norm_mode == 2) {
            const int b = a.node_batch[nd];
            const int p0 = a.ptr[b], p1 = a.ptr[b + 1];
            int tot = 0;
            for (int e = 0; e < a.n_et; ++e) tot += a.rowptr[e][p1] - a.rowptr[e][p0];
            nv = (float)tot / (float)(p1 - p0) + 1.0f;
        }
        msg = msg / nv;
        if (c < Sd) m.S[r * lds + c] = a.s[(size_t)nd * Sd + c] + msg;
        else m.V[r * (VMAX * 3) + (c - Sd)] = a.v[(size_t)nd * (3 * Vd) + (c - Sd)] + msg;
    }
    __syncthreads();
    gvp_layernorm_tile<RM_NODE>(m.S, lds, Sd, m.V, Vd, a.mln_w, a.mln_b);
    // stash the normalised features as the residual (rows of this CTA only)
    for (int idx = tid; idx < n * W; idx += NT) {
        const int r = idx / W, c = idx - r * W;
        if (c < Sd) a.s[(size_t)(n0 + r) * Sd + c] = m.S[r * lds + c];
        else a.v[(size_t)(n0 + r) * (3 * Vd) + (c - Sd)] = m.V[r * (VMAX * 3) + (c - Sd)];
    }
    __syncthreads();
    for (int i = 0; i < a.n_upd; ++i) gvp_tile<RM_NODE>(a.upd[i], m.S, lds, m.V, m.Vh, m.Bs);
    for (int idx = tid; idx < TN * W; idx += NT) {
        const int r = idx / W, c = idx - r * W;
        const int nd = n0 + min(r, n - 1);
        if (c < Sd) m.S[r * lds + c] += a.s[(size_t)nd * Sd + c];
        else m.V[r * (VMAX * 3) + (c - Sd)] += a.v[(size_t)nd * (3 * Vd) + (c - Sd)];
    }
    __syncthreads();
    gvp_layernorm_tile<RM_NODE>(m.S, lds, Sd, m.V, Vd, a.uln_w, a.uln_b);
    for (int idx = tid; idx < n * W; idx += NT) {
        const int r = idx / W, c = idx - r * W;
        if (c < Sd) a.s[(size_t)(n0 + r) * Sd + c] = m.S[r * lds + c];
        else a.v[(size_t)(n0 + r) * (3 * Vd) + (c - Sd)] = m.V[r * (VMAX * 3) + (c - Sd)];
    }
}

struct GvpHeadArgs {
    int n, Sdim, Vdim, lds, n_gvps, F, Fp, hid_out, kch;
    const float* s; const float* v;
    const __nv_bfloat16* s_hi; const __nv_bfloat16* s_lo;
    GvpW g[MAXG];
    const float* WoT; const float* bo;
    float* eps_h; float* eps_x;
};

__global__ void __launch_bounds__(NT, 1) gvp_head_kernel(const GvpHeadArgs a) {
    extern __shared__ __align__(16) float smem[];
    GvpSmem m = gvp_carve_smem<RM_NODE>(smem, a.lds);
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * TN;
    const int n = min(TN, a.n - n0);
    const int Sd = a.Sdim, Vd = a.Vdim, lds = a.lds, W = Sd + 3 * Vd;
    zero_stage(m.Bs);
    for (int idx = tid; idx < TN * W; idx += NT) {
        const int r = idx / W, c = idx - r * W;
        const int nd = n0 + min(r, n - 1);
        if (c < Sd) m.S[r * lds + c] = a.s[(size_t)nd * Sd + c];
        else m.V[r * (VMAX * 3) + (c - Sd)] = a.v[(size_t)nd * (3 * Vd) + (c - Sd)];
    }
    __syncthreads();
    for (int i = 0; i < a.n_gvps; ++i) gvp_tile<RM_NODE>(a.g[i], m.S, lds, m.V, m.Vh, m.Bs);
    // to_scalar_output + vectors.squeeze(1)  (dynamics_gvp.py:42-43)
    for (int idx = tid; idx < n * (a.F + 3); idx += NT) {
        const int r = idx / (a.F + 3), c = idx - r * (a.F + 3);
        if (c < a.F) {
            float s = a.bo[c];
            for (int k = 0; k < a.hid_out; ++k) s = fmaf(m.S[r * lds + k], a.WoT[k * a.Fp + c], s);
            a.eps_h[(size_t)(n0 + r) * a.F + c] = s;
        } else {
            a.eps_x[(size_t)(n0 + r) * 3 + (c - a.F)] = m.V[r * (VMAX * 3) + (c - a.F)];
        }
    }
}

#include "gvp_ws.inl"

}  // namespace kpd

using namespace kpd;

// a kernel as kpd_gvp_forward launches it: `threads` per CTA, `rows` edges or nodes per CTA
template <typename Arg>
struct GvpKernel {
    void (*fn)(Arg);
    int threads;
    size_t smem;
    int rows;
};

// the kernels of one precision mode
struct GvpKernels {
    GvpKernel<GvpEdgeLaunch> edge;
    GvpKernel<GvpNodeLaunch> node[2];   // [full_node_tiles] (kpd_gvp_forward)
    GvpKernel<GvpHeadArgs> head[2];     // [full_node_tiles]
};

// the tensor-core kernels: edge tiles of configuration CE, node / head tiles of CN
template <class CE, class CN>
static GvpKernels gvp_ws_kernels(int kch) {
    const size_t smem_n = ws::smem_bytes<CN>(kch);
    return {{gvp_edge_ws_kernel<CE>, CE::NT, ws::smem_bytes<CE>(kch), CE::R},
            {{gvp_node_ws_kernel<CN, NODE_ROWS>, CN::NT, smem_n, NODE_ROWS},
             {gvp_node_ws_kernel<CN, NODE_ROWS_FULL>, CN::NT, smem_n, NODE_ROWS_FULL}},
            {{gvp_head_ws_kernel<CN, NODE_ROWS>, CN::NT, smem_n, NODE_ROWS},
             {gvp_head_ws_kernel<CN, NODE_ROWS_FULL>, CN::NT, smem_n, NODE_ROWS_FULL}}};
}

static cudaError_t gvp_set_smem(const GvpKernels& k) {
    cudaError_t e = cudaFuncSetAttribute(k.edge.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.edge.smem);
    for (int f = 0; f < 2 && e == cudaSuccess; ++f) {
        e = cudaFuncSetAttribute(k.node[f].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.node[f].smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k.head[f].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.head[f].smem);
    }
    return e;
}

// launch, optionally with the highest stream priority as a launch attribute
template <typename Arg>
static void launch_with_priority(const GvpKernel<Arg>& k, dim3 grid, cudaStream_t st, const Arg& arg,
                                 bool high_priority = false) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(k.threads);
    cfg.dynamicSmemBytes = k.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    int na = 0;
    if (high_priority) {        // explicit, so that a captured kernel node carries it whatever the stream's priority
        int pr_lo = 0, pr_hi = 0;
        cudaDeviceGetStreamPriorityRange(&pr_lo, &pr_hi);
        attr[na].id = cudaLaunchAttributePriority;
        attr[na].val.priority = pr_hi;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    cudaLaunchKernelEx(&cfg, k.fn, arg);
}

struct GvpLayerW {
    int n_et, n_dst;
    GvpW msg[4][MAXG];
    GvpW upd[2][MAXG];
    const float *mln_w[2], *mln_b[2], *uln_w[2], *uln_b[2];
};

struct kpd_gvp_model {
    kpd_gvp_config cfg;
    int S, Sp, V, F, Fp, C, lds, pw;
    const float* lig_enc[4]; const float* kp_enc[4];
    std::vector<GvpLayerW> layers;
    GvpW head[MAXG];
    const float* WoT; const float* bo;
    int kch;           // k-chunks of the bf16 tile (tensor-core mode)
    int mode;          // 0 = fp32 SIMT, 1 = bf16 tcgen05, 2 = bf16x3 tcgen05 (split operands, fp32-grade)
    GvpKernels k[3];   // [mode]: filled by kpd_gvp_create (0) and kpd_gvp_attach_tc (nsplit); edge.fn null until then
    std::vector<GvpW*> all_gvps;   // enumeration order of kpd_gvp_attach_tc
    // tensor-core modes: the layers run as a dependency graph over one stream per edge type (see kpd_gvp_forward);
    // created on first use
    mutable cudaStream_t aux[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // ll, lk, kk edges; lig, kp nodes
    mutable cudaEvent_t ev_edge[4] = {nullptr, nullptr, nullptr, nullptr}, ev_node[2] = {nullptr, nullptr};
    mutable bool dag_ready = false;
    bool serial = false;          // KPD_GVP_SERIAL=1: one stream, one edge launch and one node launch per conv
};

// node features and per-edge-type aggregates exist twice (conv parity): conv l reads set l % 2 and writes set
// (l + 1) % 2, so that the kernels of neighbouring convs may overlap (kpd_gvp_forward); the fp32 SIMT mode and the
// serial tensor-core path only use set 0
struct GvpWs {
    float *s[2][2], *v[2][2], *sm[2][4], *vm[2][4], *part[2][4], *tin, *tenc;
    __nv_bfloat16 *s_hi[2][2], *s_lo[2][2];
};

static int gvp_ntiles(int cap) { return cdiv(cap > 0 ? cap : 1, TE) + 1; }

static GvpWs gvp_carve(const kpd_gvp_model* m, const kpd_batch* b, const int caps[4], void* ws, int64_t* bytes) {
    GvpWs w;
    Carver c(ws);
    const int N[2] = {b->n_lig, b->n_kp};
    const int maxN = N[0] > N[1] ? N[0] : N[1];
    const int dstN[4] = {N[0], N[0], N[1], N[1]};
    for (int p = 0; p < 2; ++p) {
        for (int nt = 0; nt < 2; ++nt) {
            w.s[p][nt] = c.take<float>((int64_t)N[nt] * m->S);
            w.v[p][nt] = c.take<float>((int64_t)N[nt] * m->V * 3);
            w.s_hi[p][nt] = c.take<__nv_bfloat16>((int64_t)N[nt] * m->S);
            w.s_lo[p][nt] = c.take<__nv_bfloat16>((int64_t)N[nt] * m->S);
        }
        for (int e = 0; e < 4; ++e) {
            w.sm[p][e] = c.take<float>((int64_t)dstN[e] * m->S);
            w.vm[p][e] = c.take<float>((int64_t)dstN[e] * m->V * 3);
            w.part[p][e] = c.take<float>((int64_t)gvp_ntiles(caps[e]) * 2 * m->pw);
        }
    }
    const int win = (m->F > m->C ? m->F : m->C) + 1;
    w.tin = c.take<float>((int64_t)maxN * win);
    w.tenc = c.take<float>((int64_t)maxN * m->S);
    if (bytes) *bytes = c.bytes();
    return w;
}

extern "C" int kpd_gvp_create(const kpd_gvp_config* cfg, const float* blob, const int64_t* off, int32_t n_off,
                              kpd_gvp_model** out) {
    KPD_REQUIRE(cfg && blob && off && out, "kpd_gvp_create: null argument");
    KPD_REQUIRE((reinterpret_cast<uintptr_t>(blob) & 15) == 0, "kpd_gvp_create: blob must be 16-byte aligned");
    KPD_REQUIRE(cfg->vector_size >= 1 && cfg->vector_size + 1 <= VMAX, "kpd_gvp_create: vector_size %d unsupported (max %d)", cfg->vector_size, VMAX - 1);
    KPD_REQUIRE(cfg->n_hidden_scalars % 4 == 0 && cfg->n_hidden_scalars <= 256, "kpd_gvp_create: n_hidden_scalars must be a multiple of 4 and <= 256 (got %d)", cfg->n_hidden_scalars);
    KPD_REQUIRE(cfg->n_message_gvps >= 1 && cfg->n_message_gvps <= MAXG && cfg->n_update_gvps >= 1 && cfg->n_update_gvps <= MAXG &&
                cfg->n_noise_gvps >= 1 && cfg->n_noise_gvps <= MAXG, "kpd_gvp_create: at most %d GVPs per block", MAXG);
    KPD_REQUIRE(cfg->rbf_dim >= 2 && cfg->rbf_dim <= 32, "kpd_gvp_create: rbf_dim %d unsupported", cfg->rbf_dim);
    auto* m = new kpd_gvp_model();
    m->cfg = *cfg;
    { const char* e = getenv("KPD_GVP_SERIAL"); m->serial = e && e[0] == '1'; }
    m->S = cfg->n_hidden_scalars; m->Sp = m->S; m->V = cfg->vector_size;
    m->F = cfg->n_lig_scalars; m->Fp = (m->F + 3) & ~3; m->C = cfg->n_kp_scalars;
    {   // widest row any GVP of this model reads or writes: message GVP 0 reads S+rbf+V+1 columns,
        // the last noise GVP writes 64 (dynamics_gvp.py:12) even when S < 64
        int wmax = m->S + cfg->rbf_dim + m->V + 1;
        if (wmax < 64 + m->V) wmax = 64 + m->V;
        m->lds = tile_ld(wmax);
    }
    m->pw = ((m->S + 3 * m->V) + 3) & ~3;
    int i = 0;
    auto P = [&](void) -> const float* { int64_t o = off[i++]; return o < 0 ? nullptr : blob + o; };
    auto G = [&](int vin, int vout, int fin, int fout, int sig) {
        GvpW g;
        g.vin = vin; g.vout = vout; g.hd = vin > vout ? vin : vout; g.fin = fin; g.fout = fout;
        g.ldf = (fout + 3) & ~3; g.sigmoid_gate = sig;
        g.Wh = P(); g.Wu = P(); g.WfT = P(); g.bf = P(); g.WgT = P(); g.bg = P();
        g.WfP = nullptr; g.WgP = nullptr; g.WfP2 = nullptr; g.WgP2 = nullptr; g.WgP2c = nullptr; g.wsmP = nullptr; g.wsmP2 = nullptr;
        g.xfirst = vin > vout && sig ? 1 : 0;
        return g;
    };
    int expect = 8 + cfg->n_noise_gvps * 6 + 2;
    for (int l = 0; l < cfg->n_convs; ++l) {
        const bool full = cfg->update_kp && l != cfg->n_convs - 1;
        expect += (full ? 4 : 2) * cfg->n_message_gvps * 6 + (full ? 2 : 1) * (cfg->n_update_gvps * 6 + 4);
    }
    if (n_off != expect) { delete m; KPD_REQUIRE(false, "kpd_gvp_create: expected %d offsets, got %d", expect, n_off); }
    for (int k = 0; k < 4; ++k) m->lig_enc[k] = P();
    for (int k = 0; k < 4; ++k) m->kp_enc[k] = P();
    m->layers.resize(cfg->n_convs);
    for (int l = 0; l < cfg->n_convs; ++l) {
        GvpLayerW& L = m->layers[l];
        const bool full = cfg->update_kp && l != cfg->n_convs - 1;
        L.n_et = full ? 4 : 2;
        L.n_dst = full ? 2 : 1;
        for (int e = 0; e < L.n_et; ++e)
            for (int k = 0; k < cfg->n_message_gvps; ++k)
                L.msg[e][k] = k == 0 ? G(m->V + 1, m->V, m->S + cfg->rbf_dim, m->S, 1) : G(m->V, m->V, m->S, m->S, 1);
        for (int nt = 0; nt < L.n_dst; ++nt) {
            for (int k = 0; k < cfg->n_update_gvps; ++k) L.upd[nt][k] = G(m->V, m->V, m->S, m->S, 1);
            L.mln_w[nt] = P(); L.mln_b[nt] = P(); L.uln_w[nt] = P(); L.uln_b[nt] = P();
        }
    }
    for (int k = 0; k < cfg->n_noise_gvps; ++k) {
        const bool last = k == cfg->n_noise_gvps - 1;
        m->head[k] = last ? G(m->V, 1, m->S, 64, 0) : G(m->V, m->V, m->S, m->S, 1);   // dynamics_gvp.py:18-25
    }
    m->WoT = P(); m->bo = P();
    for (auto& L : m->layers) {
        for (int e = 0; e < L.n_et; ++e)
            for (int k = 0; k < cfg->n_message_gvps; ++k) m->all_gvps.push_back(&L.msg[e][k]);
        for (int nt = 0; nt < L.n_dst; ++nt)
            for (int k = 0; k < cfg->n_update_gvps; ++k) m->all_gvps.push_back(&L.upd[nt][k]);
    }
    for (int k = 0; k < cfg->n_noise_gvps; ++k) m->all_gvps.push_back(&m->head[k]);
    {
        int wmax = m->S + cfg->rbf_dim + m->V + 1;
        if (wmax < 64 + m->V) wmax = 64 + m->V;
        m->kch = 2 * ((wmax + 15) / 16);
        m->mode = 0;
    }
    // fp32 SIMT: one node / head tile size whatever the batch
    const size_t smem_node = gvp_smem_bytes(m->lds, TN);
    GvpKernels& k0 = m->k[0];
    k0.edge = {gvp_edge_kernel, NT, gvp_smem_bytes(m->lds, TE), TE};
    k0.node[0] = k0.node[1] = {gvp_node_kernel, NT, smem_node, TN};
    k0.head[0] = k0.head[1] = {gvp_head_kernel, NT, smem_node, TN};
    if (gvp_set_smem(k0) != cudaSuccess) {
        delete m;
        KPD_REQUIRE(false, "kpd_gvp_create: cannot set the dynamic shared memory size of the GVP kernels");
    }
    *out = m;
    return 0;
}

// streams and events of the dependency-graph path of kpd_gvp_forward
static int gvp_dag_init(const kpd_gvp_model* m) {
    if (m->dag_ready) return 0;
    // the node kernels are the critical path (every edge launch of the next conv waits for one of them): their
    // streams get the highest priority so that their few CTAs are dispatched ahead of the queued edge tiles
    int pr_lo = 0, pr_hi = 0;
    cudaDeviceGetStreamPriorityRange(&pr_lo, &pr_hi);
    for (int i = 0; i < 5; ++i)
        KPD_REQUIRE(cudaStreamCreateWithPriority(&m->aux[i], cudaStreamNonBlocking, i >= 3 ? pr_hi : pr_lo) == cudaSuccess, "kpd_gvp: stream creation failed");
    for (int i = 0; i < 4; ++i) KPD_REQUIRE(cudaEventCreateWithFlags(&m->ev_edge[i], cudaEventDisableTiming) == cudaSuccess, "kpd_gvp: event creation failed");
    for (int i = 0; i < 2; ++i) KPD_REQUIRE(cudaEventCreateWithFlags(&m->ev_node[i], cudaEventDisableTiming) == cudaSuccess, "kpd_gvp: event creation failed");
    m->dag_ready = true;
    return 0;
}

extern "C" void kpd_gvp_destroy(kpd_gvp_model* m) {
    if (!m) return;
    if (m->dag_ready) {
        for (auto& s : m->aux) if (s) cudaStreamDestroy(s);
        for (auto& e : m->ev_edge) cudaEventDestroy(e);
        for (auto& e : m->ev_node) cudaEventDestroy(e);
    }
    delete m;
}

// bf16 tensor-core mode: tc_blob holds, for every GVP in creation order (per conv: message GVPs per edge
// type, update GVPs per node type; then the noise head), the packed to_feats_out weight and the packed
// gates weight (pack.pack_tc_weight); byte_offsets has two entries per GVP.
extern "C" int kpd_gvp_attach_tc(kpd_gvp_model* m, const void* tc_blob, const int64_t* byte_offsets, int32_t n,
                                 int32_t nsplit) {
    KPD_REQUIRE(m && tc_blob && byte_offsets, "kpd_gvp_attach_tc: null argument");
    KPD_REQUIRE(nsplit == 1 || nsplit == 2, "kpd_gvp_attach_tc: nsplit must be 1 (bf16) or 2 (bf16 hi/lo)");
    KPD_REQUIRE(n == 3 * (int)m->all_gvps.size(), "kpd_gvp_attach_tc: expected %d offsets, got %d", 3 * (int)m->all_gvps.size(), n);
    KPD_REQUIRE((reinterpret_cast<uintptr_t>(tc_blob) & 127) == 0, "kpd_gvp_attach_tc: blob must be 128-byte aligned");
    KPD_REQUIRE(m->S % 16 == 0, "kpd_gvp_attach_tc: n_hidden_scalars must be a multiple of 16 for the tensor-core mode");
    const size_t smem_ws1 = ws::smem_bytes<WsBf16>(m->kch), smem_ws2 = ws::smem_bytes<WsSplit>(m->kch),
                 smem_ws1n = ws::smem_bytes<WsBf16N>(m->kch);
    KPD_REQUIRE(smem_ws1 <= 227 * 1024 && smem_ws2 <= 227 * 1024 && smem_ws1n <= 227 * 1024,
                "kpd_gvp_attach_tc: tile needs %zu / %zu / %zu B of shared memory", smem_ws1, smem_ws2, smem_ws1n);
    const char* base = static_cast<const char*>(tc_blob);
    for (size_t i = 0; i < m->all_gvps.size(); ++i) {
        KPD_REQUIRE(byte_offsets[3 * i] % 16 == 0 && byte_offsets[3 * i + 1] % 16 == 0 && byte_offsets[3 * i + 2] % 16 == 0,
                    "kpd_gvp_attach_tc: unaligned offset");
        KPD_REQUIRE(m->all_gvps[i]->fout % 8 == 0, "kpd_gvp_attach_tc: GVP output widths must be multiples of 8");
        const uint4* wf = reinterpret_cast<const uint4*>(base + byte_offsets[3 * i]);
        const uint4* wg = reinterpret_cast<const uint4*>(base + byte_offsets[3 * i + 1]);
        const float* ws_img = reinterpret_cast<const float*>(base + byte_offsets[3 * i + 2]);
        if (nsplit == 1) { m->all_gvps[i]->WfP = wf; m->all_gvps[i]->WgP = wg; m->all_gvps[i]->wsmP = ws_img; }
        else {
            GvpW* gw = m->all_gvps[i];
            gw->WfP2 = wf; gw->WgP2 = wg; gw->wsmP2 = ws_img;
            // the (hi, lo) slab image of the gates weight follows its fragment image: both are 2 planes x 512 B per k-step
            const int ksg = ((gw->fout + 15) & ~15) >> 4;
            gw->WgP2c = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(wg) + (size_t)ksg * 1024);
        }
    }
    // bf16x3: the edge kernel keeps (hi, lo) planes of 128-row tiles (WsKS) when that tile fits in 227 KB of shared
    // memory, and runs the 64-row stacked-operand kernel (WsSplit) otherwise
    const GvpKernels k = nsplit == 1 ? gvp_ws_kernels<WsBf16, WsBf16N>(m->kch)
                       : ws::smem_bytes<WsKS>(m->kch) <= 227 * 1024 ? gvp_ws_kernels<WsKS, WsSplit>(m->kch)
                                                                   : gvp_ws_kernels<WsSplit, WsSplit>(m->kch);
    KPD_REQUIRE(gvp_set_smem(k) == cudaSuccess, "kpd_gvp_attach_tc: cannot set %zu / %zu B of dynamic shared memory",
                k.edge.smem, k.node[0].smem);
    m->k[nsplit] = k;
    return gvp_dag_init(m);
}

// event trace of one edge-kernel CTA (only with -DKPD_WS_TRACE): out = [n][3] (tag, warp, clock); returns n via *count
extern "C" int kpd_debug_ws_trace(unsigned long long* out, int32_t cap, int32_t* count) {
#ifdef KPD_WS_TRACE
    cudaError_t e = cudaDeviceSynchronize();
    int n = 0;
    if (e == cudaSuccess) e = cudaMemcpyFromSymbol(&n, g_ws_trace_n, sizeof(int));
    if (n > 2048) n = 2048;
    if (n > cap) n = cap;
    if (e == cudaSuccess && n > 0) e = cudaMemcpyFromSymbol(out, g_ws_trace, sizeof(unsigned long long) * 3 * n);
    KPD_REQUIRE(e == cudaSuccess, "kpd_debug_ws_trace: %s", cudaGetErrorString(e));
    *count = n;
    return 0;
#else
    (void)out; (void)cap;
    *count = 0;
    return 0;
#endif
}

// launch timeline of the GVP convs (only with -DKPD_TIMELINE): out = [256][3] (first CTA start ns, last CTA end ns,
// working CTAs); reset != 0 clears it afterwards.  Returns the number of slots (0 when not compiled in).
extern "C" int kpd_debug_timeline(unsigned long long* out, int32_t reset) {
#ifdef KPD_TIMELINE
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess && out) e = cudaMemcpyFromSymbol(out, g_tl, sizeof(unsigned long long) * 3 * 256);
    if (e == cudaSuccess && reset) {
        static unsigned long long z[3 * 256];
        for (int i = 0; i < 256; ++i) { z[3 * i] = ~0ull; z[3 * i + 1] = 0; z[3 * i + 2] = 0; }
        e = cudaMemcpyToSymbol(g_tl, z, sizeof(z));
    }
    KPD_REQUIRE(e == cudaSuccess, "kpd_debug_timeline: %s", cudaGetErrorString(e));
    return 256;
#else
    (void)out; (void)reset;
    return 0;
#endif
}

// same for the warp-specialised kernels (gvp_ws.inl)
extern "C" int kpd_debug_ws_times(unsigned long long* out64) {
    KPD_REQUIRE(out64, "kpd_debug_ws_times: null argument");
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out64, g_ws_times, sizeof(unsigned long long) * 64);
    unsigned long long z[64] = {0};
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_ws_times, z, sizeof(z));
    KPD_REQUIRE(e == cudaSuccess, "kpd_debug_ws_times: %s", cudaGetErrorString(e));
    return 0;
}

// mode 0 = fp32 SIMT (parity mode), 1 = bf16 operands on tcgen05 tensor cores
extern "C" int kpd_gvp_set_mode(kpd_gvp_model* m, int32_t mode) {
    KPD_REQUIRE(m, "kpd_gvp_set_mode: null model");
    KPD_REQUIRE(mode >= 0 && mode <= 2, "kpd_gvp_set_mode: mode must be 0 (fp32 SIMT), 1 (bf16) or 2 (bf16x3 tensor cores)");
    KPD_REQUIRE(m->k[mode].edge.fn, "kpd_gvp_set_mode: call kpd_gvp_attach_tc(nsplit = %d) first", mode);
    m->mode = mode;
    return 0;
}

extern "C" int kpd_gvp_dims(const kpd_gvp_model* m, int* n_kp_scalars, int* vector_size) {
    KPD_REQUIRE(m, "kpd_gvp_dims: null model");
    *n_kp_scalars = m->C; *vector_size = m->V;
    return 0;
}

extern "C" int64_t kpd_gvp_workspace_bytes(const kpd_gvp_model* m, const kpd_batch* batch, int32_t cap_ll,
                                           int32_t cap_kl, int32_t cap_kk) {
    const int caps[4] = {cap_ll, cap_kl, cap_kl, cap_kk};
    int64_t bytes = 0;
    gvp_carve(m, batch, caps, nullptr, &bytes);
    return bytes;
}

extern "C" int kpd_gvp_forward(const kpd_gvp_model* m, const kpd_batch* b, const float* h_lig, const float* x_lig,
                               const float* h_kp, const float* x_kp, const float* v_kp, const float* t_ptr,
                               int32_t t_per_complex, const kpd_csr* ll, const kpd_csr* kl, const kpd_csr* lk,
                               const kpd_csr* kk, float* eps_h, float* eps_x, void* workspace, void* stream) {
    KPD_REQUIRE(m && b && h_lig && x_lig && h_kp && x_kp && v_kp && t_ptr && ll && kl && eps_h && eps_x && workspace,
                "kpd_gvp_forward: null argument");
    const bool ukp = m->cfg.update_kp != 0;
    KPD_REQUIRE(!ukp || (lk && kk), "kpd_gvp_forward: update_kp needs lk and kk graphs");
    KPD_REQUIRE(ukp || m->cfg.n_convs == 1, "kpd_gvp_forward: update_kp=False only works with one conv in the reference (SURVEY N6)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const kpd_csr* G[4] = {ll, kl, lk, kk};
    const int caps[4] = {ll->cap, kl->cap, ukp ? lk->cap : 0, ukp ? kk->cap : 0};
    GvpWs w = gvp_carve(m, b, caps, workspace, nullptr);
    const int N[2] = {b->n_lig, b->n_kp};
    const int S = m->S, V = m->V;

    // ---- encoders: time concatenated first, Linear + SiLU + LayerNorm (dynamics_gvp.py:161-169) -> buffer set 0
    if (m->mode != 0) {       // tensor-core modes: everything up to the first conv in one launch
        GvpEncArgs ea;
        memset(&ea, 0, sizeof(ea));
        ea.n[0] = N[0]; ea.n[1] = N[1]; ea.K[0] = m->F; ea.K[1] = m->C;
        ea.in[0] = h_lig; ea.in[1] = h_kp;
        for (int nt = 0; nt < 2; ++nt) {
            const float* const* enc = nt == 0 ? m->lig_enc : m->kp_enc;
            ea.WT[nt] = enc[0]; ea.bias[nt] = enc[1]; ea.lnw[nt] = enc[2]; ea.lnb[nt] = enc[3];
            ea.s[nt] = w.s[0][nt]; ea.s_hi[nt] = w.s_hi[0][nt]; ea.s_lo[nt] = w.s_lo[0][nt]; ea.v[nt] = w.v[0][nt];
        }
        ea.batch[0] = b->lig_batch; ea.batch[1] = b->kp_batch;
        ea.v_kp = v_kp; ea.t_ptr = t_ptr; ea.t_per_complex = t_per_complex; ea.S = S; ea.Sp = m->Sp; ea.V = V;
        const int mx = N[0] > N[1] ? N[0] : N[1];
        if (mx > 0) {
            gvp_encode_kernel<<<dim3(cdiv(mx, 8 * ENC_ROWS), 2), 256, 0, st>>>(ea);
            KPD_TRY(check_launch("gvp_encode_kernel"));
        }
    } else {
    KPD_TRY(launch_concat_time(h_lig, m->F, w.tin, m->F + 1, N[0], t_ptr, b->lig_batch, t_per_complex, st));
    KPD_TRY(launch_linear(w.tin, m->F + 1, m->lig_enc[0], m->Sp, m->lig_enc[1], nullptr, 0, w.tenc, S, N[0], m->F + 1, S, 1, st));
    KPD_TRY(launch_layernorm(w.tenc, S, w.s[0][0], S, N[0], S, m->lig_enc[2], m->lig_enc[3], st));
    KPD_TRY(launch_concat_time(h_kp, m->C, w.tin, m->C + 1, N[1], t_ptr, b->kp_batch, t_per_complex, st));
    KPD_TRY(launch_linear(w.tin, m->C + 1, m->kp_enc[0], m->Sp, m->kp_enc[1], nullptr, 0, w.tenc, S, N[1], m->C + 1, S, 1, st));
    KPD_TRY(launch_layernorm(w.tenc, S, w.s[0][1], S, N[1], S, m->kp_enc[2], m->kp_enc[3], st));
    // ligand vectors start at zero (:179-184); keypoint vectors come from the receptor encoder
    cudaError_t ce = cudaMemsetAsync(w.v[0][0], 0, sizeof(float) * (size_t)N[0] * V * 3, st);
    KPD_REQUIRE(ce == cudaSuccess, "kpd_gvp_forward: memset failed: %s", cudaGetErrorString(ce));
    KPD_TRY(launch_copy_rows(v_kp, V * 3, w.v[0][1], V * 3, N[1], V * 3, st));
    }
    const int src_nt[4] = {0, 1, 0, 1}, dst_nt[4] = {0, 0, 1, 1};
    const float* X[2] = {x_lig, x_kp};
    const int norm_mode = m->cfg.norm_mode;
    const GvpKernels& K = m->k[m->mode];

    // Tensor-core modes run the convs as a DEPENDENCY GRAPH instead of a chain of launches: one edge launch per edge
    // type, one node launch per node type, each waiting only for what it reads --
    //     edge(l, e)  <- node(l-1, src type of e)                 (messages read source features only, gvp.py:472-497)
    //     node(l, nt) <- edge(l, e) for the edge types into nt
    // -- on one stream per edge type (kl: the caller's; ll, lk, kk: three auxiliary streams joined by events, which
    // stream capture turns into graph edges).  Node features and aggregates are double-buffered by conv parity, so a
    // node kernel never overwrites what a still-running edge kernel of the same conv reads.  The point: a conv's
    // 650 edge tiles are 4.4 waves of one CTA per SM and its node tiles a fifth of a wave; as separate launches their
    // tails leave SMs idle, as a graph the tail of one kernel is filled with the CTAs of the next ready one.
    // The fp32 mode, the CUDA-event profiler (bench.py's roofline leg) and KPD_GVP_SERIAL=1 run the convs serially:
    // one launch for all edge types of a conv and one for all its node types, on the caller's stream.
    const bool dag = m->mode != 0 && !m->serial && !prof_enabled();
    if (dag) KPD_TRY(gvp_dag_init(m));       // normally done by kpd_gvp_attach_tc, outside any stream capture
    // stream of edge type e (ll, kl, lk, kk) and of node type nt
    cudaStream_t es[4] = {st, st, st, st}, ns[2] = {st, st};
    if (dag) { es[0] = m->aux[0]; es[2] = m->aux[1]; es[3] = m->aux[2]; ns[0] = m->aux[3]; ns[1] = m->aux[4]; }
#define KPD_CU(x) do { cudaError_t e_ = (x); KPD_REQUIRE(e_ == cudaSuccess, "kpd_gvp_forward: %s", cudaGetErrorString(e_)); } while (0)
    if (dag) {      // the encoder output is what every first-conv edge launch waits for
        KPD_CU(cudaEventRecord(m->ev_node[0], st));
        KPD_CU(cudaEventRecord(m->ev_node[1], st));
    }
    bool used[4] = {false, false, false, false}, nused[2] = {false, false};     // auxiliary work to join at the end

    auto fill_edge = [&](GvpEdgeLaunch& L, int slot, int e, const GvpLayerW& W, int cur) {
        GvpEtypeArgs& a = L.e[slot];
        a.rowptr = G[e]->rowptr; a.src = G[e]->src; a.dst = G[e]->dst; a.n_dst = G[e]->n_dst; a.cap = caps[e] > 0 ? caps[e] : 1;
        a.s_src = w.s[cur][src_nt[e]]; a.v_src = w.v[cur][src_nt[e]];
        a.s_hi = w.s_hi[cur][src_nt[e]]; a.s_lo = w.s_lo[cur][src_nt[e]];
        a.xs = X[src_nt[e]]; a.xd = X[dst_nt[e]];
        for (int k = 0; k < L.n_msg; ++k) a.msg[k] = W.msg[e][k];
        a.sm = w.sm[cur][e]; a.vm = w.vm[cur][e]; a.part = w.part[cur][e];
    };
    auto fill_node = [&](GvpNodeLaunch& NL, int slot, int nt, const GvpLayerW& W, int cur, int nxt) {
        GvpNodeArgs& a = NL.nt[slot];
        a.n = N[nt]; a.Sdim = S; a.Vdim = V; a.lds = m->lds; a.pw = m->pw;
        a.n_upd = m->cfg.n_update_gvps; a.n_et = 2; a.kch = m->kch; a.edge_tile = K.edge.rows;
        a.s = w.s[cur][nt]; a.v = w.v[cur][nt]; a.s_hi = w.s_hi[cur][nt]; a.s_lo = w.s_lo[cur][nt];
        a.s_out = w.s[nxt][nt]; a.v_out = w.v[nxt][nt]; a.s_hi_out = w.s_hi[nxt][nt]; a.s_lo_out = w.s_lo[nxt][nt];
        for (int k = 0; k < 2; ++k) {
            const int e = nt * 2 + k;
            a.rowptr[k] = G[e]->rowptr; a.sm[k] = w.sm[cur][e]; a.vm[k] = w.vm[cur][e]; a.part[k] = w.part[cur][e];
        }
        a.norm_mode = norm_mode; a.norm_const = m->cfg.message_norm;
        a.node_batch = nt == 0 ? b->lig_batch : b->kp_batch;
        a.ptr = nt == 0 ? b->lig_ptr : b->kp_ptr;
        for (int k = 0; k < a.n_upd; ++k) a.upd[k] = W.upd[nt][k];
        a.mln_w = W.mln_w[nt]; a.mln_b = W.mln_b[nt]; a.uln_w = W.uln_w[nt]; a.uln_b = W.uln_b[nt];
    };
    // full 64-row node / head tiles for calls of >= 32 complexes (capacity: the layouts of the capacity-bucketed samplers
    // round 23 .. 31 real complexes up to 32, 16 .. 22 up to 24; tests/test_modules_cpu.py pins that): the sampler cuts batches of >= 64 complexes into four
    // concurrent groups and smaller ones into groups of >= 16, so a call this large means the GPU is kept full by its
    // siblings and SM time, not the critical path, is what counts (gvp_ws.inl: NODE_ROWS; measured: headline, groups of 25:
    // 89.3 -> 92.1 ligands/s; gvp_ca with 16 ligands in one group: 33.1 with 32-row tiles, 29.9 with 64)
    const bool full_node_tiles = b->B >= 32;
    const GvpKernel<GvpNodeLaunch>& node_k = K.node[full_node_tiles];

    int fin = 0;        // buffer set holding the final ligand features
    for (int l = 0; l < m->cfg.n_convs; ++l) {
        const GvpLayerW& W = m->layers[l];
        // serial paths update in place (set 0); the graph path ping-pongs
        const int cur = dag ? (l & 1) : 0, nxt = dag ? ((l + 1) & 1) : 0;
        // launch groups: the graph path launches each edge / node type on its own, the serial path all of them at once
        const int eg = dag ? 1 : W.n_et, ng = dag ? 1 : W.n_dst;
        GvpEdgeLaunch L;
        memset(&L, 0, sizeof(L));
        L.Sdim = S; L.Vdim = V; L.n_msg = m->cfg.n_message_gvps; L.lds = m->lds; L.pw = m->pw;
        L.rbf_dim = m->cfg.rbf_dim;
        L.rbf_step = m->cfg.rbf_dmax / (float)(m->cfg.rbf_dim - 1);   // linspace(0, D_max, D_count)
        L.rbf_sigma = m->cfg.rbf_dmax / (float)m->cfg.rbf_dim;
        L.kch = m->kch;
        for (int e0 = 0; e0 < W.n_et; e0 += eg) {
            GvpEdgeLaunch Lg = L;
            Lg.tl_slot = 8 * l + e0;
            int cap = 1;
            for (int e = e0; e < e0 + eg; ++e) {
                fill_edge(Lg, e - e0, e, W, cur);
                if (caps[e] > cap) cap = caps[e];
                if (dag) KPD_CU(cudaStreamWaitEvent(es[e], m->ev_node[src_nt[e]], 0));
            }
            prof_begin(PROF_GVP_EDGE, es[e0]);
            launch_with_priority(K.edge, dim3(cdiv(cap, K.edge.rows), eg), es[e0], Lg);
            KPD_TRY(check_launch("gvp edge kernel"));
            prof_end(PROF_GVP_EDGE, es[e0]);
            if (dag) {
                KPD_CU(cudaEventRecord(m->ev_edge[e0], es[e0]));
                used[e0] = true;
            }
        }
        for (int nt0 = 0; nt0 < W.n_dst; nt0 += ng) {
            GvpNodeLaunch NL;
            memset(&NL, 0, sizeof(NL));
            NL.tl_slot = 8 * l + 4 + nt0;
            int max_n = 0;
            for (int nt = nt0; nt < nt0 + ng; ++nt) {
                fill_node(NL, nt - nt0, nt, W, cur, nxt);
                if (N[nt] > max_n) max_n = N[nt];
            }
            if (max_n <= 0) continue;
            if (dag)
                for (int k = 0; k < 2; ++k) KPD_CU(cudaStreamWaitEvent(ns[nt0], m->ev_edge[2 * nt0 + k], 0));
            prof_begin(PROF_GVP_NODE, ns[nt0]);
            launch_with_priority(node_k, dim3(cdiv(max_n, node_k.rows), ng), ns[nt0], NL, dag);
            KPD_TRY(check_launch("gvp node kernel"));
            prof_end(PROF_GVP_NODE, ns[nt0]);
            if (dag) {
                KPD_CU(cudaEventRecord(m->ev_node[nt0], ns[nt0]));
                nused[nt0] = true;
            }
        }
        // graph path: a node type this conv does not update (the last conv is lig-only) simply keeps its current set;
        // nothing reads it afterwards (dynamics_gvp.py:71-72)
        fin = nxt;
    }
    if (dag) {
        // join: everything launched on the auxiliary streams is ordered before the head / the end of this call
        for (int e = 0; e < 4; ++e) if (used[e] && es[e] != st) KPD_CU(cudaStreamWaitEvent(st, m->ev_edge[e], 0));
        for (int nt = 0; nt < 2; ++nt) if (nused[nt]) KPD_CU(cudaStreamWaitEvent(st, m->ev_node[nt], 0));
    }
#undef KPD_CU
    {
        GvpHeadArgs a;
        memset(&a, 0, sizeof(a));
        a.n = N[0]; a.Sdim = S; a.Vdim = V; a.lds = m->lds; a.n_gvps = m->cfg.n_noise_gvps;
        a.F = m->F; a.Fp = m->Fp; a.hid_out = 64;
        a.s = w.s[fin][0]; a.v = w.v[fin][0]; a.s_hi = w.s_hi[fin][0]; a.s_lo = w.s_lo[fin][0];
        for (int k = 0; k < a.n_gvps; ++k) a.g[k] = m->head[k];
        a.WoT = m->WoT; a.bo = m->bo; a.eps_h = eps_h; a.eps_x = eps_x;
        if (a.n > 0) {
            prof_begin(PROF_GVP_HEAD, st);
            a.kch = m->kch;
            const GvpKernel<GvpHeadArgs>& head_k = K.head[full_node_tiles];
            launch_with_priority(head_k, dim3(cdiv(a.n, head_k.rows)), st, a);
            KPD_TRY(check_launch("gvp head kernel"));
            prof_end(PROF_GVP_HEAD, st);
        }
    }
    return 0;
}
