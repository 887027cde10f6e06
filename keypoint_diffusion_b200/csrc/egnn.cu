// (b)+(d) EGNN denoiser on flat tensors + dst-sorted CSR.
//
// Replaces LigRecDynamics.forward (models/dynamics.py:342-385), LigRecEGNN.forward (:266-294)
// and LigRecConv.forward/message/compute_dij (:89-217) of the reference.
//
// Per layer:
//   1. node pre-GEMM: the first Linear of edge_mlp / coord_mlp acts on [h_src, h_dst, dij]
//      (:103-111); W1.[h_s,h_d,d] = W1a.h_s + W1b.h_d + w1c.d, so the two h terms are computed
//      once per NODE and role (P = h @ [W1a|W1b]^T, bias folded into the dst role) instead of
//      once per edge -- 2/3 of the per-edge FLOPs move to an M = #nodes GEMM;
//   2. fused edge kernel (one CTA per tile of 64 dst-sorted edges, both branches):
//      gather P_src + P_dst + w1c*dij -> SiLU -> [64 x H] tile in shared memory -> second
//      Linear as a tile GEMM (weights streamed through a cp.async pipeline) -> SiLU ->
//      soft attention / coordinate weight -> deterministic segmented reduction by destination.
//      No E x H tensor is ever written to HBM;
//   3. node stage: h_neigh / x_neigh are recombined from the per-tile outputs, node MLP,
//      residual, LayerNorm, x += x_neigh.
//
// Offsets array (float offsets into the packed blob; -1 = absent), in this order:
//   globals  [12]: lig_enc.W0T, b0, W1T, b1, rec_enc.W0T, b0, W1T, b1, dec.W0T, b0, W1T, b1
//   per layer:
//     for nt in (lig, kp):               WpreT[nt], bpre[nt]
//     for et in etypes:                  for br in (edge, coord): w1c, W2T, b2, W2lo
//                                        watt, batt, w3c
//     for nt in updated ntypes:          Wn1T, bn1, Wn2T, bn2, lnw, lnb
//   etypes = (ll, kl, lk, kk) if update_kp_feat else (ll, kl); updated = (lig, kp) | (lig).
//   Roles (slot = 2*role + branch) inside P: lig: ll.s, ll.d, lk.s, kl.d  | ll.s, ll.d, kl.d
//                                            kp : kl.s, kk.s, kk.d, lk.d  | kl.s
#include "common.cuh"
#include "ws_common.cuh"
#include "tc_gemm.cuh"
#include <string.h>
#include <type_traits>
#include <vector>

namespace kpd {

struct EgnnEtypeArgs {
    const int* rowptr; const int* src; const int* dst; int n_dst; int cap;
    const float* Ps; int ldps; int slot_s;
    const float* Pd; int ldpd; int slot_d;
    const float* xs; const float* xd;
    const float* w1c[2]; const float* W2T[2]; const float* b2[2]; const float* W2lo[2];
    const float* watt; const float* batt; const float* w3c;
    float* hn; float* xn; float* part;
};

struct EgnnEdgeLaunch {
    EgnnEtypeArgs e[4];
    int H, Hp, nmain, nlo, lda, pw;
    int use_tanh;
    float coords_range;
};

__global__ void __launch_bounds__(NT, 1) egnn_edge_kernel(const EgnnEdgeLaunch L) {
    const EgnnEtypeArgs& a = L.e[blockIdx.y];
    const int E = a.rowptr[a.n_dst];
    const int tile_begin = blockIdx.x * TE;
    if (tile_begin >= E) return;
    const int n = min(TE, E - tile_begin);

    extern __shared__ __align__(16) float smem[];
    float* As = smem;                               // [TE][lda]
    float* Bs = As + TE * L.lda;                    // [2][KC][256]
    float* lo_s = Bs + BS_FLOATS;                   // [TE][4]
    float* xsc_s = lo_s + TE * 4;                   // [TE][3]  x_diff / (dij + 1)
    float* xm_s = xsc_s + TE * 3;                   // [TE][3]  coordinate messages
    float* dij_s = xm_s + TE * 3;                   // [TE]
    int* src_s = reinterpret_cast<int*>(dij_s + TE);
    int* dst_s = src_s + TE;

    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
    const int H = L.H, Hp = L.Hp, lda = L.lda, nmain = L.nmain, nlo = L.nlo;

    zero_stage(Bs);
    if (tid < TE) {
        const int e = tile_begin + min(tid, n - 1);     // rows >= n replicate the last valid edge
        const int s = a.src[e], d = a.dst[e];
        src_s[tid] = s;
        dst_s[tid] = d;
        // models/dynamics.py:160 (u_sub_v), :211 (||x_diff||), :169 (x_diff / (dij + 1))
        const float dx = a.xs[3 * s] - a.xd[3 * d], dy = a.xs[3 * s + 1] - a.xd[3 * d + 1],
                    dz = a.xs[3 * s + 2] - a.xd[3 * d + 2];
        const float dij = sqrtf(dx * dx + dy * dy + dz * dz);
        dij_s[tid] = dij;
        const float inv = 1.0f / (dij + 1.0f);
        xsc_s[3 * tid] = dx * inv; xsc_s[3 * tid + 1] = dy * inv; xsc_s[3 * tid + 2] = dz * inv;
    }
    __syncthreads();

    for (int br = 0; br < 2; ++br) {
        // ---- 1. first Linear (factorised) + SiLU -> As
        {
            const float* w1c = a.w1c[br];
            const int nf4 = Hp >> 2;
            for (int rr = 0; rr < TE / 8; ++rr) {
                const int r = warp * (TE / 8) + rr;
                const float* ps = a.Ps + (size_t)src_s[r] * a.ldps + (a.slot_s + br) * Hp;
                const float* pd = a.Pd + (size_t)dst_s[r] * a.ldpd + (a.slot_d + br) * Hp;
                const float d = dij_s[r];
                for (int f = lane; f < nf4; f += 32) {
                    const float4 u = *reinterpret_cast<const float4*>(ps + 4 * f);
                    const float4 v = *reinterpret_cast<const float4*>(pd + 4 * f);
                    const float4 w = *reinterpret_cast<const float4*>(w1c + 4 * f);
                    float4 o;
                    o.x = silu_f(u.x + v.x + w.x * d);
                    o.y = silu_f(u.y + v.y + w.y * d);
                    o.z = silu_f(u.z + v.z + w.z * d);
                    o.w = silu_f(u.w + v.w + w.w * d);
                    *reinterpret_cast<float4*>(As + r * lda + 4 * f) = o;
                }
            }
        }
        __syncthreads();
        // ---- 2. leftover output columns (H - nmain <= 3) as plain dot products
        if (nlo > 0) {
            const float* W2lo = a.W2lo[br];
            for (int rr = 0; rr < TE / 8; ++rr) {
                const int r = warp * (TE / 8) + rr;
                for (int c = 0; c < nlo; ++c) {
                    float s = 0.f;
                    for (int k = lane; k < H; k += 32) s = fmaf(As[r * lda + k], W2lo[c * Hp + k], s);
#pragma unroll
                    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane == 0) lo_s[r * 4 + c] = silu_f(s + a.b2[br][nmain + c]);
                }
            }
        }
        // ---- 3. second Linear: [TE x H] @ W2T[H x nmain]
        float acc[TE / 16][16];
#pragma unroll
        for (int i = 0; i < TE / 16; ++i)
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[i][j] = 0.f;
        tile_gemm<TE / 16>(As, lda, a.W2T[br], Hp, H, nmain, Bs, acc);
        // ---- 4. epilogue
        const float* b2 = a.b2[br];
        const float* wv = br == 0 ? a.watt : a.w3c;
#pragma unroll
        for (int i = 0; i < TE / 16; ++i) {
            const int r = ty * (TE / 16) + i;
            float dot = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int col = 4 * tx + 64 * j + q;
                    float v = 0.f;
                    if (col < nmain) {
                        v = silu_f(acc[i][4 * j + q] + b2[col]);
                        dot = fmaf(v, wv[col], dot);
                    }
                    acc[i][4 * j + q] = v;
                }
#pragma unroll
            for (int o = 8; o; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
            for (int c = 0; c < nlo; ++c) dot = fmaf(lo_s[r * 4 + c], wv[nmain + c], dot);
            if (br == 0) {
                // msg_h = m2 * sigmoid(Linear(m2))   (models/dynamics.py:111-112)
                const float att = sigmoid_f(dot + a.batt[0]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int col = 4 * tx + 64 * j;
                    if (col < nmain)
                        *reinterpret_cast<float4*>(As + r * lda + col) =
                            make_float4(acc[i][4 * j] * att, acc[i][4 * j + 1] * att,
                                        acc[i][4 * j + 2] * att, acc[i][4 * j + 3] * att);
                }
                if (tx == 0)
                    for (int c = 0; c < nlo; ++c) As[r * lda + nmain + c] = lo_s[r * 4 + c] * att;
            } else if (tx == 0) {
                // msg_x = tanh(coord_mlp(f)) * x_diff * coords_range  | coord_mlp(f) * x_diff (:117-120)
                const float cw = L.use_tanh ? tanhf(dot) * L.coords_range : dot;
                xm_s[3 * r] = cw * xsc_s[3 * r];
                xm_s[3 * r + 1] = cw * xsc_s[3 * r + 1];
                xm_s[3 * r + 2] = cw * xsc_s[3 * r + 2];
            }
        }
        __syncthreads();
        // ---- 5. deterministic segmented reduction by destination (copy_e + sum, :177-185)
        SegOut o;
        o.part0 = a.part + ((size_t)blockIdx.x * 2 + 0) * L.pw;
        o.part1 = a.part + ((size_t)blockIdx.x * 2 + 1) * L.pw;
        if (br == 0) {
            o.out = a.hn; o.ld_out = Hp;
            for (int col = tid; col < H; col += NT)
                seg_reduce_column(As, lda, col, n, dst_s, a.rowptr, tile_begin, o, col);
        } else if (tid < 3) {
            o.out = a.xn; o.ld_out = 4;
            // partial slots for x live behind the Hp feature columns
            o.part0 += Hp; o.part1 += Hp;
            seg_reduce_column(xm_s, 3, tid, n, dst_s, a.rowptr, tile_begin, o, tid);
        }
        __syncthreads();
    }
}

// node stage, part 1: cat = [h | h_neigh], x += x_neigh   (models/dynamics.py:188-206)
struct EgnnNodePrep {
    int n, H, Hp, ldcat, pw;
    const float* h; float* cat; float* x;
    int n_et;
    const int* rowptr[2]; const float* hn[2]; const float* xn[2]; const float* part[2];
    int z_mode;            // 0: no division (reference as executed), 1: constant, 2: mean in-degree + 1
    float z_const;
    const int* node_batch; const int* ptr;
};

__global__ void __launch_bounds__(128) egnn_node_prep_kernel(const EgnnNodePrep a) {
    const int nd = blockIdx.x;
    if (nd >= a.n) return;
    float z = 1.0f;
    if (a.z_mode == 1) z = a.z_const;
    else if (a.z_mode == 2) {
        const int b = a.node_batch[nd];
        const int p0 = a.ptr[b], p1 = a.ptr[b + 1];
        int tot = 0;
        for (int e = 0; e < a.n_et; ++e) tot += a.rowptr[e][p1] - a.rowptr[e][p0];
        z = (float)tot / (float)(p1 - p0) + 1.0f;     // (:281-283)
    }
    int r0[2], r1[2];
    for (int e = 0; e < a.n_et; ++e) { r0[e] = a.rowptr[e][nd]; r1[e] = a.rowptr[e][nd + 1]; }
    for (int c = threadIdx.x; c < a.H + 3; c += blockDim.x) {
        if (c < a.H) {
            float s = 0.f;
            for (int e = 0; e < a.n_et; ++e) s += seg_gather(a.hn[e], a.Hp, a.part[e], a.pw, r0[e], r1[e], nd, c);
            if (a.z_mode) s = s / z;
            a.cat[(size_t)nd * a.ldcat + c] = a.h[(size_t)nd * a.Hp + c];
            a.cat[(size_t)nd * a.ldcat + a.H + c] = s;
        } else {
            const int k = c - a.H;
            float s = 0.f;
            for (int e = 0; e < a.n_et; ++e) s += seg_gather(a.xn[e], 4, a.part[e] + a.Hp, a.pw, r0[e], r1[e], nd, k);
            if (a.z_mode) s = s / z;
            a.x[3 * nd + k] += s;                     // x = x + x_neigh (:206)
        }
    }
}

#include "egnn_ws.inl"

// the same node stage for the tensor-core mode: one warp per node, a lane per 8-feature chunk (float4 traffic, all
// loads of a node in flight together); h_neigh starts at column off_neigh of the cat row (a multiple of 4: the packed
// node_mlp.0 weight has matching zero columns, pack.pack_egnn_tc)
__device__ __forceinline__ void node_prep_warp_body(const EgnnNodePrep& a, int off_neigh, int blk) {
    const int nd = blk * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (nd >= a.n) return;
    float z = 1.0f;
    if (a.z_mode == 1) z = a.z_const;
    else if (a.z_mode == 2) {
        const int b = a.node_batch[nd];
        const int p0 = a.ptr[b], p1 = a.ptr[b + 1];
        int tot = 0;
        for (int e = 0; e < a.n_et; ++e) tot += a.rowptr[e][p1] - a.rowptr[e][p0];
        z = (float)tot / (float)(p1 - p0) + 1.0f;     // (:281-283)
    }
    const float iz = a.z_mode ? 1.0f / z : 1.0f;
    int r0[2], r1[2];
    for (int e = 0; e < 2; ++e) { r0[e] = e < a.n_et ? a.rowptr[e][nd] : 0; r1[e] = e < a.n_et ? a.rowptr[e][nd + 1] : 0; }
    float* crow = a.cat + (size_t)nd * a.ldcat;
    const float* hrow = a.h + (size_t)nd * a.Hp;
    const int nfull = a.H >> 3;
    if (lane < nfull) {
        const float4 h0 = *reinterpret_cast<const float4*>(hrow + 8 * lane), h1 = *reinterpret_cast<const float4*>(hrow + 8 * lane + 4);
        float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int e = 0; e < a.n_et; ++e) {
            if (r1[e] <= r0[e]) continue;
            const int t0 = r0[e] / TE, t1 = (r1[e] - 1) / TE;
            const float* p = t0 == t1 ? a.hn[e] + (size_t)nd * a.Hp : a.part[e] + ((size_t)t0 * 2 + 1) * a.pw;
            for (int t = t0;; ++t) {
                const float4 u0 = *reinterpret_cast<const float4*>(p + 8 * lane), u1 = *reinterpret_cast<const float4*>(p + 8 * lane + 4);
                s[0] += u0.x; s[1] += u0.y; s[2] += u0.z; s[3] += u0.w; s[4] += u1.x; s[5] += u1.y; s[6] += u1.z; s[7] += u1.w;
                if (t + 1 > t1 || t0 == t1) break;
                p = a.part[e] + ((size_t)(t + 1) * 2 + 0) * a.pw;
            }
        }
        *reinterpret_cast<float4*>(crow + 8 * lane) = h0;
        *reinterpret_cast<float4*>(crow + 8 * lane + 4) = h1;
        *reinterpret_cast<float4*>(crow + off_neigh + 8 * lane) = make_float4(s[0] * iz, s[1] * iz, s[2] * iz, s[3] * iz);
        *reinterpret_cast<float4*>(crow + off_neigh + 8 * lane + 4) = make_float4(s[4] * iz, s[5] * iz, s[6] * iz, s[7] * iz);
    }
    // leftover features (H = 257: feature 256), the zero gap up to off_neigh, and x += x_neigh (:206)
    for (int c = 8 * nfull + lane; c < a.H + 3; c += 32) {
        if (c < a.H) {
            float s = 0.f;
            for (int e = 0; e < a.n_et; ++e) s += seg_gather(a.hn[e], a.Hp, a.part[e], a.pw, r0[e], r1[e], nd, c);
            crow[c] = hrow[c];
            crow[off_neigh + c] = s * iz;
        } else {
            const int k = c - a.H;
            float s = 0.f;
            for (int e = 0; e < a.n_et; ++e) s += seg_gather(a.xn[e], 4, a.part[e] + a.Hp, a.pw, r0[e], r1[e], nd, k);
            a.x[3 * nd + k] += s * iz;
        }
    }
    for (int c = a.H + lane; c < off_neigh; c += 32) crow[c] = 0.f;
}
__global__ void __launch_bounds__(256) egnn_node_prep_warp_kernel(const EgnnNodePrep a, int off_neigh) {
    node_prep_warp_body(a, off_neigh, blockIdx.x);
}
// both updated node types in one launch (blocks [0, blocks0) = ligand atoms, the rest = keypoints): each of these kernels is
// ~7 us of latency, not of work
struct EgnnNodePrepPair { EgnnNodePrep a[2]; };
__global__ void __launch_bounds__(256) egnn_node_prep_pair_kernel(const __grid_constant__ EgnnNodePrepPair p, int off_neigh, int blocks0) {
    if ((int)blockIdx.x < blocks0) node_prep_warp_body(p.a[0], off_neigh, blockIdx.x);
    else node_prep_warp_body(p.a[1], off_neigh, (int)blockIdx.x - blocks0);
}

}  // namespace kpd

using namespace kpd;

struct EgnnLayerW {
    const float* WpreT[2]; const float* bpre[2];
    const float* w1c[4][2]; const float* W2T[4][2]; const float* b2[4][2]; const float* W2lo[4][2];
    const float* watt[4]; const float* batt[4]; const float* w3c[4];
    const float* Wn1T[2]; const float* bn1[2]; const float* Wn2T[2]; const float* bn2[2];
    const float* lnw[2]; const float* lnb[2];
    // tensor-core modes (kpd_egnn_attach_tc): packed k-step slabs, [nsplit - 1] = bf16 | bf16x3
    struct Tc { const void* WpreP[2]; const uint4* W2P[4][2]; const void* Wn1P[2]; const void* Wn2P[2]; } tc[2];
};

struct kpd_egnn_model {
    kpd_egnn_config cfg;
    int H, Hp, nmain, nlo, lda, pw, F, F2p, Fp, C, C2p, hid, hidp;
    int n_et, n_upd, nslot[2];
    const float* lig_enc[4]; const float* rec_enc[4]; const float* dec[4];
    std::vector<EgnnLayerW> layers;
    size_t edge_smem, edge_smem_ws[2];      // edge_smem_ws[nsplit - 1]
    int mode;          // 0 = fp32 SIMT, 1 = bf16 tcgen05 (plain operands), 2 = bf16x3 tcgen05 (split operands, fp32-grade)
    bool tc_ready[2];  // [nsplit - 1]
};

struct EgnnWs {
    float *h[2], *xc[2], *P[2], *hn[4], *xn[4], *part[4], *cat[2], *tmp1[2], *y[2], *t1, *t2;
};

static int egnn_ntiles(int cap) { return cdiv(cap > 0 ? cap : 1, TE) + 1; }

static EgnnWs egnn_carve(const kpd_egnn_model* m, const kpd_batch* b, const int caps[4], void* ws, int64_t* bytes) {
    EgnnWs w;
    Carver c(ws);
    const int N[2] = {b->n_lig, b->n_kp};
    const int maxN = N[0] > N[1] ? N[0] : N[1];
    for (int nt = 0; nt < 2; ++nt) {
        w.h[nt] = c.take<float>((int64_t)N[nt] * m->Hp);
        w.xc[nt] = c.take<float>((int64_t)N[nt] * 3);
        w.P[nt] = c.take<float>((int64_t)N[nt] * m->nslot[nt] * m->Hp);
    }
    const int dstN[4] = {N[0], N[0], N[1], N[1]};   // ll, kl -> lig ; lk, kk -> kp
    for (int e = 0; e < 4; ++e) {
        w.hn[e] = c.take<float>((int64_t)dstN[e] * m->Hp);
        w.xn[e] = c.take<float>((int64_t)dstN[e] * 4);
        w.part[e] = c.take<float>((int64_t)egnn_ntiles(caps[e]) * 2 * m->pw);
    }
    for (int nt = 0; nt < 2; ++nt) {
        w.cat[nt] = c.take<float>((int64_t)N[nt] * (m->Hp + m->H + 4));
        w.tmp1[nt] = c.take<float>((int64_t)N[nt] * m->Hp);
        w.y[nt] = c.take<float>((int64_t)N[nt] * m->Hp);
    }
    const int t1w = 64 > m->C2p ? 64 : m->C2p;
    w.t1 = c.take<float>((int64_t)maxN * t1w);
    w.t2 = c.take<float>((int64_t)N[0] * m->F2p);
    if (bytes) *bytes = c.bytes();
    return w;
}

extern "C" int kpd_egnn_create(const kpd_egnn_config* cfg, const float* blob, const int64_t* off,
                               int32_t n_off, kpd_egnn_model** out) {
    KPD_REQUIRE(cfg && blob && off && out, "kpd_egnn_create: null argument");
    KPD_REQUIRE((reinterpret_cast<uintptr_t>(blob) & 15) == 0, "kpd_egnn_create: blob must be 16-byte aligned");
    auto* m = new kpd_egnn_model();
    m->cfg = *cfg;
    m->hid = cfg->hidden_nf;
    m->hidp = (m->hid + 3) & ~3;
    m->H = cfg->hidden_nf + 1;
    m->Hp = (m->H + 3) & ~3;
    if (m->H > KPD_MAX_HIDDEN) { delete m; KPD_REQUIRE(false, "kpd_egnn_create: hidden_nf+1=%d > %d unsupported", cfg->hidden_nf + 1, KPD_MAX_HIDDEN); }
    m->nmain = (m->H < 256 ? m->H : 256) & ~3;
    m->nlo = m->H - m->nmain;
    if (m->nlo > 3) { const int Hh = m->H, lo = m->nlo; delete m; KPD_REQUIRE(false, "kpd_egnn_create: hidden width %d leaves %d leftover columns (>3)", Hh, lo); }
    m->lda = tile_ld(m->Hp);
    m->pw = m->Hp + 4;
    m->F = cfg->atom_nf; m->Fp = (m->F + 3) & ~3; m->F2p = (2 * m->F + 3) & ~3;
    m->C = cfg->rec_nf; m->C2p = (2 * m->C + 3) & ~3;
    m->n_et = cfg->update_kp_feat ? 4 : 2;
    m->n_upd = cfg->update_kp_feat ? 2 : 1;
    m->nslot[0] = cfg->update_kp_feat ? 8 : 6;
    m->nslot[1] = cfg->update_kp_feat ? 8 : 2;
    const int per_layer = 4 + m->n_et * 11 + m->n_upd * 6;
    const int expect = 12 + cfg->n_layers * per_layer;
    if (n_off != expect) { delete m; KPD_REQUIRE(false, "kpd_egnn_create: expected %d offsets, got %d", expect, n_off); }
    int i = 0;
    auto P = [&](void) -> const float* { int64_t o = off[i++]; return o < 0 ? nullptr : blob + o; };
    for (int k = 0; k < 4; ++k) m->lig_enc[k] = P();
    for (int k = 0; k < 4; ++k) m->rec_enc[k] = P();
    for (int k = 0; k < 4; ++k) m->dec[k] = P();
    m->layers.resize(cfg->n_layers);
    for (int l = 0; l < cfg->n_layers; ++l) {
        EgnnLayerW& L = m->layers[l];
        for (int nt = 0; nt < 2; ++nt) { L.WpreT[nt] = P(); L.bpre[nt] = P(); }
        for (int e = 0; e < m->n_et; ++e) {
            for (int br = 0; br < 2; ++br) { L.w1c[e][br] = P(); L.W2T[e][br] = P(); L.b2[e][br] = P(); L.W2lo[e][br] = P(); }
            L.watt[e] = P(); L.batt[e] = P(); L.w3c[e] = P();
        }
        for (int nt = 0; nt < m->n_upd; ++nt) {
            L.Wn1T[nt] = P(); L.bn1[nt] = P(); L.Wn2T[nt] = P(); L.bn2[nt] = P(); L.lnw[nt] = P(); L.lnb[nt] = P();
        }
    }
    m->edge_smem = sizeof(float) * ((size_t)TE * m->lda + BS_FLOATS + TE * 4 + TE * 3 + TE * 3 + TE) + sizeof(int) * 2 * TE;
    cudaError_t e = cudaFuncSetAttribute(egnn_edge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->edge_smem);
    if (e != cudaSuccess) { const size_t sm = m->edge_smem; delete m; KPD_REQUIRE(false, "kpd_egnn_create: cannot set %zu B shared memory: %s", sm, cudaGetErrorString(e)); }
    m->mode = 0;
    m->tc_ready[0] = m->tc_ready[1] = false;
    m->edge_smem_ws[0] = egws::smem_bytes<1>(2 * cdiv(m->H, 16));
    m->edge_smem_ws[1] = egws::smem_bytes<2>(2 * cdiv(m->H, 16));
    *out = m;
    return 0;
}

extern "C" void kpd_egnn_destroy(kpd_egnn_model* m) { delete m; }

// Tensor-core modes (nsplit = 1: "bf16", plain bf16 operands; nsplit = 2: "bf16x3", split (hi, lo) bf16 operands,
// fp32-grade): tc_blob holds, per layer, the packed (pack.pack_tc_weight(split = nsplit == 2)) weights  Wpre[lig],
// Wpre[kp]; per edge type W2 of edge_mlp and coord_mlp (rows [0, nmain)); per updated node type node_mlp.0 and
// node_mlp.2 -- pack.pack_egnn_tc.  The two packs are kept side by side: set_mode switches between them.
extern "C" int kpd_egnn_attach_tc(kpd_egnn_model* m, const void* tc_blob, const int64_t* byte_offsets, int32_t n, int32_t nsplit) {
    KPD_REQUIRE(m && tc_blob && byte_offsets, "kpd_egnn_attach_tc: null argument");
    KPD_REQUIRE(nsplit == 1 || nsplit == 2, "kpd_egnn_attach_tc: nsplit must be 1 (bf16) or 2 (bf16x3)");
    const int per_layer = 2 + m->n_et * 2 + m->n_upd * 2;
    KPD_REQUIRE(n == m->cfg.n_layers * per_layer, "kpd_egnn_attach_tc: expected %d offsets, got %d", m->cfg.n_layers * per_layer, n);
    KPD_REQUIRE((reinterpret_cast<uintptr_t>(tc_blob) & 127) == 0, "kpd_egnn_attach_tc: blob must be 128-byte aligned");
    KPD_REQUIRE(m->nmain % 8 == 0 && m->H <= 257, "kpd_egnn_attach_tc: hidden width %d unsupported by the tensor-core tiles", m->H);
    const size_t smem = m->edge_smem_ws[nsplit - 1];
    KPD_REQUIRE(smem <= 227 * 1024, "kpd_egnn_attach_tc: tile needs %zu B of shared memory", smem);
    const char* base = static_cast<const char*>(tc_blob);
    int i = 0;
    auto P = [&](void) -> const void* { return base + byte_offsets[i++]; };
    for (int l = 0; l < m->cfg.n_layers; ++l) {
        EgnnLayerW::Tc& T = m->layers[l].tc[nsplit - 1];
        for (int nt = 0; nt < 2; ++nt) T.WpreP[nt] = P();
        for (int e = 0; e < m->n_et; ++e)
            for (int br = 0; br < 2; ++br) T.W2P[e][br] = static_cast<const uint4*>(P());
        for (int nt = 0; nt < m->n_upd; ++nt) { T.Wn1P[nt] = P(); T.Wn2P[nt] = P(); }
    }
    cudaError_t e;
    if (nsplit == 1) {
        e = cudaFuncSetAttribute(egnn_edge_ws_kernel<257, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(egnn_edge_ws_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    } else {
        e = cudaFuncSetAttribute(egnn_edge_ws_kernel<257, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(egnn_edge_ws_kernel<0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    KPD_REQUIRE(e == cudaSuccess, "kpd_egnn_attach_tc: cannot set %zu B shared memory: %s", smem, cudaGetErrorString(e));
    m->tc_ready[nsplit - 1] = true;
    return 0;
}

// debug: read (and reset) the phase timers of the warp-specialised edge kernel (cycles summed over CTAs)
extern "C" int kpd_debug_eg_times(unsigned long long* out16) {
    KPD_REQUIRE(out16, "kpd_debug_eg_times: null argument");
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out16, g_eg_times, sizeof(unsigned long long) * 16);
    unsigned long long z[16] = {0};
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_eg_times, z, sizeof(z));
    KPD_REQUIRE(e == cudaSuccess, "kpd_debug_eg_times: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int kpd_egnn_set_mode(kpd_egnn_model* m, int32_t mode) {
    KPD_REQUIRE(m, "kpd_egnn_set_mode: null model");
    KPD_REQUIRE(mode >= 0 && mode <= 2, "kpd_egnn_set_mode: mode must be 0 (fp32 SIMT), 1 (bf16) or 2 (bf16x3 tensor cores)");
    KPD_REQUIRE(mode == 0 || (m->tc_ready[mode - 1] && m->tc_ready[1]),
                "kpd_egnn_set_mode: mode %d needs kpd_egnn_attach_tc(nsplit = 2)%s first", mode, mode == 1 ? " and (nsplit = 1)" : "");
    m->mode = mode;
    return 0;
}

extern "C" int kpd_egnn_dims(const kpd_egnn_model* m, int* rec_nf, int* hidden_nf) {
    KPD_REQUIRE(m, "kpd_egnn_dims: null model");
    *rec_nf = m->C; *hidden_nf = m->hid;
    return 0;
}

extern "C" int64_t kpd_egnn_workspace_bytes(const kpd_egnn_model* m, const kpd_batch* batch, int32_t cap_ll,
                                            int32_t cap_kl, int32_t cap_kk) {
    const int caps[4] = {cap_ll, cap_kl, cap_kl, cap_kk};
    int64_t bytes = 0;
    egnn_carve(m, batch, caps, nullptr, &bytes);
    return bytes;
}

static int egnn_encode_kp_impl(const kpd_egnn_model* m, const float* h_kp, int n_kp, float* out, int ldo,
                               float* t1, cudaStream_t st) {
    if (m->cfg.has_rec_encoder) {
        // Sequential(Linear(C,2C), SiLU, Linear(2C,hid), SiLU)   (models/dynamics.py:326-332)
        KPD_TRY(launch_linear(h_kp, m->C, m->rec_enc[0], m->C2p, m->rec_enc[1], nullptr, 0, t1, m->C2p, n_kp, m->C, 2 * m->C, 1, st));
        KPD_TRY(launch_linear(t1, m->C2p, m->rec_enc[2], m->hidp, m->rec_enc[3], nullptr, 0, out, ldo, n_kp, 2 * m->C, m->hid, 1, st));
    } else {
        KPD_TRY(launch_copy_rows(h_kp, m->C, out, ldo, n_kp, m->hid, st));   // nn.Identity (:333-334)
    }
    return 0;
}

extern "C" int kpd_egnn_encode_kp(const kpd_egnn_model* m, const float* h_kp, int32_t n_kp, float* out,
                                  void* workspace, void* stream) {
    KPD_REQUIRE(m && h_kp && out && workspace, "kpd_egnn_encode_kp: null argument");
    return egnn_encode_kp_impl(m, h_kp, n_kp, out, m->hid, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream));
}

extern "C" int kpd_egnn_forward(const kpd_egnn_model* m, const kpd_batch* b, const float* h_lig,
                                const float* x_lig, const float* h_kp, const float* x_kp,
                                const float* kp_feat_enc, const float* t_ptr, int32_t t_per_complex,
                                const kpd_csr* ll, const kpd_csr* kl, const kpd_csr* lk, const kpd_csr* kk,
                                float* eps_h, float* eps_x, void* workspace, void* stream) {
    KPD_REQUIRE(m && b && h_lig && x_lig && x_kp && t_ptr && ll && kl && eps_h && eps_x && workspace,
                "kpd_egnn_forward: null argument");
    KPD_REQUIRE(h_kp || kp_feat_enc, "kpd_egnn_forward: need h_kp or kp_feat_enc");
    const bool ukp = m->cfg.update_kp_feat != 0;
    KPD_REQUIRE(!ukp || (lk && kk), "kpd_egnn_forward: update_kp_feat needs lk and kk graphs");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const kpd_csr* G[4] = {ll, kl, lk, kk};
    const int caps[4] = {ll->cap, kl->cap, ukp ? lk->cap : 0, ukp ? kk->cap : 0};
    EgnnWs w = egnn_carve(m, b, caps, workspace, nullptr);
    const int N[2] = {b->n_lig, b->n_kp};
    const int H = m->H, Hp = m->Hp, hid = m->hid;

    // ---- encoders + time channel (models/dynamics.py:355-363)
    KPD_TRY(launch_linear(h_lig, m->F, m->lig_enc[0], 64, m->lig_enc[1], nullptr, 0, w.t1, 64, N[0], m->F, 64, 1, st));
    KPD_TRY(launch_linear(w.t1, 64, m->lig_enc[2], m->hidp, m->lig_enc[3], nullptr, 0, w.h[0], Hp, N[0], 64, hid, 1, st));
    if (kp_feat_enc) KPD_TRY(launch_copy_rows(kp_feat_enc, hid, w.h[1], Hp, N[1], hid, st));
    else KPD_TRY(egnn_encode_kp_impl(m, h_kp, N[1], w.h[1], Hp, w.t1, st));
    KPD_TRY(launch_set_time_col(w.h[0], Hp, hid, N[0], t_ptr, b->lig_batch, t_per_complex, st));
    KPD_TRY(launch_set_time_col(w.h[1], Hp, hid, N[1], t_ptr, b->kp_batch, t_per_complex, st));
    KPD_TRY(launch_copy_rows(x_lig, 3, w.xc[0], 3, N[0], 3, st));
    KPD_TRY(launch_copy_rows(x_kp, 3, w.xc[1], 3, N[1], 3, st));

    // role tables: {src ntype, src role, dst ntype, dst role} per etype (ll, kl, lk, kk)
    const int src_nt[4] = {0, 1, 0, 1}, dst_nt[4] = {0, 0, 1, 1};
    int role_s[4], role_d[4];
    if (ukp) { role_s[0] = 0; role_d[0] = 1; role_s[1] = 0; role_d[1] = 3; role_s[2] = 2; role_d[2] = 3; role_s[3] = 1; role_d[3] = 2; }
    else     { role_s[0] = 0; role_d[0] = 1; role_s[1] = 0; role_d[1] = 2; role_s[2] = role_d[2] = role_s[3] = role_d[3] = 0; }

    int max_tiles = 1;
    for (int e = 0; e < m->n_et; ++e) { int t = cdiv(caps[e] > 0 ? caps[e] : 1, TE); if (t > max_tiles) max_tiles = t; }

    for (int l = 0; l < m->cfg.n_layers; ++l) {
        const EgnnLayerW& W = m->layers[l];
        // edge kernel: the mode's own pack (nsplit = mode).  Node GEMMs: split operands in both tensor-core modes --
        // tc_linear<1> takes 128 rows per CTA, half the CTAs of tc_linear<2>, and at a sampling batch's node counts
        // that left the GPU idle (egnn_20kp 72 -> 49 ligands/s on B200 with nsplit = 1 here, DESIGN.md 4.1)
        const EgnnLayerW::Tc& T = W.tc[m->mode == 1 ? 0 : 1];
        const EgnnLayerW::Tc& TN = W.tc[1];
        prof_begin(PROF_EGNN_PRE, st);
        if (m->mode != 0) {       // both node types in one launch
            TcLinBatch TB;
            memset(&TB, 0, sizeof(TB));
            for (int nt = 0; nt < 2; ++nt) {
                const int ncol = m->nslot[nt] * Hp;
                TB.p[nt] = tc_problem(w.h[nt], Hp, TN.WpreP[nt], W.bpre[nt], nullptr, 0, w.P[nt], ncol, N[nt], H, ncol, 0);
            }
            KPD_TRY(launch_tc_batch(TB, 2, 2, st));
        } else {
            for (int nt = 0; nt < 2; ++nt) {
                const int ncol = m->nslot[nt] * Hp;
                KPD_TRY(launch_linear(w.h[nt], Hp, W.WpreT[nt], ncol, W.bpre[nt], nullptr, 0, w.P[nt], ncol, N[nt], H, ncol, 0, st));
            }
        }
        prof_end(PROF_EGNN_PRE, st);
        EgnnEdgeLaunch L;
        memset(&L, 0, sizeof(L));
        L.H = H; L.Hp = Hp; L.nmain = m->nmain; L.nlo = m->nlo; L.lda = m->lda; L.pw = m->pw;
        L.use_tanh = m->cfg.use_tanh; L.coords_range = m->cfg.coords_range;
        for (int e = 0; e < m->n_et; ++e) {
            EgnnEtypeArgs& a = L.e[e];
            a.rowptr = G[e]->rowptr; a.src = G[e]->src; a.dst = G[e]->dst; a.n_dst = G[e]->n_dst; a.cap = G[e]->cap;
            a.Ps = w.P[src_nt[e]]; a.ldps = m->nslot[src_nt[e]] * Hp; a.slot_s = 2 * role_s[e];
            a.Pd = w.P[dst_nt[e]]; a.ldpd = m->nslot[dst_nt[e]] * Hp; a.slot_d = 2 * role_d[e];
            a.xs = w.xc[src_nt[e]]; a.xd = w.xc[dst_nt[e]];
            for (int br = 0; br < 2; ++br) { a.w1c[br] = W.w1c[e][br]; a.W2T[br] = W.W2T[e][br]; a.b2[br] = W.b2[e][br]; a.W2lo[br] = W.W2lo[e][br]; }
            a.watt = W.watt[e]; a.batt = W.batt[e]; a.w3c = W.w3c[e];
            a.hn = w.hn[e]; a.xn = w.xn[e]; a.part = w.part[e];
        }
        prof_begin(PROF_EGNN_EDGE, st);
        if (m->mode != 0) {
            EgnnWsLaunch WL;
            memset(&WL, 0, sizeof(WL));
            WL.L = L;
            WL.kch = 2 * cdiv(H, 16);
            for (int e = 0; e < m->n_et; ++e)
                for (int br = 0; br < 2; ++br) WL.t[e].W2P[br] = T.W2P[e][br];
            for (int e = 0; e < 4; ++e) WL.tile_off[e + 1] = WL.tile_off[e] + (e < m->n_et ? cdiv(caps[e] > 0 ? caps[e] : 1, egws::R) : 0);
            // (the constants the kernel derives from HS = 257 are exactly what this function passes for H = 257)
            const dim3 grid(WL.tile_off[4]);
            const size_t smem = m->edge_smem_ws[m->mode - 1];
            if (m->mode == 1) {
                if (H == 257) egnn_edge_ws_kernel<257, 1><<<grid, egws::NT, smem, st>>>(WL);
                else egnn_edge_ws_kernel<0, 1><<<grid, egws::NT, smem, st>>>(WL);
            } else {
                if (H == 257) egnn_edge_ws_kernel<257, 2><<<grid, egws::NT, smem, st>>>(WL);
                else egnn_edge_ws_kernel<0, 2><<<grid, egws::NT, smem, st>>>(WL);
            }
            KPD_TRY(check_launch("egnn_edge_ws_kernel"));
        } else {
            egnn_edge_kernel<<<dim3(max_tiles, m->n_et), NT, m->edge_smem, st>>>(L);
            KPD_TRY(check_launch("egnn_edge_kernel"));
        }
        prof_end(PROF_EGNN_EDGE, st);
        prof_begin(PROF_EGNN_NODE, st);

        // tensor-core mode: h_neigh starts at the 4-aligned column Hp of the cat row (zero gap [H, Hp))
        const int off_neigh = m->mode != 0 ? Hp : H;
        const int ldcat = (off_neigh + H + 3) & ~3;
        EgnnNodePrepPair NP;
        memset(&NP, 0, sizeof(NP));
        for (int nt = 0; nt < m->n_upd; ++nt) {
            EgnnNodePrep& a = NP.a[nt];
            a.n = N[nt]; a.H = H; a.Hp = Hp; a.pw = m->pw;
            a.ldcat = ldcat;
            a.h = w.h[nt]; a.cat = w.cat[nt]; a.x = w.xc[nt];
            a.n_et = 2;
            for (int k = 0; k < 2; ++k) {
                const int e = nt * 2 + k;   // lig <- (ll, kl); kp <- (lk, kk)
                a.rowptr[k] = G[e]->rowptr; a.hn[k] = w.hn[e]; a.xn[k] = w.xn[e]; a.part[k] = w.part[e];
            }
            a.z_mode = !m->cfg.z_effective ? 0 : (m->cfg.message_norm == 0.0f ? 2 : 1);
            a.z_const = m->cfg.message_norm;
            a.node_batch = nt == 0 ? b->lig_batch : b->kp_batch;
            a.ptr = nt == 0 ? b->lig_ptr : b->kp_ptr;
            if (a.n > 0 && m->mode == 0) {
                egnn_node_prep_kernel<<<a.n, 128, 0, st>>>(a);
                KPD_TRY(check_launch("egnn_node_prep_kernel"));
            }
        }
        if (m->mode != 0) {
            const int blocks0 = cdiv(NP.a[0].n > 0 ? NP.a[0].n : 0, 8), blocks1 = m->n_upd > 1 ? cdiv(NP.a[1].n > 0 ? NP.a[1].n : 0, 8) : 0;
            if (blocks0 + blocks1 > 0) {
                egnn_node_prep_pair_kernel<<<blocks0 + blocks1, 256, 0, st>>>(NP, off_neigh, blocks0);
                KPD_TRY(check_launch("egnn_node_prep_pair_kernel"));
            }
        }
        // node_mlp = Linear(2H,H), SiLU, Linear(H,H); residual; LayerNorm  (:202-205)
        if (m->mode != 0) {       // all updated node types in one launch per Linear
            TcLinBatch T1, T2;
            memset(&T1, 0, sizeof(T1));
            memset(&T2, 0, sizeof(T2));
            for (int nt = 0; nt < m->n_upd; ++nt) {
                T1.p[nt] = tc_problem(w.cat[nt], ldcat, TN.Wn1P[nt], W.bn1[nt], nullptr, 0, w.tmp1[nt], Hp, N[nt], off_neigh + H, H, 1);
                T2.p[nt] = tc_problem(w.tmp1[nt], Hp, TN.Wn2P[nt], W.bn2[nt], w.h[nt], Hp, w.y[nt], Hp, N[nt], H, H, 0);
            }
            KPD_TRY(launch_tc_batch(T1, m->n_upd, 2, st));
            KPD_TRY(launch_tc_batch(T2, m->n_upd, 2, st));
        }
        for (int nt = 0; nt < m->n_upd; ++nt) {
            if (m->mode == 0) {
                KPD_TRY(launch_linear(w.cat[nt], ldcat, W.Wn1T[nt], Hp, W.bn1[nt], nullptr, 0, w.tmp1[nt], Hp, N[nt], 2 * H, H, 1, st));
                KPD_TRY(launch_linear(w.tmp1[nt], Hp, W.Wn2T[nt], Hp, W.bn2[nt], w.h[nt], Hp, w.y[nt], Hp, N[nt], H, H, 0, st));
            }
            if (m->cfg.norm && m->mode != 0) continue;      // (one launch for all node types below)
            if (m->cfg.norm) KPD_TRY(launch_layernorm(w.y[nt], Hp, w.h[nt], Hp, N[nt], H, W.lnw[nt], W.lnb[nt], st));
            else KPD_TRY(launch_copy_rows(w.y[nt], Hp, w.h[nt], Hp, N[nt], H, st));
        }
        if (m->cfg.norm && m->mode != 0) {
            const bool two = m->n_upd > 1;
            KPD_TRY(launch_layernorm_pair(w.y[0], w.h[0], N[0], W.lnw[0], W.lnb[0], two ? w.y[1] : nullptr, two ? w.h[1] : nullptr,
                                          two ? N[1] : 0, two ? W.lnw[1] : nullptr, two ? W.lnb[1] : nullptr, Hp, Hp, H, st));
        }
        prof_end(PROF_EGNN_NODE, st);
    }
    // ---- decoder on h[:, :-1] and eps_x (models/dynamics.py:376-381)
    KPD_TRY(launch_linear(w.h[0], Hp, m->dec[0], m->F2p, m->dec[1], nullptr, 0, w.t2, m->F2p, N[0], hid, 2 * m->F, 1, st));
    KPD_TRY(launch_linear(w.t2, m->F2p, m->dec[2], m->Fp, m->dec[3], nullptr, 0, eps_h, m->F, N[0], 2 * m->F, m->F, 0, st));
    KPD_TRY(launch_sub(w.xc[0], x_lig, eps_x, 3 * N[0], st));
    return 0;
}
