// tcgen05 GEMM for node-level rows, and the unit under test for the tensor-core primitives of tc.cuh:
//     Y[m, 0:N] = act( X[m, 0:K] @ W^T + bias ) (+R)
//   X fp32 row-major, staged into shared memory as the bf16 UMMA A operand; W pre-packed bf16 "k-step slabs"
//   (keypoint_diffusion_b200/pack.py: pack_tc_weight), streamed through a cp.async.bulk ring (as deep as shared memory
//   allows beside the A tile); the A tile is staged in ONE round trip to L2 (9 16-byte-pair items per lane in flight);
//   interior 64-column epilogue chunks take a lean path (every global load before the TMEM wait); fp32 accumulation in
//   TMEM, fp32 output.  NS = 1: plain bf16 operands, 128 rows per CTA.  NS = 2 ("bf16x3"): 64 rows per CTA, the
//   (hi, lo) bf16 rows stacked into one 128-row operand and two MMAs per k-step (W_hi, W_lo), which together give
//   all four hi/lo products -- fp32-grade results on the tensor cores (ws_common.cuh).
// blockIdx.y selects a 256-column block of the output (UMMA N <= 256).
#include "common.cuh"
#include "ws_common.cuh"
#include "tc_gemm.cuh"
#include <string.h>

namespace kpd {

// Weight ring: as many 16 KB (bf16x3) stages as fit beside the A tile, at most TCG_MAX_STAGES.  The ring is latency-bound --
// a slab is re-requested when its MMAs have completed and lands ~1500 cycles later --, so with four stages a k-step took
// (256 + 1500) / 4 = 440 cycles against 256 of tensor-core time.
#ifndef KPD_TCG_MAX_STAGES
#define KPD_TCG_MAX_STAGES 8
#endif
constexpr int TCG_MAX_STAGES = KPD_TCG_MAX_STAGES;
#ifndef KPD_TCG_EW
#define KPD_TCG_EW 8
#endif
constexpr int TCG_EW = KPD_TCG_EW;    // SIMT warps: stage A + epilogues (TCG_EW / 4 per TMEM lane quarter)
constexpr int TCG_CS = TCG_EW / 4;    // ... which take every TCG_CS-th column chunk of a block
constexpr int TCG_THREADS = 32 * TCG_EW + 64;      // + warp TCG_EW: MMA issuer | warp TCG_EW + 1: weight producer

// phase timers of tools/tc_linear_bench.py (variant builds with -DKPD_TCG_TIMERS only): cycles summed over CTAs, thread 0 of
// the SIMT warps [0] set-up, [1] A staged, [2] first accumulator waited for, [3] remaining blocks, [4] teardown, [5] CTAs;
// MMA warp [8] waiting for A, [9] first slab, [10] issue loop
#ifdef KPD_TCG_TIMERS
__device__ unsigned long long g_tcg_times[16];
#define TCG_T(var) const long long var = clock64()
#define TCG_ACC(slot, a, b) atomicAdd(&g_tcg_times[slot], (unsigned long long)((b) - (a)))
#else
#define TCG_T(var)
#define TCG_ACC(slot, a, b)
#endif

template <int NS>
__global__ void __launch_bounds__(TCG_THREADS, 1) tc_linear_kernel(const __grid_constant__ TcLinBatch B) {
    using C = ws::Cfg<128 / NS, NS>;
    const TcLinProblem& P = B.p[blockIdx.z];
    const int M = P.M, K = P.K, N = P.N;
    const int m0 = blockIdx.x * C::R;
    const int nblocks = (N + 255) / 256;
    const int blk0 = blockIdx.y * B.bpc;
    if (m0 >= M || blk0 >= nblocks) return;
    const int nb_cta = min(B.bpc, nblocks - blk0);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int ksteps = (K + 15) / 16;
    unsigned char* a_s = smem_raw;                     // [2 * ksteps] k-chunks of C::KCS bytes
    unsigned char* b_s = a_s + (((size_t)2 * ((B.kmax + 15) / 16) * C::KCS + 127) & ~(size_t)127);   // [STAGES] ring
    const int slab_stride = NS * 2 * (B.NBmax / 8) * 128;
    const uint32_t stages = (uint32_t)B.stages;
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_s + (size_t)stages * slab_stride);
    uint64_t* full = bars;
    uint64_t* empty = bars + TCG_MAX_STAGES;
    uint64_t* a_ready = bars + 2 * TCG_MAX_STAGES;
    uint64_t* acc_done = a_ready + 1;                  // [2]
    uint64_t* acc_free = acc_done + 2;                 // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    TCG_T(t_begin);

    if (tid == 0) {
        for (int i = 0; i < TCG_MAX_STAGES; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
        tc::mbar_init(a_ready, TCG_EW);
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&acc_done[i], 1); tc::mbar_init(&acc_free[i], TCG_EW); }
        tc::fence_barrier_init();
    }
    if (warp == TCG_EW) { tc::tmem_alloc(tmem_slot, 512); tc::tmem_relinquish(); }     // two 256-column accumulators
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    TCG_T(t_setup);

    auto block_NB = [&](int blk) { const int r = N - 256 * blk; return r > 256 ? 256 : (r + 15) & ~15; };
    // all blocks before the last one are full (256 rows): their slabs are NS * 2 * 32 * 128 B per k-step
    auto block_W = [&](int blk) { return P.Wp + (size_t)blk * ksteps * (NS * 2 * 32 * 128 / 16); };

    if (warp == TCG_EW + 1) {
        // ---- weight producer: the k-step slabs of this CTA's column blocks through the ring
        if (lane == 0) {
            uint32_t it = 0;
            for (int bi = 0; bi < nb_cta; ++bi) {
                const int NB = block_NB(blk0 + bi);
                const uint32_t slab_bytes = NS * 2 * (NB / 8) * 128;
                const uint4* Wb = block_W(blk0 + bi);
                for (int j = 0; j < ksteps; ++j, ++it) {
                    const uint32_t st = it % stages;
                    if (it >= stages) tc::mbar_wait(&empty[st], ((it / stages) - 1) & 1);
                    tc::mbar_arrive_expect_tx(&full[st], slab_bytes);
                    tc::bulk_g2s(b_s + (size_t)st * slab_stride, Wb + (size_t)j * (slab_bytes / 16), slab_bytes, &full[st]);
                }
            }
        }
    } else if (warp == TCG_EW) {
        // ---- MMA issuer: accumulator bi % 2, so that the epilogue of one block overlaps the MMAs of the next.  The whole
        //      (converged) warp runs the loop, one elected lane executes the tcgen05 instructions (tc::elect_one())
        {
            tc::mbar_wait(a_ready, 0);
            tc::fence_after_sync();
            TCG_T(m_a);
            [[maybe_unused]] long long m_first = 0;
            uint32_t it = 0;
            for (int bi = 0; bi < nb_cta; ++bi) {
                const int buf = bi & 1, NB = block_NB(blk0 + bi);
                const uint32_t idesc = tc::make_idesc_bf16(128, NB);
                const uint32_t b_k = (NB / 8) * 128, slab1 = 2 * b_k;
                if (bi >= 2) { tc::mbar_wait(&acc_free[buf], ((bi >> 1) - 1) & 1); tc::fence_after_sync(); }
                for (int j = 0; j < ksteps; ++j, ++it) {
                    const uint32_t st = it % stages;
                    tc::mbar_wait(&full[st], (it / stages) & 1);
                    tc::fence_after_sync();
#ifdef KPD_TCG_TIMERS
                    if (it == 0) m_first = clock64();
#endif
                    const uint64_t adesc = tc::make_smem_desc(tc::smem_u32(a_s + (size_t)2 * j * C::KCS), C::KCS, 128);
                    const uint32_t bs = tc::smem_u32(b_s + (size_t)st * slab_stride);
                    const uint64_t b0 = tc::make_smem_desc(bs, b_k, 128), b1 = tc::make_smem_desc(bs + slab1, b_k, 128);
                    if (tc::elect_one()) {
                        tc::mma_bf16_ss(tmem_base + 256 * buf, adesc, b0, idesc, j > 0 ? 1u : 0u);
                        if (NS == 2) tc::mma_bf16_ss(tmem_base + 256 * buf, adesc, b1, idesc, 1u);
                        tc::mma_commit(&empty[st]);
                    }
                }
                if (tc::elect_one()) tc::mma_commit(&acc_done[buf]);
            }
#ifdef KPD_TCG_TIMERS
            if (lane == 0) { const long long m_end = clock64(); TCG_ACC(8, t_setup, m_a); TCG_ACC(9, m_a, m_first); TCG_ACC(10, m_first, m_end); }
#endif
        }
    } else {
        // ---- stage the A tile once: each warp owns R/4 consecutive rows; (row, 8-element k-chunk) items are dealt to
        //      the lanes in order (coalesced 32-byte reads), four items per lane in flight
        {
            // NI items per lane and round: the 8 rows x 34 chunks of a K = 257 tile (272 items per warp) are ONE round trip to
            // L2, K = 517 two.  A chunk is read as two 16-byte loads wherever the row (ldx floats, a multiple of 4) has them --
            // the columns beyond K are masked afterwards: they may hold anything -- so there is no scalar path.
            const int nch = 2 * ksteps;
            constexpr int RPW = C::R / TCG_EW;
            constexpr int NI = 9;
            const int items = RPW * nch;
            for (int base = 0; base < items; base += 32 * NI) {
                float4 va[NI], vb[NI];
                int ri = (base + lane) / nch, c = (base + lane) - ri * nch;
                int ri0 = ri, c0 = c;
#pragma unroll
                for (int u = 0; u < NI; ++u) {
                    const int i = base + 32 * u + lane;
                    const int gm = m0 + warp * RPW + ri;
                    va[u] = vb[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (i < items && gm < M) {
                        const float* xr = P.X + (size_t)gm * P.ldx + 8 * c;
                        if (8 * c + 4 <= P.ldx && 8 * c < K) va[u] = __ldg(reinterpret_cast<const float4*>(xr));
                        if (8 * c + 8 <= P.ldx && 8 * c + 4 < K) vb[u] = __ldg(reinterpret_cast<const float4*>(xr + 4));
                    }
                    c += 32;
                    while (c >= nch) { c -= nch; ++ri; }
                }
                ri = ri0; c = c0;
#pragma unroll
                for (int u = 0; u < NI; ++u) {
                    const int i = base + 32 * u + lane;
                    if (i < items) {
                        float v[8] = {va[u].x, va[u].y, va[u].z, va[u].w, vb[u].x, vb[u].y, vb[u].z, vb[u].w};
                        if (8 * c + 8 > K) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) v[q] = 8 * c + q < K ? v[q] : 0.0f;
                        }
                        uint4 hi, lo;
                        ws::split8(v, hi, lo);
                        const uint32_t off = (uint32_t)(c * C::KCS) + ws::row_off<C>(warp * RPW + ri);
                        *reinterpret_cast<uint4*>(a_s + off) = hi;
                        if (NS == 2) *reinterpret_cast<uint4*>(a_s + off + 256) = lo;
                    }
                    c += 32;
                    while (c >= nch) { c -= nch; ++ri; }
                }
            }
            tc::fence_proxy_async();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(a_ready);
        }
        TCG_T(t_staged);
        [[maybe_unused]] long long t_first = 0;
        // ---- epilogues
        const int q = warp & 3, chalf = warp >> 2;       // TMEM lane quarter; which 64-column chunks (c0 / 64 parity)
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        for (int bi = 0; bi < nb_cta; ++bi) {
            const int buf = bi & 1, blk = blk0 + bi, NB = block_NB(blk);
            tc::mbar_wait(&acc_done[buf], (bi >> 1) & 1);
            tc::fence_after_sync();
#ifdef KPD_TCG_TIMERS
            if (bi == 0) t_first = clock64();
#endif
            if (NS == 1) {          // thread r reads its accumulator row from TMEM
                const int gm = m0 + 32 * q + lane;
                for (int c0 = 32 * chalf; c0 < NB; c0 += 32 * TCG_CS) {
                    uint32_t v[32];
                    tc::tmem_ld_x32(lane_addr + 256 * buf + c0, v);
                    tc::tmem_ld_wait();
                    if (gm < M) {
#pragma unroll
                        for (int q = 0; q < 32; ++q) {
                            const int gn = blk * 256 + c0 + q;
                            if (c0 + q < NB && gn < N) {
                                float f = __uint_as_float(v[q]) + (P.bias ? P.bias[gn] : 0.0f);
                                if (P.act == 1) f = silu_f(f);
                                if (P.R) f += P.R[(size_t)gm * P.ldr + gn];
                                P.Y[(size_t)gm * P.ldy + gn] = f;
                            }
                        }
                    }
                }
            } else {                // lanes [32w, 32w+16) = hi rows, [32w+16, 32w+32) = lo rows of tile rows [16w, 16w+16)
                const int ra = 16 * q + (lane >> 2), cp = 2 * (lane & 3);
                const bool vec2 = (P.ldy & 1) == 0 && (!P.R || (P.ldr & 1) == 0);      // 8-byte accesses possible
                for (int c0 = 64 * chalf; c0 < NB; c0 += 64 * TCG_CS) {
                    uint32_t v0[32], v1[32];
                    tc::tmem_ld_16x256b_x8(lane_addr + 256 * buf + c0, v0);
                    tc::tmem_ld_16x256b_x8(lane_addr + (16u << 16) + 256 * buf + c0, v1);
                    // interior chunk (all 64 columns exist, 8-byte accesses possible): every global load of the chunk -- bias
                    // and both rows' residuals -- is issued before the TMEM wait, nothing is predicated per element.  (The
                    // general path below is ~1400 instructions per chunk and warp, three dependent L2 round trips.)
                    if (vec2 && blk * 256 + c0 + 64 <= N && (!P.bias || (reinterpret_cast<uintptr_t>(P.bias) & 7) == 0)) {
                        const int gn0 = blk * 256 + c0 + cp;
                        const int gma = m0 + ra, gmb = gma + 8;
                        float2 bz[8], rza[8], rzb[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            bz[i] = P.bias ? __ldg(reinterpret_cast<const float2*>(P.bias + gn0 + 8 * i)) : make_float2(0.f, 0.f);
                            rza[i] = rzb[i] = make_float2(0.f, 0.f);
                        }
                        if (P.R) {
                            const float* rpa = P.R + (size_t)gma * P.ldr + gn0;
                            const float* rpb = P.R + (size_t)gmb * P.ldr + gn0;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                if (gma < M) rza[i] = *reinterpret_cast<const float2*>(rpa + 8 * i);
                                if (gmb < M) rzb[i] = *reinterpret_cast<const float2*>(rpb + 8 * i);
                            }
                        }
                        tc::tmem_ld_wait();
                        float* ypa = P.Y + (size_t)gma * P.ldy + gn0;
                        float* ypb = P.Y + (size_t)gmb * P.ldy + gn0;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float2 fa, fb;
                            fa.x = __uint_as_float(v0[4 * i + 0]) + __uint_as_float(v1[4 * i + 0]) + bz[i].x;
                            fa.y = __uint_as_float(v0[4 * i + 1]) + __uint_as_float(v1[4 * i + 1]) + bz[i].y;
                            fb.x = __uint_as_float(v0[4 * i + 2]) + __uint_as_float(v1[4 * i + 2]) + bz[i].x;
                            fb.y = __uint_as_float(v0[4 * i + 3]) + __uint_as_float(v1[4 * i + 3]) + bz[i].y;
                            if (P.act == 1) { fa.x = ws::silu_acc(fa.x); fa.y = ws::silu_acc(fa.y); fb.x = ws::silu_acc(fb.x); fb.y = ws::silu_acc(fb.y); }
                            fa.x += rza[i].x; fa.y += rza[i].y; fb.x += rzb[i].x; fb.y += rzb[i].y;
                            if (gma < M) *reinterpret_cast<float2*>(ypa + 8 * i) = fa;
                            if (gmb < M) *reinterpret_cast<float2*>(ypb + 8 * i) = fb;
                        }
                        continue;
                    }
                    // bias of this lane's column pairs: independent loads, in flight with the TMEM reads
                    float2 bz[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int gn = blk * 256 + c0 + 8 * i + cp;
                        bz[i] = make_float2(0.f, 0.f);
                        if (P.bias && c0 + 8 * i < NB) {
                            if (gn < N) bz[i].x = __ldg(P.bias + gn);
                            if (gn + 1 < N) bz[i].y = __ldg(P.bias + gn + 1);
                        }
                    }
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int gm = m0 + ra + 8 * h;
                        if (gm < M) {
                            float2 f[8], rz[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const int gn = blk * 256 + c0 + 8 * i + cp;
                                rz[i] = make_float2(0.f, 0.f);
                                if (P.R && c0 + 8 * i < NB) {
                                    const float* rp = P.R + (size_t)gm * P.ldr + gn;
                                    if (vec2 && gn + 1 < N) rz[i] = *reinterpret_cast<const float2*>(rp);
                                    else { if (gn < N) rz[i].x = rp[0]; if (gn + 1 < N) rz[i].y = rp[1]; }
                                }
                            }
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                f[i].x = __uint_as_float(v0[4 * i + 2 * h]) + __uint_as_float(v1[4 * i + 2 * h]) + bz[i].x;
                                f[i].y = __uint_as_float(v0[4 * i + 2 * h + 1]) + __uint_as_float(v1[4 * i + 2 * h + 1]) + bz[i].y;
                                if (P.act == 1) { f[i].x = ws::silu_acc(f[i].x); f[i].y = ws::silu_acc(f[i].y); }
                                f[i].x += rz[i].x; f[i].y += rz[i].y;
                            }
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const int gn = blk * 256 + c0 + 8 * i + cp;
                                if (c0 + 8 * i < NB) {
                                    float* yp = P.Y + (size_t)gm * P.ldy + gn;
                                    if (vec2 && gn + 1 < N) *reinterpret_cast<float2*>(yp) = f[i];
                                    else { if (gn < N) yp[0] = f[i].x; if (gn + 1 < N) yp[1] = f[i].y; }
                                }
                            }
                        }
                    }
                }
            }
            tc::fence_before_sync();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&acc_free[buf]);
        }
#ifdef KPD_TCG_TIMERS
        if (tid == 0) {
            const long long t_end = clock64();
            TCG_ACC(0, t_begin, t_setup); TCG_ACC(1, t_setup, t_staged); TCG_ACC(2, t_staged, t_first); TCG_ACC(3, t_first, t_end); TCG_ACC(5, 0, 1);
        }
#endif
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == TCG_EW) tc::tmem_dealloc(tmem_base, 512);
}

template <int NS>
static size_t tc_linear_smem(int K, int NB, int stages) {
    using C = ws::Cfg<128 / NS, NS>;
    const int ksteps = (K + 15) / 16;
    return (((size_t)2 * ksteps * C::KCS + 127) & ~(size_t)127) + (size_t)stages * NS * 2 * (NB / 8) * 128 + (2 * TCG_MAX_STAGES + 5) * 8 + 16;
}

// Wp: packed by pack_tc_weight(W[N,K], split = (nsplit == 2)) -> for each 256-row block nb: [ksteps][hi(, lo)][2][NB/8][8][8]
// bf16, NB = rows of the block rounded up to 16 (all blocks but the last have NB = 256).
// X rows must be 16-byte aligned (ldx % 4 == 0).  Up to two problems per launch (blockIdx.z).
template <int NS>
static int launch_tc_batch_ns(TcLinBatch& B, int nprob, cudaStream_t st) {
    int maxM = 0, maxBlocks = 0;
    B.NBmax = 16; B.kmax = 16;
    for (int i = 0; i < nprob; ++i) {
        const TcLinProblem& p = B.p[i];
        KPD_REQUIRE(p.ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(p.X) & 15) == 0, "tc_linear: X rows must be 16-byte aligned (ldx=%d)", p.ldx);
        const int NB = p.N >= 256 ? 256 : (p.N + 15) / 16 * 16;
        if (NB > B.NBmax) B.NBmax = NB;
        if (p.K > B.kmax) B.kmax = p.K;
        if (p.M > maxM) maxM = p.M;
        if (cdiv(p.N, 256) > maxBlocks) maxBlocks = cdiv(p.N, 256);
    }
    if (maxM <= 0) return 0;
    B.stages = TCG_MAX_STAGES;
    while (B.stages > 2 && tc_linear_smem<NS>(B.kmax, B.NBmax, B.stages) > 227 * 1024) --B.stages;
    const size_t smem = tc_linear_smem<NS>(B.kmax, B.NBmax, B.stages);
    KPD_REQUIRE(smem <= 227 * 1024, "tc_linear: K=%d needs %zu B of shared memory", B.kmax, smem);
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(tc_linear_kernel<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        KPD_REQUIRE(e == cudaSuccess, "tc_linear: cannot set %zu B shared memory: %s", smem, cudaGetErrorString(e));
        configured = smem;
    }
    // column blocks per CTA: keep the launch near one wave of 148 CTAs while re-using each staged A tile
    const int row_tiles = cdiv(maxM, 128 / NS) * nprob;
    int groups = 148 / (row_tiles > 0 ? row_tiles : 1);
    if (groups < 1) groups = 1;
    if (groups > maxBlocks) groups = maxBlocks;
    B.bpc = cdiv(maxBlocks, groups);
    tc_linear_kernel<NS><<<dim3(cdiv(maxM, 128 / NS), cdiv(maxBlocks, B.bpc), nprob), TCG_THREADS, smem, st>>>(B);
    return check_launch("tc_linear_kernel");
}

int launch_tc_batch(TcLinBatch& B, int nprob, int nsplit, cudaStream_t st) {
    KPD_REQUIRE(nsplit == 1 || nsplit == 2, "tc_linear: nsplit must be 1 (bf16) or 2 (bf16x3)");
    KPD_REQUIRE(nprob >= 1 && nprob <= 2, "tc_linear: 1 or 2 problems per launch");
    return nsplit == 1 ? launch_tc_batch_ns<1>(B, nprob, st) : launch_tc_batch_ns<2>(B, nprob, st);
}

TcLinProblem tc_problem(const float* X, int ldx, const void* Wp, const float* bias, const float* R, int ldr, float* Y, int ldy,
                        int M, int K, int N, int act) {
    TcLinProblem p;
    p.X = X; p.Wp = static_cast<const uint4*>(Wp); p.bias = bias; p.R = R; p.Y = Y;
    p.ldx = ldx; p.ldr = ldr; p.ldy = ldy; p.M = M; p.K = K; p.N = N; p.act = act;
    return p;
}

int launch_tc_linear(const float* X, int ldx, const void* Wp, const float* bias, const float* R, int ldr, float* Y,
                     int ldy, int M, int K, int N, int act, int nsplit, cudaStream_t st) {
    if (M <= 0 || N <= 0) return 0;
    TcLinBatch B;
    memset(&B, 0, sizeof(B));
    B.p[0] = tc_problem(X, ldx, Wp, bias, R, ldr, Y, ldy, M, K, N, act);
    return launch_tc_batch(B, 1, nsplit, st);
}

}  // namespace kpd

#ifdef KPD_TCG_TIMERS
extern "C" int kpd_debug_tcg_times(unsigned long long* out16) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out16, kpd::g_tcg_times, sizeof(unsigned long long) * 16);
    unsigned long long z[16] = {0};
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(kpd::g_tcg_times, z, sizeof(z));
    return e == cudaSuccess ? 0 : 1;
}
#endif

extern "C" int kpd_tc_linear(const float* X, int32_t ldx, const void* Wp, const float* bias, const float* R, int32_t ldr,
                             float* Y, int32_t ldy, int32_t M, int32_t K, int32_t N, int32_t act, int32_t nsplit, void* stream) {
    return kpd::launch_tc_linear(X, ldx, Wp, bias, R, ldr, Y, ldy, M, K, N, act, nsplit, static_cast<cudaStream_t>(stream));
}
