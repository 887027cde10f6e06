// Shared pieces of the warp-specialised tensor-core kernels (gvp_ws.inl, egnn_ws.inl): tile configuration, the
// row addressing of the UMMA A operand (plain or hi/lo-stacked), activation intrinsics, warp-level MMA.
#pragma once
#include "tc.cuh"

namespace kpd {

// phase timers (cycles, read with clock64 by one thread and summed over CTAs); see kpd_debug_ws_times()
#define TC_T(var) const long long var = clock64()

// bf16 mode does not need fp32-faithful transcendentals: one MUFU op per element,
// silu(x) = x * sigmoid(x) = h + h * tanh(h), sigmoid(x) = 0.5 + 0.5 * tanh(h), h = x / 2
__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float silu_fast(float x) { const float h = 0.5f * x; return fmaf(h, tanh_fast(h), h); }
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }

namespace ws {

// small fp32 weights of one GVP in shared memory, laid out as mma.sync B fragments (see vector MMAs below):
//   Wh pairs [12][WH_LD][2]: (our channel 2p, 2p+1; h)   Wu pairs [12][WU_LD][2]: (h = 2p, 2p+1; u)
// leading dimensions == 4 (mod 16) in 8-byte units make the 64-bit fragment loads conflict-free
constexpr int WH_LD = 36, WU_LD = 20;
constexpr int WH_SZ = 12 * WH_LD * 2, WU_SZ = 12 * WU_LD * 2;
template <int NS> constexpr int wsm_floats() { return NS * (WH_SZ + WU_SZ) + 256 + 16; }   // (hi[, lo]) Wh | Wu | bf | bg

// NS = 2 ("bf16x3", split (hi, lo) bf16 operands) comes in two layouts:
//   STACK (KS_ = false): the hi and lo rows of 64 tile rows stacked along M into one 128-row A operand; two MMAs per
//         k-step ([A_hi; A_lo] x W_hi, x W_lo) give all FOUR hi/lo products, the epilogue adds the two accumulator rows;
//   KS    (KS_ = true):  hi and lo PLANES of a 128-row tile, three MMAs per k-step (A_hi W_hi + A_lo W_hi + A_hi W_lo:
//         the lo x lo product is below the fp32 rounding of the sum) into ONE accumulator -- a weight slab streamed
//         from L2 serves 128 tile rows instead of 64 (the slab stream is what bounds the k-step rate, DESIGN.md 4.3),
//         3 instead of 4 tensor-core MACs per algorithmic MAC, half the TMEM read traffic per tile row.
template <int R_, int NS_, int NWX_ = 0, bool KS_ = false>
struct Cfg {
    static constexpr int R = R_, NS = NS_;
    static constexpr bool KS = KS_ && NS_ == 2;
    static constexpr bool STACK = NS_ == 2 && !KS_;
    static constexpr int NWV = R / 8;                // vector-owning SIMT warps: 8 tile rows each (mma.sync fragments)
    static constexpr int NW = NWV + NWX_;            // all SIMT warps; the NWX extra ones only help with the epilogues,
                                                     // gathers and reductions (more warps in flight per SM quadrant)
    static constexpr int NT_SIMT = 32 * NW;
    static constexpr int NT = NT_SIMT + 64;
    static constexpr int MMA_M = STACK ? 2 * R : R;  // STACK: the hi and lo rows of a tile form ONE 128-row A operand
    static constexpr int KCS = (MMA_M / 8) * 128 + 16;   // bytes between k-chunks of A (+16: bank rotation for column walks)
    static constexpr int STAGES = NS == 1 ? 8 : 4;
    static constexpr int SLAB = NS * 8192;           // one ring stage: one k-step of a 256-row weight (hi [, lo])
    static constexpr int WG_BYTES = NS * 8192;       // gates weight: 16 k-steps x 512 B (hi [, lo])
    static constexpr int WGB = KS ? 0 : NS == 1 ? 2 : 1;   // gates weight buffers (KS: the gates weight travels through the ring)
    static constexpr int WSM = wsm_floats<NS>();
    // its Wh | Wu part (dead after the Vu GEMM); KS keeps plain fp32 [24][28] / [24][20] images instead (vec_fma) ...
    static constexpr int WSM_W = KS ? 24 * 28 + 24 * 20 : NS * (WH_SZ + WU_SZ);
    static constexpr int WSM_B = 256 + 16;               // ... and its bias part bf | bg (live until epilogue 2)
    static constexpr int NCG = NW / 4;               // column groups of the epilogues (4 TMEM lane quarters x NCG)
};

// Byte offset of tile row r inside a k-chunk of A.  NS = 1 and KS: plain canonical rows.  STACK: MMA rows are ordered
// (16-row group q, plane, row % 16): TMEM lanes [32q, 32q+16) hold the hi rows and [32q+16, 32q+32) the lo rows of
// tile rows [16q, 16q+16), so one warp reads both halves of a row's accumulator (16x256b loads) and adds them.
// The lo row of r sits 256 bytes after its hi row.
template <class C>
__device__ __forceinline__ uint32_t row_off(int r) {
    if (C::STACK) return (uint32_t)((4 * (r >> 4) + ((r >> 3) & 1)) * 128 + (r & 7) * 16);
    return (uint32_t)((r >> 3) * 128 + (r & 7) * 16);
}

__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// warp-level tensor-core MMA, D(16x8) += A(16x8) B(8x8), tf32 operands, fp32 accumulation
__device__ __forceinline__ void mma_tf32(float& d0, float& d1, float& d2, float& d3, float a0, float a1, float a2, float a3,
                                         float b0, float b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3)
                 : "r"(__float_as_uint(a0)), "r"(__float_as_uint(a1)), "r"(__float_as_uint(a2)), "r"(__float_as_uint(a3)),
                   "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

__device__ __forceinline__ float sqrt_fast(float x) { float y; asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// fp32-grade logistic on two MUFU ops (ex2 and rcp are good to ~2^-22; no range fix-ups: 1 + 2^t never overflows
// to a value rcp cannot take, and a huge argument gives rcp(inf) = 0, the right limit)
__device__ __forceinline__ float sigmoid_acc(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return r;
}
__device__ __forceinline__ float silu_acc(float x) { return x * sigmoid_acc(x); }

template <int NS>
__device__ __forceinline__ float act_silu(float x) { return NS == 1 ? silu_fast(x) : silu_acc(x); }
template <int NS>
__device__ __forceinline__ float act_sigmoid(float x) { return NS == 1 ? sigmoid_fast(x) : sigmoid_acc(x); }

// Paired fp32 arithmetic (FADD2 / FMUL2 / FFMA2: two IEEE round-to-nearest operations in one instruction, the same bits
// as two scalar ones -- no .ftz, no contraction).  The operands of one instruction live in an aligned register pair, so
// the bf16x3 epilogues keep their values as float2.
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
    unsigned long long d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 bcast2(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 u2f2(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }

// fp32-grade logistic of two values on three MUFU ops: an ex2 each and ONE reciprocal shared through the product of the
// denominators, sigmoid(x0) = d1 / (d0 d1).  The ex2 argument is clamped at 62: then d <= 2^62 + 1, d0 d1 <= 2^124 stays
// finite and its reciprocal >= 2^-124 stays normal under .ftz (an unclamped e = inf would give 0 * inf = NaN).  The clamp
// only acts for x < -42.9, where sigmoid(x) < 2^-62: the result is off by less than 2^-62 absolute.  The product and the
// extra multiply add two fp32 roundings to the ~2^-22 of ex2 and rcp.
__device__ __forceinline__ float2 sigmoid2_acc(float2 x) {
    const float2 t = mul2(x, bcast2(-1.4426950408889634f));
    float e0, e1, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fminf(t.x, 62.f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fminf(t.y, 62.f)));
    const float2 d = add2(bcast2(1.f), make_float2(e0, e1));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d.x * d.y));
    return mul2(bcast2(r), make_float2(d.y, d.x));
}
__device__ __forceinline__ float2 silu2_acc(float2 x) { return mul2(x, sigmoid2_acc(x)); }

// 2 fp32 values -> packed bf16 pair hi and the packed bf16 pair of the residuals lo
__device__ __forceinline__ void split2(float2 f, uint32_t& hi, uint32_t& lo) {
    hi = tc::pack_bf16x2(f.x, f.y);
    const float2 r = sub2(f, u2f2(hi << 16, hi & 0xffff0000u));
    lo = tc::pack_bf16x2(r.x, r.y);
}

// 8 fp32 values -> packed bf16 hi (and the bf16 residual lo)
__device__ __forceinline__ void split8(const float (&f)[8], uint4& hi, uint4& lo) {
    hi.x = tc::pack_bf16x2(f[0], f[1]); hi.y = tc::pack_bf16x2(f[2], f[3]);
    hi.z = tc::pack_bf16x2(f[4], f[5]); hi.w = tc::pack_bf16x2(f[6], f[7]);
    lo.x = tc::pack_bf16x2(f[0] - __uint_as_float(hi.x << 16), f[1] - __uint_as_float(hi.x & 0xffff0000u));
    lo.y = tc::pack_bf16x2(f[2] - __uint_as_float(hi.y << 16), f[3] - __uint_as_float(hi.y & 0xffff0000u));
    lo.z = tc::pack_bf16x2(f[4] - __uint_as_float(hi.z << 16), f[5] - __uint_as_float(hi.z & 0xffff0000u));
    lo.w = tc::pack_bf16x2(f[6] - __uint_as_float(hi.w << 16), f[7] - __uint_as_float(hi.w & 0xffff0000u));
}

}  // namespace ws
}  // namespace kpd
