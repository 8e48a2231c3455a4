// Implicit-GEMM convolution on tcgen05 / TMEM for NHWC bf16 activations (sm_100a).
//
// Replaces Conv.forward_fuse = SiLU(conv2d(x, w', b')) (ultralytics/nn/modules/conv.py:83-93) with BN
// folded (utils/torch_utils.py:255-286), the Bottleneck residual add (block.py:493-495) and the bias-only
// 1x1 convs of Detect (head.py:93-96).
//
// GEMM view:  D[M = B*Ho*Wo pixels, N = Cout] = sum over (tap, channel chunk) A[M, BK] * W[N, BK]^T
//   * M tile = 128 output pixels.  "tap" mode (1x1, stride 2, small maps): the tile is an (NB x TH x TW)
//     patch and the A operand of filter tap (kh,kw) is ONE tiled 4-D TMA box of the NHWC input shifted by
//     (kw-pad, kh-pad).  "halo" mode (3x3 stride 1): the tile is 16 rows x 8 columns and ONE box of 18 rows
//     per (kw, channel chunk) serves the three kh taps -- the tap operands are the same shared-memory tile
//     at row offsets 0 / 8 / 16 (swizzle-atom aligned), so the input is fetched 3.4x instead of 9x.
//     Image borders are the TMA's out-of-bounds zero fill (= conv zero padding).  Stride-2 convs read one
//     of four parity-decimated views of the input, each again a plain tiled map.
//   * Channels are cut into a "segment" of 64-channel chunks (128-byte rows, SWIZZLE_128B) and, when Cin is
//     not a multiple of 64, a second segment of 32- or 16-channel chunks (SWIZZLE_64B / 32B), all in the
//     K-major canonical UMMA layout consumed by tcgen05.mma (M=128, N=n_tile, K=16) from shared memory.
//   * Weights stay resident in shared memory for the life of the CTA when they fit (all P2/P3-level layers).
//   * Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner (whole warp runs the loop with
//     uniform control flow, one elected lane issues), warps 2..9 = epilogue (TMEM -> registers -> +bias ->
//     SiLU -> (+residual) -> bf16 -> 256-bit stores into the output channel slice).
//   * Persistent CTAs (1 or 2 per SM), multi-stage smem ring (mbarrier full/empty), two TMEM accumulator
//     stages so the epilogue of tile i overlaps the MMAs of tile i+1.
//   * Output goes to a channel slice [coff, coff+Cout) of a wider NHWC buffer: torch.cat / chunk of
//     C2f / SPPF / Concat / Detect become offset writes and offset reads.
#include "common.cuh"

#include <limits.h>

#include <algorithm>
#include <mutex>

namespace {

constexpr int kMaxStages = 12;
constexpr int kThreadsMw1 = 32 * (1 + 1 + 8), kThreadsMw2 = 32 * (1 + 2 + 8);   // warp 0 TMA, 1 or 2 MMA warps, 8 epilogue warps
constexpr int kMaxNTile = 256;
constexpr int kMaxAcc = 4;                         // accumulator stages in tensor memory
constexpr int kMaxSeg = 4;                         // up to two sources (Concat folded into the conv) x two chunk widths
constexpr int kMaxChainBlk = 6;                    // K blocks of a chained 1x1 conv (<= 384 channels)

// One K segment: `kchunks` chunks of `bk` channels starting at channel `c_off`.
struct alignas(64) Seg {
    CUtensorMap tmA[4];
    CUtensorMap tmB;
    int c_off, bk, kchunks;   // c_off: first channel in the (concatenated) GEMM-K order; src_c: first channel inside its source
    int src_c;
    int up;                   // 2: the source is stored at half resolution (nearest-2x upsample folded into a 5-D tensor map)
    int h_lo;                 // up == 2: rows of one low-resolution image
    uint32_t a_tx;            // bytes one A box delivers
    uint32_t b_block_bytes;   // n_tile * bk * 2
    uint32_t b_block_stride;  // rounded up to 1024
    uint32_t b_base;          // resident weights: offset of this segment's blocks inside the weight region
    uint32_t kh_step16;       // halo mode: (8 rows * row bytes) >> 4
    uint32_t desc_hi;         // high word of the shared-memory matrix descriptor (SBO, version, swizzle)
    uint32_t desc_hi_w;       // the same for weight blocks (8-row pitch) where the pixel operand has another pitch (halo 2 / 3)
    uint32_t a_tx4[4];        // halo 3 (stride 2): bytes delivered by the box of parity view 0..3
    uint32_t desc_hi9;        // halo 3: pixel-operand descriptor high word for the 9-pixel-wide boxes (pw = 1)
};

struct alignas(64) ConvParams {
    Seg seg[kMaxSeg];
    int nseg;
    int B, Ho, Wo;
    int TW, TH, NB;
    int tiles_w, tiles_h, tiles_nb;
    int n_tiles, n_tile, Cout;
    int Cin, ksize, stride, pad;
    int num_stages;
    int halo;                 // 3x3 stride-1: 1 = one 18-row box per (kw, K chunk) serves the 3 kh taps;
                              // 2 = one (TW+2) x (TH+2) box per K chunk serves all 9 taps by descriptor start row;
                              // 3 = 3x3 stride 2: one box per input parity (row, column) serves the 1 / 2 / 2 / 4 taps that read it
    int b_resident;           // 1: every weight block stays in shared memory for the lifetime of the CTA
    uint32_t a_bytes;         // shared-memory stride of one A stage (1024-aligned)
    uint32_t b_stage_stride;  // streamed weights: bytes of weight blocks per stage
    uint32_t b_res_bytes;     // resident weights: total bytes delivered by the preload
    uint32_t tmem_cols;
    __nv_bfloat16* out; int out_cstride, out_coff;
    const __nv_bfloat16* res; int res_cstride, res_coff;
    const float* bias;
    int act;
    int wide;                 // 1: output (and residual) chunks are 32-byte aligned -> 256-bit accesses
    int epi;                  // 0: bf16 channel-slice store; 1: DFL head (N = 64 -> 4 fp32 distances per pixel);
                              // 2: class head (N = nc -> fp32 {best logit, class} per pixel)   [Detect._inference fused]
    float* out_f32;           // epi 1: [pixels][4], epi 2: [pixels][2]
    int mma_warps;            // 1 or 2 MMA-issuing warps (2: alternate tiles, two stage rings)
    int epi_warps;            // 8 or 16 epilogue warps (16 only with two MMA warps, one CTA per SM)
    int acc_stages;           // accumulator stages in tensor memory (2..4): tile t uses stage t % acc_stages
    uint32_t magic_nt, magic_tw, magic_th;   // ceil(2^32 / d) for d = n_tiles, tiles_w, tiles_h (0: d == 1) -- tile index -> coordinates
    int tma_lanes;            // halo 3: 4 = the producer issues four stage fills per instruction (lanes 0..3), 1 = one by one
    int halo3_k;              // halo 3: K chunks of all segments together (stage fills per parity view)
    // ---- chained 1x1 conv (conv_tc_kernel<.., CH = 1>): the activated bf16 tile of this conv never leaves the SM.  Half of the
    //      epilogue warps ("E1") write it into shared memory in the UMMA operand layout, the MMA warps run a second GEMM on it
    //      against the resident weights of the following 1x1 conv -- optionally together with K blocks loaded by TMA from the
    //      channels that the 1x1 conv reads besides this conv's output (C2f: cat(y0, y1, m_1..m_n-1) | m_n, block.py:315-319) --
    //      and the other half ("E2") runs the final epilogue (EPI) on the second accumulator.  out / out_f32 / epi describe the
    //      CHAINED conv's output; bias / act / res stay this conv's. ----
    int chain;
    int c2_n, c2_cout, c2_act;            // N tile (padded to 16), real Cout and activation of the chained conv
    const float* c2_bias;
    int c2_nblk;                          // K blocks of the chained GEMM, in K order: TMA-fed ("x") blocks first, then E1's blocks
    int c2_nx;                            // how many of them are TMA-fed
    int c2_bk[kMaxChainBlk];              // channels of block i (64 / 32 / 16)
    int c2_src_c[kMaxChainBlk];           // x blocks: first channel inside the extra source; E1 blocks: first channel of the main conv's tile
    uint32_t c2_a_off[kMaxChainBlk];      // byte offset of the block inside one staged-tile buffer
    uint32_t c2_w_off[kMaxChainBlk];      // byte offset of the block's weights inside the W2 region
    uint32_t c2_desc_hi[kMaxChainBlk];    // descriptor high word (8-row pitch, swizzle of the block's row width)
    uint32_t c2_w_bytes[kMaxChainBlk];    // bytes the block's weight box delivers
    CUtensorMap tmW2[kMaxChainBlk];       // [Cout2][K2] weights, box (bk, c2_n)
    CUtensorMap tmX[kMaxChainBlk];        // x blocks: (C, W, H, B) view of the extra source, box (bk, TW, TH, NB)
    uint32_t c2_x_tx;                     // bytes the x blocks of one tile deliver
    uint32_t c2_buf_off, c2_buf_bytes;    // shared-memory offset of the two staged-tile buffers, bytes per buffer
    uint32_t c2_wreg_off;                 // shared-memory offset of the W2 region
    uint32_t c2_tmem_col;                 // first tensor-memory column of the two chained accumulators
};

// x / d by one multiply-high (magic = ceil(2^32 / d), exact while x * d < 2^32 -- checked on the host); magic 0 means d == 1
__device__ __forceinline__ int fast_div(int x, uint32_t magic) { return magic ? (int)__umulhi((uint32_t)x, magic) : x; }

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&o)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
                 "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
}
__device__ __forceinline__ void ld_global_v8(const void* p, uint32_t (&o)[8]) {
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=r"(o[0]), "=r"(o[1]), "=r"(o[2]), "=r"(o[3]),
                 "=r"(o[4]), "=r"(o[5]), "=r"(o[6]), "=r"(o[7]) : "l"(p));
}

// bias + activation + residual + bf16 pack + store of one 16-column chunk held in registers.
// WIDE: pointers are 32-byte aligned -> one 256-bit access per thread (a full L2 sector per instruction).
template <bool WIDE, bool BIAS = true>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[16], const float* __restrict__ sb, int act, int nv,
                                               __nv_bfloat16* __restrict__ optr, const __nv_bfloat16* __restrict__ rptr) {
    // act: sb holds HALF the bias, h = (acc + bias) / 2 comes out of one FFMA (bit-identical to 0.5f * (acc + bias): scaling by
    // a power of two commutes with rounding) and SiLU(x) = h + h tanh(h) (silu_fast) is one MUFU + one FFMA more
    float f[16];
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (BIAS) b4 = *reinterpret_cast<const float4*>(sb + i);
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float a = __uint_as_float(v[i + k]);
            if (act) {
                const float h = fmaf(a, 0.5f, bb[k]);
                float t;
                asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
                f[i + k] = fmaf(h, t, h);
            } else {
                f[i + k] = a + bb[k];
            }
        }
    }
    if (nv == 16) {
        uint32_t o[8];
        if (rptr) {
            uint32_t rr[8];
            if (WIDE) ld_global_v8(rptr, rr);
            else {
                const uint4 r0 = *reinterpret_cast<const uint4*>(rptr);
                const uint4 r1 = *reinterpret_cast<const uint4*>(rptr + 8);
                rr[0] = r0.x; rr[1] = r0.y; rr[2] = r0.z; rr[3] = r0.w; rr[4] = r1.x; rr[5] = r1.y; rr[6] = r1.z; rr[7] = r1.w;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) { f[2 * i] += bf16_lo(rr[i]); f[2 * i + 1] += bf16_hi(rr[i]); }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = pack_bf16x2(f[2 * i], f[2 * i + 1]);
        if (WIDE) st_global_v8(optr, o);
        else {
            *reinterpret_cast<uint4*>(optr) = make_uint4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uint4*>(optr + 8) = make_uint4(o[4], o[5], o[6], o[7]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if (i < nv) {
                float x = f[i];
                if (rptr) x += __bfloat162float(rptr[i]);
                optr[i] = __float2bfloat16_rn(x);
            }
        }
    }
}

// E1 of a chained conv: bias + activation (+ residual) + bf16 pack of one 16-column chunk, stored as two 16-byte units of
// its row of a K-major operand block.  p0 / p1 are the units' shared-memory addresses with the swizzle already applied (the
// swizzle is a function of the absolute address, DESIGN.md fact 3: unit index ^= address bits [7, 7 + log2(row_bytes / 16));
// a thread's row and chunk never change, so the caller computes them once per kernel, not per tile).
__device__ __forceinline__ void epilogue_chunk_smem(const uint32_t (&v)[16], const float* __restrict__ sb, int act,
                                                    const __nv_bfloat16* __restrict__ rptr, uint32_t p0, uint32_t p1) {
    float f[16];
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(sb + i);
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float a = __uint_as_float(v[i + k]);
            if (act) {
                const float h = fmaf(a, 0.5f, bb[k]);
                float t;
                asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
                f[i + k] = fmaf(h, t, h);
            } else {
                f[i + k] = a + bb[k];
            }
        }
    }
    if (rptr) {
        const uint4 r0 = *reinterpret_cast<const uint4*>(rptr);
        const uint4 r1 = *reinterpret_cast<const uint4*>(rptr + 8);
        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) { f[2 * i] += bf16_lo(rr[i]); f[2 * i + 1] += bf16_hi(rr[i]); }
    }
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = pack_bf16x2(f[2 * i], f[2 * i + 1]);
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(p0), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(p1), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
}

// ---- Detect head fused into the epilogue (ultralytics/nn/modules/head.py:152-187, block.py:78-81 DFL) ----
// Logits are rounded to bf16 first, exactly as the unfused path stores them, so both paths give the same bits.
__device__ __forceinline__ float bf16_rt(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// one DFL side: softmax expectation over 16 bins (same summation order as decode_kernel: bins 0-7, bins 8-15, add)
__device__ __forceinline__ float dfl_side(const uint32_t (&v)[16], const float* __restrict__ sb) {
    float f[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 b4 = *reinterpret_cast<const float4*>(sb + 4 * q);
        const __nv_bfloat162 p0 = __floats2bfloat162_rn(__uint_as_float(v[4 * q]) + b4.x, __uint_as_float(v[4 * q + 1]) + b4.y);
        const __nv_bfloat162 p1 = __floats2bfloat162_rn(__uint_as_float(v[4 * q + 2]) + b4.z, __uint_as_float(v[4 * q + 3]) + b4.w);
        const uint32_t u0 = *reinterpret_cast<const uint32_t*>(&p0), u1 = *reinterpret_cast<const uint32_t*>(&p1);
        f[4 * q] = __uint_as_float(u0 << 16); f[4 * q + 1] = __uint_as_float(u0 & 0xFFFF0000u);
        f[4 * q + 2] = __uint_as_float(u1 << 16); f[4 * q + 3] = __uint_as_float(u1 & 0xFFFF0000u);
    }
    float m = f[0];
#pragma unroll
    for (int i = 1; i < 16; ++i) m = fmaxf(m, f[i]);
    const float ml = m * kLog2e;
    float se0 = 0.f, sw0 = 0.f, se1 = 0.f, sw1 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float e = dfl_exp(f[i], ml); se0 += e; sw0 = fmaf(e, (float)i, sw0); }
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float e = dfl_exp(f[8 + i], ml); se1 += e; sw1 = fmaf(e, 8.f + (float)i, sw1); }
    return (sw0 + sw1) / (se0 + se1);
}
// Class head: running argmax as ONE integer max per element.  The logit is rounded to bf16 first (as the unfused path
// stores it), so the low 16 bits of its fp32 pattern are free: key = order-preserving integer image of the value in
// the high half, 0xFFFF - class in the low half (ties -> lowest class, as torch.max / decode_kernel).
// Two logits per conversion (one packed cvt.rn.bf16x2), no per-element predicate: channels past Cout carry a bias of
// -inf (set where s_bias is filled), so they never win.
__device__ __forceinline__ int cls_key_bits(int t, int low) {            // t: bf16 pattern in the high half, low half anything
    const int k = t ^ ((t >> 31) & 0x7FFF0000);                          // signed-int order == float order (high half)
    return (k & (int)0xFFFF0000) | low;
}
// chunk = 16 classes starting at c0 (a multiple of 16): inside the chunk the low bits are the immediates 15 - i, the
// chunk's own 12 bits are OR-ed in once after the 16-way max.
__device__ __forceinline__ void cls_chunk(const uint32_t (&v)[16], const float* __restrict__ sb, int c0, int& best) {
    int m[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 b4 = *reinterpret_cast<const float4*>(sb + 4 * q);
        const __nv_bfloat162 p0 = __floats2bfloat162_rn(__uint_as_float(v[4 * q]) + b4.x, __uint_as_float(v[4 * q + 1]) + b4.y);
        const __nv_bfloat162 p1 = __floats2bfloat162_rn(__uint_as_float(v[4 * q + 2]) + b4.z, __uint_as_float(v[4 * q + 3]) + b4.w);
        const int u0 = *reinterpret_cast<const int*>(&p0), u1 = *reinterpret_cast<const int*>(&p1);
        const int k0 = cls_key_bits(u0 << 16, 15 - 4 * q), k1 = cls_key_bits(u0, 14 - 4 * q);
        const int k2 = cls_key_bits(u1 << 16, 13 - 4 * q), k3 = cls_key_bits(u1, 12 - 4 * q);
        m[q] = max(max(k0, k1), max(k2, k3));
    }
    const int m16 = max(max(m[0], m[1]), max(m[2], m[3])) | (0xFFF0 - c0);
    best = max(best, m16);
}
__device__ __forceinline__ float2 cls_unkey(int key) {
    const int kb = key & (int)0xFFFF0000;
    const int b = key >= 0 ? kb : ((kb | 0xFFFF) ^ 0x7FFFFFFF);
    return make_float2(__int_as_float(b), (float)(0xFFFF - (key & 0xFFFF)));
}

// EPI: epilogue variant (ConvParams::epi), HALO: ConvParams::halo -- compile-time copies of the two fields, so that each
// instance carries only its own loops (the kernel is sensitive to registers / code size in the issue and epilogue paths)
// All 9 x MPS MMAs of one single-box (halo 2) stage, fully unrolled: every descriptor is one uniform add away from the
// stage's pixel-box base (tap (kh, kw) starts (kh * 10 + kw) rows in, one row = 2 * MPS descriptor units) and from the
// weight block of (tap 0, this K chunk) (taps are tb_step apart).
template <int MPS>
__device__ __forceinline__ void ss_issue_halo2(uint32_t leader, uint32_t d_addr, uint32_t idesc, uint64_t hi_a, uint64_t hi_b,
                                               uint32_t a_lo, uint32_t tb_lo, uint32_t tb_step, uint32_t& accum) {
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const uint32_t ta = a_lo + (uint32_t)(((t / 3) * 10 + (t % 3)) * 2 * MPS);
        const uint32_t tb = tb_lo + (uint32_t)t * tb_step;
#pragma unroll
        for (int j = 0; j < MPS; ++j) {
            tc_mma_bf16_if(leader, d_addr, hi_a | (uint64_t)(ta + 2u * j), hi_b | (uint64_t)(tb + 2u * j), idesc, accum);
            accum = 1;
        }
    }
}

// TPG taps x MPS K-steps of one stage of the tap / three-box modes, unrolled: tap t reads the stage's A tile t * a_step further
// in (halo 1: 8 rows = 16 * MPS units; tap mode: TPG == 1) and weight block t * b_step further (resident: tap stride in blocks;
// streamed: the stage's t-th block).
template <int MPS, int TPG>
__device__ __forceinline__ void ss_issue_taps(uint32_t leader, uint32_t d_addr, uint32_t idesc, uint64_t hi, uint32_t a_lo, uint32_t tb_lo,
                                              uint32_t b_step, uint32_t& accum) {
#pragma unroll
    for (int t = 0; t < TPG; ++t) {
        const uint32_t ta = a_lo + (uint32_t)(t * 16 * MPS), tb = tb_lo + (uint32_t)t * b_step;
#pragma unroll
        for (int j = 0; j < MPS; ++j) {
            tc_mma_bf16_if(leader, d_addr, hi | (uint64_t)(ta + 2u * j), hi | (uint64_t)(tb + 2u * j), idesc, accum);
            accum = 1;
        }
    }
}

// MW: MMA-issuing warps.  1: warp 0 TMA, warp 1 MMA, warps 2..9 epilogue, up to two CTAs per SM.  2 (plans with ONE CTA per SM):
// warps 1 and 2 issue alternate tiles, each with its own accumulator stage and its own ring of pipeline stages.
template <int EPI, int HALO, int MW, int EW = 8, int CH = 0>
__global__ void __launch_bounds__(32 * (1 + MW + EW), MW == 1 ? 2 : 1) conv_tc_kernel(const __grid_constant__ ConvParams p) {
    // EW epilogue warps, kSub per TMEM lane quadrant (the epilogue is latency bound -- TMEM load, MUFU, stores -- so the
    // one-CTA-per-SM plans run 16: four warps per scheduler hide each other's stalls)
    constexpr int kEpiWarps = EW, kMmaWarps = MW, kThreads = 32 * (1 + MW + EW), kSub = EW / 4;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
    __shared__ __align__(8) uint64_t tfull_bar[kMaxAcc];
    __shared__ __align__(8) uint64_t tempty_bar[kMaxAcc];
    __shared__ __align__(8) uint64_t bres_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float s_bias[kMaxNTile];
    __shared__ int s_key[2][128];                      // class-head epilogue: partial argmax keys of the second warp of each quadrant
    // chained conv (CH): staged-tile buffers k & 1 (k = ordinal of the tile inside this CTA)
    __shared__ __align__(8) uint64_t a2_full[2];       // E1 has written its blocks            (E1 threads arrive)
    __shared__ __align__(8) uint64_t a2_empty[2];      // the chained MMAs have read the buffer (tcgen05.commit)
    __shared__ __align__(8) uint64_t x_full[2];        // the TMA-fed blocks have landed
    __shared__ __align__(8) uint64_t t2_full[2];       // chained accumulator complete          (tcgen05.commit)
    __shared__ __align__(8) uint64_t t2_empty[2];      // E2 has drained it                     (E2 threads arrive)
    __shared__ __align__(16) float s_bias2[CH ? kMaxNTile : 4];
    constexpr int kE1Warps = CH ? EW / 2 : EW;         // warps that drain the main accumulator

    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + (size_t)p.num_stages * p.a_bytes;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.nseg; ++s) {
            tma_prefetch_desc(&p.seg[s].tmA[0]);
            if (p.stride == 2) { tma_prefetch_desc(&p.seg[s].tmA[1]); tma_prefetch_desc(&p.seg[s].tmA[2]); tma_prefetch_desc(&p.seg[s].tmA[3]); }
            tma_prefetch_desc(&p.seg[s].tmB);
        }
        for (int s = 0; s < p.num_stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < kMaxAcc; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 32 * kE1Warps); }
        mbar_init(&bres_bar, 1);
        if (CH) {
            for (int s = 0; s < 2; ++s) {
                mbar_init(&a2_full[s], 32 * kE1Warps); mbar_init(&a2_empty[s], 1); mbar_init(&x_full[s], 1);
                mbar_init(&t2_full[s], 1); mbar_init(&t2_empty[s], 32 * (EW - kE1Warps));
            }
        }
        fence_mbar_init();
    }
    if (warp == 1) {
        tmem_alloc(&tmem_base_s, p.tmem_cols);
        tmem_relinquish();
    }
    const float bias_scale = ((EPI == 0 || CH) && p.act) ? 0.5f : 1.f;      // SiLU layers keep bias / 2 (epilogue_chunk)
    if (p.n_tiles == 1)
        for (int i = threadIdx.x; i < p.n_tile; i += kThreads) s_bias[i] = i < p.Cout ? __ldg(p.bias + i) * bias_scale : ((EPI == 2 && !CH) ? -INFINITY : 0.f);
    if (CH) {
        const float scale2 = (EPI == 0 && p.c2_act) ? 0.5f : 1.f;
        for (int i = threadIdx.x; i < p.c2_n; i += kThreads) s_bias2[i] = i < p.c2_cout ? __ldg(p.c2_bias + i) * scale2 : (EPI == 2 ? -INFINITY : 0.f);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    pdl_launch_dependents();        // the next conv of the stream may begin its prologue on SMs this grid has left

    const int tiles_m = p.tiles_w * p.tiles_h * p.tiles_nb;
    const int total_tiles = tiles_m * p.n_tiles;
    const int taps = p.ksize * p.ksize;
    // pipeline stages consumed per K chunk / filter taps served by one stage:
    //   halo 1: one 18-row box per kw serves the three kh taps; halo 2: ONE (TW+2) x (TH+2) box serves all nine taps
    const int groups = HALO == 3 ? 4 : HALO == 2 ? 1 : HALO ? 3 : taps;
    const int taps_per_group = HALO == 2 ? 9 : HALO == 1 ? 3 : 1;
    const int nseg = p.nseg;

    // Producer and MMA warps run their loops with the whole warp (uniform control flow keeps descriptors and
    // addresses in uniform registers); one elected lane issues the TMA / tcgen05 instructions.
    if (warp == 0) {
        // ===================== TMA producer =====================
        const bool leader = elect_one();
        constexpr int halo = HALO;
        const int b_res = p.b_resident, Cin = p.Cin, num_stages = p.num_stages;
        const int ksz = p.ksize, pad = p.pad, stride = p.stride, n_tiles = p.n_tiles, n_tile = p.n_tile;
        const int tiles_w = p.tiles_w, tiles_h = p.tiles_h, TW = p.TW, TH = p.TH, NB = p.NB;
        const uint32_t a_bytes = p.a_bytes, b_stage_stride = p.b_stage_stride;
        if (b_res && leader) {
            mbar_expect_tx(&bres_bar, p.b_res_bytes);
            for (int s = 0; s < nseg; ++s) {
                const Seg& sg = p.seg[s];
                for (int tap = 0; tap < taps; ++tap)
                    for (int kc = 0; kc < sg.kchunks; ++kc)
                        tma_load_2d(smem_b + sg.b_base + (size_t)(tap * sg.kchunks + kc) * sg.b_block_stride, &sg.tmB, &bres_bar,
                                    tap * Cin + sg.c_off + kc * sg.bk, 0);
            }
            if (CH) {               // weights of the chained conv: block i = K columns [k0, k0 + bk) of [Cout2][K2]
                int k0 = 0;
                for (int i = 0; i < p.c2_nblk; ++i) { tma_load_2d(smem + p.c2_wreg_off + p.c2_w_off[i], &p.tmW2[i], &bres_bar, k0, 0); k0 += p.c2_bk[i]; }
            }
        }
        pdl_wait();                 // activations of the previous layer: only after the predecessor grid has completed
        // p.mma_warps == 2: two stage rings of num_stages / 2 slots; ring r holds the tiles issued by MMA warp r (a ring with
        // two consumers would let one of them run a whole revolution ahead, which mbarrier phase parity cannot tell apart)
        const int ring_stages = MW == 2 ? num_stages >> 1 : num_stages;
        const int tma_lanes = p.tma_lanes;
        int stage = 0; uint32_t phase = 0;                  // MW == 1: the one ring; MW == 2: the ring of the current tile
        int ostage = ring_stages; uint32_t ophase = 0;      // MW == 2: saved position in the other ring
        int stage_lo = 0, stage_hi = ring_stages;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int m0 = fast_div(tile, p.magic_nt), n_idx = tile - m0 * n_tiles;
            const int m1 = fast_div(m0, p.magic_tw), m2 = fast_div(m1, p.magic_th);
            const int w0 = (m0 - m1 * tiles_w) * TW;
            const int h0 = (m1 - m2 * tiles_h) * TH;
            const int n0 = m2 * NB;
            if (halo == 3 && tma_lanes > 1) {
                // stride 2, four stage fills per instruction: the tile's fills in consumption order (parity view g, then K chunk)
                // are dealt to lanes 0..3, which wait for their own stage and issue their own box side by side -- the producer warp
                // ran ~110 instructions per box and was 87 % busy on the 32 -> 64 stride-2 layer (profiles/r02_conv_chain_summary.md);
                // tools/tma_probe.cu: boxes issued by several lanes of one instruction proceed in parallel
                const int K = p.halo3_k, n_fill = 4 * K;
                int r = lane, g = 0;
                while (r >= K) { r -= K; ++g; }
                for (int b0 = 0; b0 < n_fill; b0 += 4) {
                    if (lane < 4) {
                        int st = stage + lane; uint32_t ph = phase;
                        if (st >= stage_hi) { st -= ring_stages; ph ^= 1; }
                        int s = 0, kc = r;
                        while (s + 1 < nseg && kc >= p.seg[s].kchunks) { kc -= p.seg[s].kchunks; ++s; }
                        const Seg& sg = p.seg[s];
                        mbar_wait(&empty_bar[st], ph ^ 1);
                        mbar_expect_tx(&full_bar[st], sg.a_tx4[g]);
                        tma_load_4d(smem_a + (size_t)st * a_bytes, &sg.tmA[g], &full_bar[st], sg.src_c + kc * sg.bk, w0 - (g & 1), h0 - (g >> 1), n0);
                        r += 4;
                        while (r >= K) { r -= K; ++g; }
                    }
                    __syncwarp();
                    stage += 4;
                    if (stage >= stage_hi) { stage -= ring_stages; phase ^= 1; }
                }
            } else
            for (int g = 0; g < groups; ++g) {
                int map = 0, cw, chh;
                if (halo == 3) {                  // stride 2: g = input parity (row parity * 2 + column parity); odd views start one earlier
                    map = g; cw = w0 - (g & 1); chh = h0 - (g >> 1);
                } else if (halo == 2) {           // the tile's whole halo box
                    cw = w0 - 1; chh = h0 - 1;
                } else if (halo) {                // g == kw: rows h0-1 .. h0+TH, columns w0+kw-1 .. +7
                    cw = w0 + g - 1; chh = h0 - 1;
                } else {
                    const int kh = g / ksz, kw = g % ksz;
                    if (stride == 1) {
                        cw = w0 + kw - pad; chh = h0 + kh - pad;
                    } else {
                        const int ih0 = kh - pad, iw0 = kw - pad;       // input = 2*out + i?0
                        const int ph = ih0 & 1, pw = iw0 & 1;
                        map = ph * 2 + pw;
                        chh = h0 + (ih0 - ph) / 2; cw = w0 + (iw0 - pw) / 2;
                    }
                }
                for (int s = 0; s < nseg; ++s) {
                    const Seg& sg = p.seg[s];
                    const int kchunks = sg.kchunks, bk = sg.bk, c_off = sg.c_off;
                    const uint32_t b_blk = sg.b_block_stride;
                    const uint32_t stage_tx = (halo == 3 ? sg.a_tx4[g] : sg.a_tx) + (b_res ? 0u : (uint32_t)taps_per_group * sg.b_block_bytes);
                    for (int kc = 0; kc < kchunks; ++kc) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        if (leader) {
                            mbar_expect_tx(&full_bar[stage], stage_tx);
                            if (sg.up == 2)     // (c, dup_w, w/2, dup_h, image*h_lo + h/2): zero-stride dims replicate each low-res pixel 2x2
                                tma_load_5d(smem_a + (size_t)stage * a_bytes, &sg.tmA[0], &full_bar[stage], sg.src_c + kc * bk, 0, cw >> 1, 0, n0 * sg.h_lo + (chh >> 1));
                            else
                                tma_load_4d(smem_a + (size_t)stage * a_bytes, &sg.tmA[map], &full_bar[stage], sg.src_c + kc * bk, cw, chh, n0);
                            if (!b_res) {
                                uint8_t* bdst = smem_b + (size_t)stage * b_stage_stride;
                                for (int t = 0; t < taps_per_group; ++t) {
                                    const int tap = halo == 2 ? t : halo ? t * 3 + g : g;
                                    tma_load_2d(bdst + (size_t)t * b_blk, &sg.tmB, &full_bar[stage], tap * Cin + c_off + kc * bk, n_idx * n_tile);
                                }
                            }
                        }
                        __syncwarp();
                        if (++stage == stage_hi) { stage = stage_lo; phase ^= 1; }
                    }
                }
            }
            if (MW == 2) {                                  // the next tile belongs to the other MMA warp: switch rings
                const int ts_ = stage; stage = ostage; ostage = ts_;
                const uint32_t tp_ = phase; phase = ophase; ophase = tp_;
                stage_lo = stage_lo ? 0 : ring_stages; stage_hi = stage_lo + ring_stages;
            }
        }
    } else if (warp <= kMmaWarps) {
        // ===================== MMA issuers (warps 1, 2) =====================
        // Measured (tools/cp_probe.cu): ONE issuing stream gets at most one tcgen05.mma per ~64 cycles whatever N is, two
        // streams together reach the operand-fetch rate (max(N/2, 32 + N/4) cycles per MMA per SM: 48 at N = 64).  Layers whose
        // resident weights leave room for one CTA per SM therefore run two issuing warps: warp r takes tiles r, r+2, ...,
        // owns accumulator stage r and its own ring of pipeline stages.
        // everything the issue loop computes with must be provably warp-uniform for the compiler (else it falls back to vector
        // registers + R2UR per MMA): the warp index comes through a shuffle (MW == 2) or is a constant (MW == 1)
        const int mw = MW == 1 ? 0 : (int)__reduce_max_sync(0xffffffffu, (unsigned)warp) - 1;      // REDUX: result lives in a uniform register
        pdl_wait();
        {
        const uint32_t leader = elect_one() ? 1u : 0u;
        const uint32_t tmem_base_u = __reduce_or_sync(0xffffffffu, tmem_base);
        // InstrDescriptor: c_format F32 (bit 4), a/b format BF16 (bits 7, 10), K-major A and B, N>>3 at 17, M>>4 at 24
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((128u >> 4) << 24);
        // shared-memory matrix descriptors: lo word = (address >> 4) | LBO field, hi word per segment
        const uint32_t a_lo0 = ((smem_u32(smem_a) >> 4) & 0x3FFFu) | (1u << 16);
        const uint32_t b_lo0 = ((smem_u32(smem_b) >> 4) & 0x3FFFu) | (1u << 16);
        const uint32_t a_stage16 = p.a_bytes >> 4, b_stage16 = p.b_stage_stride >> 4;
        constexpr int halo = HALO;
        const int b_res = p.b_resident, num_stages = p.num_stages, n_tile = p.n_tile;
        // per-segment constants in registers (nseg <= 2)
        int sg_kch[kMaxSeg], sg_mps[kMaxSeg];
        uint32_t sg_hi[kMaxSeg], sg_hiw[kMaxSeg], sg_hi9[kMaxSeg], sg_kh16[kMaxSeg], sg_blk16[kMaxSeg], sg_base16[kMaxSeg];
#pragma unroll
        for (int s = 0; s < kMaxSeg; ++s) {
            sg_kch[s] = s < nseg ? p.seg[s].kchunks : 0; sg_mps[s] = p.seg[s].bk >> 4;
            sg_hi[s] = p.seg[s].desc_hi; sg_hiw[s] = p.seg[s].desc_hi_w; sg_hi9[s] = p.seg[s].desc_hi9; sg_kh16[s] = p.seg[s].kh_step16;
            sg_blk16[s] = p.seg[s].b_block_stride >> 4; sg_base16[s] = p.seg[s].b_base >> 4;
        }
        constexpr bool two = MW == 2;
        const int ring_stages = two ? num_stages >> 1 : num_stages;
        const int stage_lo = mw * ring_stages, stage_hi = stage_lo + ring_stages;
        int stage = stage_lo; uint32_t phase = 0;
        int acc = mw; uint32_t acc_phase = 0;
        const int acc_stages = p.acc_stages;
        if (b_res) { mbar_wait_uniform(&bres_bar, 0); tc_fence_after(); }
        // CH: the chained GEMM of this warp's previous tile is issued right after the main MMAs of the current one -- by then
        // E1 has had a whole tile of tensor-pipe time to stage it, and the pipe never idles waiting for the epilogue
        const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.c2_n >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t smem_lo0 = smem_u32(smem);
        const int c2_nblk = p.c2_nblk;
        auto chain_issue = [&](int k) {
            const int buf = k & 1;
            const uint32_t par = (uint32_t)(k >> 1) & 1u;
            mbar_wait_uniform(&a2_full[buf], par);
            if (p.c2_nx) mbar_wait_uniform(&x_full[buf], par);
            mbar_wait_uniform(&t2_empty[buf], par ^ 1u);
            tc_fence_after();
            const uint32_t d2 = tmem_base_u + p.c2_tmem_col + (uint32_t)(buf * p.c2_n);
            uint32_t accum2 = 0;
            const uint32_t buf_lo = smem_lo0 + p.c2_buf_off + (uint32_t)buf * p.c2_buf_bytes, w_lo0 = smem_lo0 + p.c2_wreg_off;
            for (int i = 0; i < c2_nblk; ++i) {
                const uint32_t a_lo = (((buf_lo + p.c2_a_off[i]) >> 4) & 0x3FFFu) | (1u << 16);
                const uint32_t w_lo = (((w_lo0 + p.c2_w_off[i]) >> 4) & 0x3FFFu) | (1u << 16);
                const uint64_t hi = (uint64_t)p.c2_desc_hi[i] << 32;
                for (int j = 0; j < (p.c2_bk[i] >> 4); ++j) {
                    tc_mma_bf16_if(leader, d2, hi | (uint64_t)(a_lo + 2u * j), hi | (uint64_t)(w_lo + 2u * j), idesc2, accum2);
                    accum2 = 1;
                }
            }
            tc_commit_if(leader, &t2_full[buf]);
            tc_commit_if(leader, &a2_empty[buf]);
        };
        int it = 0;
        for (int tile = blockIdx.x + mw * gridDim.x; tile < total_tiles; tile += (two ? 2 : 1) * gridDim.x) {
            mbar_wait_uniform(&tempty_bar[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t d_addr = tmem_base_u + (uint32_t)(acc * n_tile);
            uint32_t accum = 0;
            for (int g = 0; g < groups; ++g) {
#pragma unroll
                for (int s = 0; s < kMaxSeg; ++s) {
                    const int kchunks = sg_kch[s], mma_per_step = sg_mps[s];
                    const uint64_t desc_hi = (uint64_t)sg_hi[s] << 32, desc_hi_w = (uint64_t)sg_hiw[s] << 32;
                    const uint32_t kh16 = sg_kh16[s], b_blk16 = sg_blk16[s], b_base16 = sg_base16[s];
                    for (int kc = 0; kc < kchunks; ++kc) {
                        mbar_wait_uniform(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t a_lo = a_lo0 + (uint32_t)stage * a_stage16;
                        if (halo == 3) {
                            // stride 2: this stage holds the (TW + pw) x (TH + ph) box of input parity (ph, pw) = (g >> 1, g & 1); it
                            // serves taps kh in {0, 2} (box rows 0 / 1) or {1}, kw likewise (kh16 = one row); resident weights
                            const int ph = g >> 1, pw = g & 1;
                            const uint64_t hi_a = pw ? (uint64_t)sg_hi9[s] << 32 : desc_hi_w;
                            const uint32_t row_pitch = (uint32_t)(8 + pw) * kh16;
                            for (int a = 0; a <= ph; ++a) {
                                const int kh = ph ? 2 * a : 1;
                                for (int c = 0; c <= pw; ++c) {
                                    const int kw = pw ? 2 * c : 1;
                                    const uint32_t ta_lo = a_lo + (uint32_t)a * row_pitch + (uint32_t)c * kh16;
                                    const uint32_t tb_lo = b_lo0 + b_base16 + (uint32_t)((kh * 3 + kw) * kchunks + kc) * b_blk16;
                                    for (int j = 0; j < mma_per_step; ++j) {
                                        tc_mma_bf16_if(leader, d_addr, hi_a | (ta_lo + 2u * j), desc_hi_w | (tb_lo + 2u * j), idesc, accum);
                                        accum = 1;
                                    }
                                }
                            }
                        } else if (halo == 2) {
                            // one box, nine taps, resident weights: block (tap, kc)
                            const uint32_t tb_lo = b_lo0 + b_base16 + (uint32_t)kc * b_blk16, tb_step = (uint32_t)kchunks * b_blk16;
                            if (mma_per_step == 4) ss_issue_halo2<4>(leader, d_addr, idesc, desc_hi, desc_hi_w, a_lo, tb_lo, tb_step, accum);
                            else if (mma_per_step == 2) ss_issue_halo2<2>(leader, d_addr, idesc, desc_hi, desc_hi_w, a_lo, tb_lo, tb_step, accum);
                            else ss_issue_halo2<1>(leader, d_addr, idesc, desc_hi, desc_hi_w, a_lo, tb_lo, tb_step, accum);
                        } else {
                            // tap mode (one tap per stage, tap g) / halo 1 (taps g, 3 + g, 6 + g of the stage's 18-row box); weights
                            // resident: block (tap, kc); streamed: the stage's own blocks.  K steps advance 32 bytes inside the
                            // swizzle atom: +2 in the >>4 address field.
                            const uint32_t tb_lo = b_res ? b_lo0 + b_base16 + (uint32_t)(g * kchunks + kc) * b_blk16 : b_lo0 + (uint32_t)stage * b_stage16;
                            const uint32_t b_step = b_res ? 3u * (uint32_t)kchunks * b_blk16 : b_blk16;
                            if (halo == 1) {
                                if (mma_per_step == 4) ss_issue_taps<4, 3>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                                else if (mma_per_step == 2) ss_issue_taps<2, 3>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                                else ss_issue_taps<1, 3>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                            } else {
                                if (mma_per_step == 4) ss_issue_taps<4, 1>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                                else if (mma_per_step == 2) ss_issue_taps<2, 1>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                                else ss_issue_taps<1, 1>(leader, d_addr, idesc, desc_hi, a_lo, tb_lo, b_step, accum);
                            }
                        }
                        tc_commit_if(leader, &empty_bar[stage]);     // frees the smem slot when these MMAs retire
                        if (++stage == stage_hi) { stage = stage_lo; phase ^= 1; }
                    }
                }
            }
            tc_commit_if(leader, &tfull_bar[acc]);               // accumulator complete -> epilogue
            acc += MW;
            if (acc >= acc_stages) { acc -= acc_stages; acc_phase ^= 1; }
            if (CH) { if (it > 0) chain_issue((it - 1) * MW + mw); ++it; }
        }
        if (CH && it > 0) chain_issue((it - 1) * MW + mw);
        }
    } else {
        // ===================== epilogue (warps 2..9) =====================
        pdl_wait();                                         // residual reads and output writes: after the predecessor grid
        const int quad = warp & 3;                          // TMEM lane quadrant this warp may read
        const int ew = warp - 1 - kMmaWarps;                // epilogue warp index; CH: the first kE1Warps drain the main accumulator
        const bool is_e1 = CH && ew < kE1Warps;
        constexpr int kSubR = CH ? kSub / 2 : kSub;         // warps of one role per lane quadrant
        const int half = (CH ? (ew % kE1Warps) : ew) >> 2;  // which of the kSubR warps of the quadrant
        const int row = quad * 32 + lane;                   // row of the 128-row tile == TMEM lane
        const int tw = row % p.TW, th = (row / p.TW) % p.TH, nb = row / (p.TW * p.TH);
        const int n_tiles = p.n_tiles, n_tile = p.n_tile, tiles_w = p.tiles_w, tiles_h = p.tiles_h, TW = p.TW, TH = p.TH, NB = p.NB;
        constexpr int epi = EPI;
        const int Wo = p.Wo, Ho = p.Ho, Bn = p.B, Cout = p.Cout, act = p.act, wide = p.wide;
        const int out_cstride = p.out_cstride, res_cstride = p.res_cstride;
        __nv_bfloat16* const out0 = p.out + p.out_coff;
        const __nv_bfloat16* const res0 = p.res ? p.res + p.res_coff : nullptr;
        int acc = 0; uint32_t acc_phase = 0; int par = 0;
        const int acc_stages = p.acc_stages;
        const uint32_t magic_nt = p.magic_nt, magic_tw = p.magic_tw, magic_th = p.magic_th;
        int kk = 0;                                         // CH: ordinal of the tile inside this CTA (buffer kk & 1, parity (kk >> 1) & 1)
        const uint32_t smem_lo = smem_u32(smem);
        // CH with TMA-fed K blocks (the channels the 1x1 conv reads besides this conv's output): one lane of the first E2 warp
        // loads them -- for tiles 0 and 1 up front, for tile kk + 2 as soon as the chained MMAs of tile kk have completed (which is
        // what this warp waits for anyway, and what frees staged-tile buffer kk & 1).  The producer warp never waits on the chain.
        const bool x_issuer = CH && p.c2_nx > 0 && ew == kE1Warps && lane == 0;
        auto x_load = [&](int t, int buf) {
            const int m0 = fast_div(t, magic_nt);
            const int m1 = fast_div(m0, magic_tw), m2 = fast_div(m1, magic_th);
            const int w0 = (m0 - m1 * tiles_w) * TW, h0 = (m1 - m2 * tiles_h) * TH, n0 = m2 * NB;
            mbar_expect_tx(&x_full[buf], p.c2_x_tx);
            for (int i = 0; i < p.c2_nx; ++i)
                tma_load_4d(smem + p.c2_buf_off + (size_t)buf * p.c2_buf_bytes + p.c2_a_off[i], &p.tmX[i], &x_full[buf], p.c2_src_c[i], w0, h0, n0);
        };
        if (x_issuer)
            for (int j = 0; j < 2; ++j) if ((int)blockIdx.x + j * (int)gridDim.x < total_tiles) x_load((int)blockIdx.x + j * (int)gridDim.x, j);
        // E1: this thread's first two chunks are half and half + kSubR (all of them when n_tile <= 32 kSubR); the swizzled shared-memory
        // address of a chunk's first 16-byte unit inside staged-tile buffer 0 is fixed for the whole kernel.  The second unit is
        // that address ^ 16 (a chunk starts at an even unit and the swizzle only XORs bits 4..6 with row bits); buffer 1 is
        // c2_buf_bytes, a multiple of 1024, further on (the swizzle bits do not change).
        uint32_t e1_pa = 0, e1_pb = 0;
        int e1_nq = 0;
        const uint32_t c2_buf_bytes = p.c2_buf_bytes;
        if (CH && is_e1) {
            const int nch1 = n_tile >> 4;                   // padding channels (>= Cout) carry zero weights and bias: they stage SiLU(0) = 0
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int jj = half + q * kSubR;
                if (jj < nch1) {
                    int bi = p.c2_nx;                       // chunk jj -> E1 block holding main channel 16 jj (blocks c2_nx.. are E1's, in channel order)
                    while (bi + 1 < p.c2_nblk && jj * 16 >= p.c2_src_c[bi + 1]) ++bi;
                    const uint32_t rb = (uint32_t)p.c2_bk[bi] * 2u, mask = (rb >> 4) - 1u;     // row bytes 128 / 64 / 32, swizzle mask 7 / 3 / 1
                    const uint32_t a0 = smem_lo + p.c2_buf_off + p.c2_a_off[bi] + (uint32_t)row * rb + ((uint32_t)(jj * 16 - p.c2_src_c[bi]) >> 3) * 16u;
                    const uint32_t pq = a0 ^ (((a0 >> 7) & mask) << 4);
                    if (q) e1_pb = pq; else e1_pa = pq;
                    e1_nq = q + 1;
                }
            }
        }
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++kk) {
            const int m0 = fast_div(tile, magic_nt), n_idx = tile - m0 * n_tiles;
            const int m1 = fast_div(m0, magic_tw), m2 = fast_div(m1, magic_th);
            const int w = (m0 - m1 * tiles_w) * TW + tw;
            const int h = (m1 - m2 * tiles_h) * TH + th;
            const int n = m2 * NB + nb;
            const bool valid = (w < Wo) && (h < Ho) && (n < Bn);
            const size_t pix = ((size_t)n * Ho + h) * Wo + w;
            const int n_base = n_idx * n_tile;
            __nv_bfloat16* optr = out0 + pix * out_cstride + n_base;
            const __nv_bfloat16* rptr = (res0 && (!CH || is_e1)) ? res0 + pix * res_cstride + n_base : nullptr;
            if (CH && is_e1) {
                // ===== E1: main accumulator -> bias / SiLU (+ shortcut) -> bf16 -> staged operand tile kk & 1 in shared memory =====
                const int buf = kk & 1;
                if (rptr && valid && e1_nq > 0) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rptr + half * 16));
                    if (e1_nq > 1) asm volatile("prefetch.global.L2 [%0];" ::"l"(rptr + (half + kSubR) * 16));
                }
                mbar_wait(&tfull_bar[acc], acc_phase);
                mbar_wait(&a2_empty[buf], ((uint32_t)(kk >> 1) & 1u) ^ 1u);     // the chained MMAs of tile kk - 2 have read this buffer
                tc_fence_after();
                const uint32_t t_addr1 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * n_tile) + (uint32_t)(half * 16);
                const uint32_t boff = buf ? c2_buf_bytes : 0u;
                const bool res_ok = rptr && valid;
                if (e1_nq > 0) {                            // (n_tile = 16: the second warp of a quadrant has no chunk, it only keeps the barriers' counts)
                    const bool two = e1_nq > 1;
                    uint32_t v0[16], v1[16];
                    tmem_ld16(t_addr1, v0);
                    if (two) tmem_ld16(t_addr1 + kSubR * 16, v1);
                    tmem_ld_wait();
                    const int c0 = half * 16, c1 = c0 + kSubR * 16;
                    epilogue_chunk_smem(v0, s_bias + c0, act, (res_ok && c0 < Cout) ? rptr + c0 : nullptr, e1_pa + boff, (e1_pa + boff) ^ 16u);
                    if (two) epilogue_chunk_smem(v1, s_bias + c1, act, (res_ok && c1 < Cout) ? rptr + c1 : nullptr, e1_pb + boff, (e1_pb + boff) ^ 16u);
                }
                // wider main convs (n_tile > 32 kSubR, e.g. the 80-channel class branch): further chunks, address worked out per tile
                for (int jj = half + 2 * kSubR; jj < (n_tile >> 4); jj += kSubR) {
                    uint32_t v0[16];
                    tmem_ld16(t_addr1 + (uint32_t)(jj - half) * 16u, v0);
                    tmem_ld_wait();
                    int bi = p.c2_nx;
                    while (bi + 1 < p.c2_nblk && jj * 16 >= p.c2_src_c[bi + 1]) ++bi;
                    const uint32_t rb = (uint32_t)p.c2_bk[bi] * 2u, mask = (rb >> 4) - 1u;
                    const uint32_t a0 = smem_lo + p.c2_buf_off + boff + p.c2_a_off[bi] + (uint32_t)row * rb + ((uint32_t)(jj * 16 - p.c2_src_c[bi]) >> 3) * 16u;
                    const uint32_t pq = a0 ^ (((a0 >> 7) & mask) << 4);
                    epilogue_chunk_smem(v0, s_bias + jj * 16, act, (res_ok && jj * 16 < Cout) ? rptr + jj * 16 : nullptr, pq, pq ^ 16u);
                }
                fence_proxy_async();                        // generic-proxy stores -> visible to the tensor core's async-proxy reads
                mbar_arrive(&a2_full[buf]);
                tc_fence_before();
                mbar_arrive(&tempty_bar[acc]);
                if (++acc == acc_stages) { acc = 0; acc_phase ^= 1; }
                continue;
            }
            const int ncols = CH ? p.c2_cout : min(n_tile, Cout - n_base);
            const int nchunks = (ncols + 15) >> 4;
            if (n_tiles > 1) {
                // per-tile bias slice (named barrier over the epilogue warps only)
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps));
                for (int i = threadIdx.x - 32 * (1 + kMmaWarps); i < n_tile; i += 32 * kEpiWarps) s_bias[i] = (n_base + i) < Cout ? __ldg(p.bias + n_base + i) * bias_scale : (EPI == 2 ? -INFINITY : 0.f);
                asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps));
            }

            // Bottleneck shortcut: pull this thread's residual chunks towards L2 while the tile's MMAs still run (no registers held)
            if (rptr && valid)
                for (int j = half; j < nchunks; j += kSubR) asm volatile("prefetch.global.L2 [%0];" ::"l"(rptr + j * 16));

            // final epilogue: the conv's own accumulator, or (CH) the chained accumulator kk & 1
            const float* const s_bias_f = CH ? s_bias2 : s_bias;
            const int act_f = CH ? p.c2_act : act;
            if (CH) {
                mbar_wait(&t2_full[kk & 1], (uint32_t)(kk >> 1) & 1u);
                if (x_issuer && tile + 2 * (int)gridDim.x < total_tiles) x_load(tile + 2 * (int)gridDim.x, kk & 1);
            } else mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (CH ? p.c2_tmem_col + (uint32_t)((kk & 1) * p.c2_n) : (uint32_t)(acc * n_tile));
            if (epi == 0) {
                // this warp's chunks: half, half + kSubR, half + 2 kSubR, ... ; two chunks in flight per iteration
                for (int j = half; j < nchunks; j += 2 * kSubR) {
                    const int j2 = j + kSubR;
                    const bool two = j2 < nchunks;
                    uint32_t v0[16], v1[16];
                    tmem_ld16(t_addr + j * 16, v0);
                    if (two) tmem_ld16(t_addr + j2 * 16, v1);
                    tmem_ld_wait();
                    if (valid) {
                        if (wide) {
                            epilogue_chunk<true>(v0, s_bias_f + j * 16, act_f, min(16, ncols - j * 16), optr + j * 16, rptr ? rptr + j * 16 : nullptr);
                            if (two) epilogue_chunk<true>(v1, s_bias_f + j2 * 16, act_f, min(16, ncols - j2 * 16), optr + j2 * 16, rptr ? rptr + j2 * 16 : nullptr);
                        } else {
                            epilogue_chunk<false>(v0, s_bias_f + j * 16, act_f, min(16, ncols - j * 16), optr + j * 16, rptr ? rptr + j * 16 : nullptr);
                            if (two) epilogue_chunk<false>(v1, s_bias_f + j2 * 16, act_f, min(16, ncols - j2 * 16), optr + j2 * 16, rptr ? rptr + j2 * 16 : nullptr);
                        }
                    }
                }
            } else if (epi == 1) {
                // DFL head: chunk j == box side j (l, t, r, b); this warp takes sides half and half + 2
                uint32_t v0[16], v1[16];
                tmem_ld16(t_addr + half * 16, v0);
                tmem_ld16(t_addr + (half + 2) * 16, v1);
                tmem_ld_wait();
                if (valid) {
                    float* o = p.out_f32 + pix * 4;
                    o[half] = dfl_side(v0, s_bias_f + half * 16);
                    o[half + 2] = dfl_side(v1, s_bias_f + (half + 2) * 16);
                }
            } else {
                // class head: the two warps of a lane quadrant take alternate pairs of 16-class chunks, then combine
                // through shared memory (double buffered by tile parity: one named barrier per tile and quadrant)
                int best = INT_MIN;
                for (int j = 2 * half; j < nchunks; j += 4) {
                    const bool two = j + 1 < nchunks;
                    uint32_t v0[16], v1[16];
                    tmem_ld16(t_addr + j * 16, v0);
                    if (two) tmem_ld16(t_addr + (j + 1) * 16, v1);
                    tmem_ld_wait();
                    cls_chunk(v0, s_bias_f + j * 16, j * 16, best);
                    if (two) cls_chunk(v1, s_bias_f + (j + 1) * 16, (j + 1) * 16, best);
                }
                const int key = best;
                int* const slot = &s_key[par][row];
                if (half) *slot = key;
                asm volatile("bar.sync %0, 64;" ::"r"(2 + quad) : "memory");
                if (!half && valid) *reinterpret_cast<float2*>(p.out_f32 + pix * 2) = cls_unkey(max(key, *slot));
            }
            tc_fence_before();
            if (CH) mbar_arrive(&t2_empty[kk & 1]);
            else {
                mbar_arrive(&tempty_bar[acc]);
                if (++acc == acc_stages) { acc = 0; acc_phase ^= 1; }
            }
            par ^= 1;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, p.tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
    });
    return fn;
}

CUtensorMapSwizzle swizzle_for(int bk) {
    return bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : bk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
}

inline size_t up1k(size_t v) { return (v + 1023) & ~(size_t)1023; }
constexpr size_t kOneCtaSmem = 220 * 1024;       // dynamic shared memory one CTA may plan with (227 KB - static - alignment slack)

}  // namespace

// Choose the (TW, TH, NB) patch (product 128, powers of two) that wastes the fewest tile slots.
void b2_pick_tile(int B, int Ho, int Wo, int* TW, int* TH, int* NB) {
    double best = -1; int bw = 16, bh = 8, bn = 1;
    for (int tw = 1; tw <= 128; tw *= 2)
        for (int th = 1; tw * th <= 128; th *= 2) {
            const int nb = 128 / (tw * th);
            const double slots = (double)b2_ceil_div(Wo, tw) * tw * b2_ceil_div(Ho, th) * th * b2_ceil_div(B, nb) * nb;
            double score = (double)B * Ho * Wo / slots;
            score += 1e-6 * tw - 1e-5 * nb;   // tie-break: wide rows, few images per tile
            if (score > best) { best = score; bw = tw; bh = th; bn = nb; }
        }
    *TW = bw; *TH = bh; *NB = bn;
}

struct B2ConvLaunch {
    ConvParams p;
    int grid;
    size_t smem;
};

size_t b2_conv_launch_size() { return sizeof(B2ConvLaunch); }

// One input of a convolution: channels [coff, coff+C) of an NHWC buffer with `cstride` channels per pixel, stored
// at full resolution (up = 1) or at half resolution (up = 2: nearest-2x upsample folded into the loads).
struct B2ConvSrc { const void* ptr; int cstride, coff, C, up; };
// A 1x1 conv chained onto the conv being prepared (ConvParams::chain): weights [Cout2][xC + Cout] (K order: the extra source's
// channels, then the main conv's), the extra source = channels [x_coff, x_coff + xC) of an NHWC buffer at the main conv's OUTPUT
// resolution (xsrc may be NULL: the 1x1 conv reads the main conv's output alone).
struct B2ConvChain { const void* w2; const float* bias2; int Cout2, act2; const void* xsrc; int x_cstride, x_coff, xC; };

// Build the launch descriptor (tensor maps + geometry) for a conv whose input is the channel concatenation of
// `nsrc` sources.  `storage` must hold b2_conv_launch_size() bytes, 64B aligned.  H x W: conv input resolution.
int b2_conv_prepare_chain(void* storage, const B2ConvSrc* srcs, int nsrc, int B, int H, int W,
                          const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                          void* out, int out_cstride, int out_coff, const void* residual, int res_cstride, int res_coff,
                          const B2ConvChain* chain);

int b2_conv_prepare_ms(void* storage, const B2ConvSrc* srcs, int nsrc, int B, int H, int W,
                       const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                       void* out, int out_cstride, int out_coff, const void* residual, int res_cstride, int res_coff) {
    return b2_conv_prepare_chain(storage, srcs, nsrc, B, H, W, w, bias, Cout, ksize, stride, act, out, out_cstride, out_coff,
                                 residual, res_cstride, res_coff, nullptr);
}

// `chain` != NULL: out / out_cstride / out_coff describe the CHAINED conv's output (Cout2 channels); B2_ERR_UNSUPPORTED when the
// pair does not fit the chained kernel's plan (the caller then launches the two convs separately).
static thread_local bool g_plan_only = false;     // b2_conv_chain_plan_ok: geometry / shared-memory plan only, no CUDA call

int b2_conv_prepare_chain(void* storage, const B2ConvSrc* srcs, int nsrc, int B, int H, int W,
                          const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                          void* out, int out_cstride, int out_coff, const void* residual, int res_cstride, int res_coff,
                          const B2ConvChain* chain) {
    const bool plan_only = g_plan_only;
    B2_REQUIRE(ksize == 1 || ksize == 3, "conv: ksize %d unsupported (1 or 3)", ksize);
    B2_REQUIRE(stride == 1 || stride == 2, "conv: stride %d unsupported (1 or 2)", stride);
    B2_REQUIRE(nsrc >= 1 && nsrc <= 2, "conv: 1 or 2 sources");
    int Cin = 0; bool any_up = false;
    for (int i = 0; i < nsrc; ++i) {
        const B2ConvSrc& sc = srcs[i];
        B2_REQUIRE(sc.ptr && sc.C > 0 && sc.C % 16 == 0, "conv: source %d: channels=%d must be a positive multiple of 16", i, sc.C);
        B2_REQUIRE(sc.cstride % 8 == 0 && sc.coff % 8 == 0 && (uintptr_t)sc.ptr % 16 == 0, "conv: channel strides/offsets must be multiples of 8 (16-byte TMA / vector alignment)");
        B2_REQUIRE(sc.up == 1 || sc.up == 2, "conv: source scale must be 1 or 2");
        if (sc.up == 2) { any_up = true; B2_REQUIRE(ksize == 1 && stride == 1 && H % 2 == 0 && W % 2 == 0, "conv: an upsampled source needs a 1x1 stride-1 conv on an even-sized map"); }
        Cin += sc.C;
    }
    B2_REQUIRE(out_cstride % 8 == 0 && out_coff % 8 == 0, "conv: channel strides/offsets must be multiples of 8 (16-byte TMA / vector alignment)");
    B2_REQUIRE(!residual || (res_cstride % 8 == 0 && res_coff % 8 == 0), "conv: residual stride/offset must be multiples of 8");
    B2_REQUIRE(Cout > 0 && B > 0 && H > 0 && W > 0, "conv: bad shape");
    B2_REQUIRE(((uintptr_t)out % 16 == 0) && ((uintptr_t)w % 16 == 0), "conv: pointers must be 16-byte aligned");
    if (!plan_only) {   // opt in to the large dynamic shared memory carve-out (not a stream operation: safe before graph capture).
        // The attribute belongs to the current device's context, so it is set on every plan (plan time, a few microseconds), not once
        // per process: a process that drives a second GPU would otherwise launch there without the opt-in.
        cudaError_t attr_err = cudaSuccess;
        {
            const int bytes = 227 * 1024 - 4096;
            cudaError_t e = cudaSuccess;
            auto set = [&](const void* fn) { cudaError_t r = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); if (r != cudaSuccess) e = r; };
            set((const void*)conv_tc_kernel<0, 0, 1>); set((const void*)conv_tc_kernel<0, 1, 1>); set((const void*)conv_tc_kernel<0, 2, 1>);
            set((const void*)conv_tc_kernel<0, 3, 1>); set((const void*)conv_tc_kernel<1, 0, 1>); set((const void*)conv_tc_kernel<2, 0, 1>);
            set((const void*)conv_tc_kernel<0, 2, 2>); set((const void*)conv_tc_kernel<0, 3, 2>);
            set((const void*)conv_tc_kernel<0, 2, 2, 16>); set((const void*)conv_tc_kernel<0, 3, 2, 16>);
            set((const void*)conv_tc_kernel<0, 2, 2, 16, 1>); set((const void*)conv_tc_kernel<0, 3, 2, 16, 1>);
            set((const void*)conv_tc_kernel<1, 2, 2, 16, 1>); set((const void*)conv_tc_kernel<2, 2, 2, 16, 1>);
            attr_err = e;
        }
        B2_CUDA(attr_err);
    }
    EncodeTiledFn encode = plan_only ? nullptr : get_encode();
    if (!plan_only && !encode) { b2_set_error("cuTensorMapEncodeTiled not available from the driver"); return B2_ERR_CUDA; }

    B2ConvLaunch* L = reinterpret_cast<B2ConvLaunch*>(storage);
    memset(L, 0, sizeof(*L));
    ConvParams& p = L->p;
    const int pad = ksize / 2;
    p.B = B; p.Ho = (H + 2 * pad - ksize) / stride + 1; p.Wo = (W + 2 * pad - ksize) / stride + 1;
    p.Cout = Cout; p.Cin = Cin; p.ksize = ksize; p.stride = stride; p.pad = pad;
    // 3x3 stride-1 "halo" mode: 8 x 16 pixel tiles; each (kw, K chunk) loads one 18-row box that serves the 3 kh taps
    p.halo = 0;
    if (ksize == 3 && stride == 1) {
        const double eff = (double)p.Wo * p.Ho / ((double)b2_ceil_div(p.Wo, 8) * 8 * b2_ceil_div(p.Ho, 16) * 16);
        if (eff >= 0.6) p.halo = 1;
    }
    if (p.halo) { p.TW = 8; p.TH = 16; p.NB = 1; }
    else if (any_up) {
        // tiles of one image, even extents (each low-resolution pixel is replicated 2x2 inside the box)
        double best = -1;
        for (int tw = 2; tw <= 64; tw *= 2) {
            const int th = 128 / tw;
            const double score = (double)p.Wo * p.Ho / ((double)b2_ceil_div(p.Wo, tw) * tw * b2_ceil_div(p.Ho, th) * th) + 1e-6 * tw;
            if (score > best) { best = score; p.TW = tw; p.TH = th; }
        }
        p.NB = 1;
    } else b2_pick_tile(B, p.Ho, p.Wo, &p.TW, &p.TH, &p.NB);
    p.tiles_w = b2_ceil_div(p.Wo, p.TW); p.tiles_h = b2_ceil_div(p.Ho, p.TH); p.tiles_nb = b2_ceil_div(B, p.NB);

    // ---- K segments: per source, 64-channel chunks, then the remainder in 32- or 16-channel chunks ----
    int a_rows = p.halo ? (p.TH + 2) * 8 : 128;
    const int taps = ksize * ksize;
    p.nseg = 0;
    int src_of[kMaxSeg];
    {
        int c_base = 0;
        for (int i = 0; i < nsrc; ++i) {
            const int n64 = srcs[i].C / 64, rem = srcs[i].C % 64;
            if (n64) { Seg& s = p.seg[p.nseg]; src_of[p.nseg++] = i; s.c_off = c_base; s.src_c = 0; s.bk = 64; s.kchunks = n64; }
            if (rem) { Seg& s = p.seg[p.nseg]; src_of[p.nseg++] = i; s.c_off = c_base + n64 * 64; s.src_c = n64 * 64; s.bk = (rem % 32 == 0) ? 32 : 16; s.kchunks = rem / s.bk; }
            c_base += srcs[i].C;
        }
    }
    int bk_max = 16;
    for (int si = 0; si < p.nseg; ++si) bk_max = p.seg[si].bk > bk_max ? p.seg[si].bk : bk_max;
    p.a_bytes = (uint32_t)up1k((size_t)a_rows * bk_max * 2);

    const int cout16 = b2_ceil_div(Cout, 16) * 16;
    // ---- chained 1x1 conv: K blocks (TMA-fed extra source first, then this conv's own channels), their shared-memory cost ----
    size_t chain_bytes = 0;
    int c2n = 0;
    if (chain) {
        B2_REQUIRE(chain->w2 && chain->bias2 && chain->Cout2 > 0 && (uintptr_t)chain->w2 % 16 == 0, "conv(chain): bad chained conv");
        B2_REQUIRE(!chain->xsrc || (chain->xC > 0 && chain->xC % 16 == 0 && chain->x_cstride % 8 == 0 && chain->x_coff % 8 == 0 && (uintptr_t)chain->xsrc % 16 == 0),
                   "conv(chain): extra source channels / strides must be multiples of 16 / 8");
        c2n = b2_ceil_div(chain->Cout2, 16) * 16;
        if (cout16 > 256 || c2n > 256 || ksize != 3 || any_up || nsrc != 1 || !(p.halo == 1 || stride == 2)) { b2_set_error("conv(chain): unsupported shape"); return B2_ERR_UNSUPPORTED; }
        p.chain = 1; p.c2_n = c2n; p.c2_cout = chain->Cout2; p.c2_act = chain->act2; p.c2_bias = chain->bias2;
        p.c2_nblk = 0; p.c2_nx = 0;
        uint32_t a_off = 0, w_off = 0;
        auto add_blocks = [&](int C, bool is_x) {
            int c = 0;
            while (c < C) {
                const int rem = C - c, bk = rem >= 64 ? 64 : (rem % 32 == 0 ? 32 : 16);
                if (p.c2_nblk >= kMaxChainBlk) return false;
                const int i = p.c2_nblk++;
                if (is_x) p.c2_nx = p.c2_nblk;
                p.c2_bk[i] = bk; p.c2_src_c[i] = c;
                p.c2_a_off[i] = a_off; a_off += (uint32_t)up1k((size_t)128 * bk * 2);
                p.c2_w_off[i] = w_off; w_off += (uint32_t)up1k((size_t)c2n * bk * 2);
                p.c2_w_bytes[i] = (uint32_t)c2n * bk * 2u;
                const uint32_t rb = (uint32_t)bk * 2u, swz = bk == 64 ? 2u : bk == 32 ? 4u : 6u;
                p.c2_desc_hi[i] = (((8u * rb) >> 4) & 0x3FFFu) | (1u << 14) | (swz << 29);
                c += bk;
            }
            return true;
        };
        if ((chain->xsrc && !add_blocks(chain->xC, true)) || !add_blocks(cout16, false)) { b2_set_error("conv(chain): too many K blocks"); return B2_ERR_UNSUPPORTED; }
        p.c2_buf_bytes = a_off;
        p.c2_x_tx = 0;
        for (int i = 0; i < p.c2_nx; ++i) p.c2_x_tx += 128u * (uint32_t)p.c2_bk[i] * 2u;
        chain_bytes = (size_t)w_off + 2 * (size_t)a_off;
    }
    const size_t one_cta_budget = kOneCtaSmem - chain_bytes;
    // ---- 3x3 stride 2 with resident weights: parity boxes (halo 3).  Each of the four (row, column) parity views of the
    //      input is loaded once per K chunk as a (8 + pw) x (16 + ph) box and serves every tap that reads it by
    //      descriptor start row: 561 box rows instead of 9 x 128 per tile and K chunk ----
    if (ksize == 3 && stride == 2 && nsrc == 1 && !any_up && Cout <= 256) {
        const double eff = (double)p.Wo * p.Ho / ((double)b2_ceil_div(p.Wo, 8) * 8 * b2_ceil_div(p.Ho, 16) * 16);
        size_t w_all = 0;
        for (int si = 0; si < p.nseg; ++si) w_all += (size_t)taps * p.seg[si].kchunks * up1k((size_t)b2_ceil_div(Cout, 16) * 16 * p.seg[si].bk * 2);
        const size_t a3 = up1k((size_t)9 * 17 * bk_max * 2);
        int mode3 = 1;
        if (const char* hv = getenv("B2_CONV_S2BOX")) mode3 = atoi(hv);
        if (mode3 && eff >= 0.6 && w_all + 3 * a3 <= one_cta_budget) {
            p.halo = 3; p.TW = 8; p.TH = 16; p.NB = 1;
            p.tiles_w = b2_ceil_div(p.Wo, p.TW); p.tiles_h = b2_ceil_div(p.Ho, p.TH); p.tiles_nb = b2_ceil_div(B, p.NB);
            a_rows = 9 * 17;
            p.a_bytes = (uint32_t)a3;
        }
    }

    // ---- resident-weight 3x3 stride-1 layers: single halo box per K chunk (halo 2) when the weights and enough box stages fit;
    //      decided on the resident footprint, which does not depend on the stage layout.  The shared-memory operand of
    //      tcgen05.mma may start at ANY row with ANY 8-row-group pitch (the swizzle is a function of the absolute address,
    //      DESIGN.md fact 3, profiles/r01_shift_probe.txt), so the tile's whole (TW+2) x (TH+2) box is loaded ONCE per K chunk
    //      (180 rows instead of 3 x 144) and serves all nine taps: tap (kh, kw) starts kh * (TW+2) + kw rows in, pitch TW+2 ----
    if (p.halo == 1 && cout16 <= 256) {
        size_t w_all = 0;
        for (int si = 0; si < p.nseg; ++si) w_all += (size_t)taps * p.seg[si].kchunks * up1k((size_t)cout16 * p.seg[si].bk * 2);
        const size_t a2 = up1k((size_t)(p.TW + 2) * (p.TH + 2) * bk_max * 2);
        int halo2_mode = 2;       // 1: only with three box stages (the rule before the two-stage plans were measured)
        if (const char* hv = getenv("B2_CONV_HALO2")) halo2_mode = atoi(hv);
        // three box stages, or two when the weights leave no room for a third (64 -> 144 at P2, 162 KB of weights: with two
        // issuing warps and a one-stage ring each, ring B loads tile i+1 while warp A works on tile i -- 0.69 ms against 0.77 ms
        // for the streamed-weight plan, tools/conv_bench.py)
        const size_t min_stages = halo2_mode >= 2 ? 2 : 3;
        if (halo2_mode && w_all + min_stages * a2 <= one_cta_budget) { p.halo = 2; a_rows = (p.TW + 2) * (p.TH + 2); p.a_bytes = (uint32_t)a2; }
    }
    const int tpg = p.halo == 2 ? 9 : p.halo == 1 ? 3 : 1;
    // ---- N tiling: streamed-weight stage = A box + tpg weight blocks; shrink the N tile until two stages fit ----
    int n_cap = 256;
    while (n_cap > 16 && p.halo < 2) {           // halo 2 / 3 imply resident weights: one N tile
        const int nt = cout16 < n_cap ? cout16 : n_cap;
        if (2 * (p.a_bytes + tpg * up1k((size_t)nt * bk_max * 2)) <= 200 * 1024) break;
        n_cap /= 2;
    }
    if (cout16 <= n_cap) { p.n_tiles = 1; p.n_tile = cout16; }
    else {
        p.n_tiles = b2_ceil_div(cout16, n_cap);
        p.n_tile = b2_ceil_div(b2_ceil_div(cout16, p.n_tiles), 16) * 16;
        p.n_tiles = b2_ceil_div(cout16, p.n_tile);
    }
    size_t b_all = 0;
    int steps_per_tile = 0;
    p.b_res_bytes = 0;
    uint32_t b_blk_max = 0;
    for (int si = 0; si < p.nseg; ++si) {
        Seg& s = p.seg[si];
        const uint32_t row_bytes = (uint32_t)s.bk * 2u;
        s.a_tx = (uint32_t)a_rows * row_bytes;
        s.b_block_bytes = (uint32_t)p.n_tile * row_bytes;
        s.b_block_stride = (uint32_t)up1k(s.b_block_bytes);
        b_blk_max = s.b_block_stride > b_blk_max ? s.b_block_stride : b_blk_max;
        s.b_base = (uint32_t)b_all;
        b_all += (size_t)taps * s.kchunks * s.b_block_stride;
        p.b_res_bytes += (uint32_t)(taps * s.kchunks) * s.b_block_bytes;
        s.kh_step16 = p.halo >= 2 ? row_bytes >> 4 : p.halo ? (8u * row_bytes) >> 4 : 0u;
        for (int m = 0; m < 4; ++m) s.a_tx4[m] = (uint32_t)((8 + (m & 1)) * (16 + (m >> 1))) * row_bytes;
        const uint32_t sbo = 8u * row_bytes, swz = s.bk == 64 ? 2u : s.bk == 32 ? 4u : 6u;   // UMMA layout type: 128B / 64B / 32B swizzle
        const uint32_t sbo_a = p.halo == 2 ? (uint32_t)(p.TW + 2) * row_bytes : sbo;        // pixel operand: 8-row groups (TW+2) rows apart in the halo box
        s.desc_hi = ((sbo_a >> 4) & 0x3FFFu) | (1u << 14) | (swz << 29);
        s.desc_hi_w = ((sbo >> 4) & 0x3FFFu) | (1u << 14) | (swz << 29);
        s.desc_hi9 = (((9u * row_bytes) >> 4) & 0x3FFFu) | (1u << 14) | (swz << 29);
        s.up = srcs[src_of[si]].up;
        s.h_lo = H / 2;
        steps_per_tile += (p.halo == 3 ? 4 : p.halo == 2 ? 1 : p.halo ? 3 : taps) * s.kchunks;
    }
    p.b_stage_stride = (uint32_t)tpg * b_blk_max;
    uint32_t cols = 2u * p.n_tile, pw = 32;
    while (pw < cols) pw <<= 1;
    p.tmem_cols = pw;

    // ---- shared memory plan: resident weights when they fit, 2 CTAs per SM when both fit ----
    const size_t kTwoCta = chain ? 0 : 106 * 1024, kOneCta = one_cta_budget;       // a chained conv runs one CTA per SM (16 epilogue warps)
    const size_t a_stage = p.a_bytes, ab_stage = a_stage + p.b_stage_stride;
    p.b_resident = 0;
    auto fit = [&](size_t budget, bool resident) {
        const size_t fixed = resident ? b_all : 0, per = resident ? a_stage : ab_stage;
        if (fixed + 2 * per > budget) return 0;
        size_t s_ = (budget - fixed) / per;
        return (int)(s_ > (size_t)kMaxStages ? kMaxStages : s_);
    };
    const bool can_res = p.n_tiles == 1;
    const bool tmem2 = p.tmem_cols * 2 <= 512;
    const int want = steps_per_tile < 4 ? 4 : (steps_per_tile < kMaxStages ? steps_per_tile : kMaxStages);   // >= one tile of look-ahead
    const int s2r = (can_res && tmem2) ? fit(kTwoCta, true) : 0, s2s = tmem2 ? fit(kTwoCta, false) : 0;
    const int s1r = can_res ? fit(kOneCta, true) : 0, s1s = fit(kOneCta, false);
    int ctas, stages;
    if (s2r >= 3) { ctas = 2; stages = s2r; p.b_resident = 1; }
    else if (s1r >= 3 || (p.halo == 2 && s1r >= 2)) { ctas = 1; stages = s1r; p.b_resident = 1; }
    else if (s2s >= 4) { ctas = 2; stages = s2s; }
    else { ctas = 1; stages = s1s; }
    int tmal = 4;                                       // B2_CONV_TMAL=1: stride-2 boxes issued one by one (experiments)
    if (const char* tv = getenv("B2_CONV_TMAL")) tmal = atoi(tv);
    const bool lanes3 = p.halo == 3 && tmal > 1;        // four fills per instruction want rings of >= 4 stages: keep every stage that fits
    if (!lanes3 && stages > want + 2 && stages > 4) stages = want + 2 > 4 ? want + 2 : 4;
    if (stages > kMaxStages) stages = kMaxStages;
    B2_REQUIRE(stages >= 2, "conv: tile does not fit in shared memory (Cin=%d Cout=%d k=%d)", Cin, Cout, ksize);
    // two MMA-issuing warps when each can have a ring of >= 2 stages (B2_CONV_MMAW=1 forces one)
    int mmaw = 2;
    if (const char* mv = getenv("B2_CONV_MMAW")) mmaw = atoi(mv);
    // measured: pays on the resident-weight single-box layers that run one CTA per SM (one issuing stream per SM otherwise);
    // streamed-weight layers lose more from the halved look-ahead of each ring than they gain
    // (a ring of ONE stage per issuing warp still double-buffers: ring B loads tile i+1 while warp A works on tile i)
    p.mma_warps = (mmaw >= 2 && (stages >= 4 || (p.halo == 2 && stages == 2)) && p.halo >= 2 && ctas == 1) ? 2 : 1;
    if (p.mma_warps == 2) stages &= ~1;
    p.num_stages = stages;
    p.halo3_k = 0;
    for (int si = 0; si < p.nseg; ++si) p.halo3_k += p.seg[si].kchunks;
    p.tma_lanes = (lanes3 && p.b_resident && (p.mma_warps == 2 ? stages / 2 : stages) >= 4) ? 4 : 1;
    p.epi_warps = 8;
    if (p.mma_warps == 2) {
        // measured (tools/conv_bench.py --ab B2_CONV_EPIW=8,16): 16 warps pay when a quadrant has more than four 16-column
        // chunks to drain or the epilogue also reads the shortcut tensor (80->80 3x3 at P2: 0.53 -> 0.47 ms); 8 otherwise
        p.epi_warps = (p.n_tile > 64 || residual) ? 16 : 8;
        if (const char* ev = getenv("B2_CONV_EPIW")) p.epi_warps = atoi(ev) == 8 ? 8 : atoi(ev) == 16 ? 16 : p.epi_warps;   // experiments only
    }
    if (chain) {
        // the chained kernel exists for resident weights, one CTA per SM, two issuing warps and 8 + 8 epilogue warps
        if (ctas != 1 || !p.b_resident || p.halo < 2 || p.mma_warps != 2 || p.n_tiles != 1 || 2 * p.n_tile + 2 * c2n > 512) {
            b2_set_error("conv(chain): plan not supported (ctas=%d resident=%d halo=%d mma_warps=%d n_tile=%d)", ctas, p.b_resident, p.halo, p.mma_warps, p.n_tile);
            return B2_ERR_UNSUPPORTED;
        }
        p.epi_warps = 16;
    }
    // accumulator stages: as many (<= kMaxAcc) as this CTA's share of the 512 tensor-memory columns holds -- the epilogue of a
    // tile is latency bound (tcgen05.ld -> SiLU -> stores), so the MMA warps need more than one tile of run-ahead
    {
        int acc = (512 - 2 * c2n) / ctas / p.n_tile;
        if (const char* av = getenv("B2_CONV_ACC")) { const int cap = atoi(av); if (cap >= 2 && cap < acc) acc = cap; }   // experiments only
        p.acc_stages = acc > kMaxAcc ? kMaxAcc : acc < 2 ? 2 : acc;
        if (p.mma_warps == 2 && (p.acc_stages & 1)) --p.acc_stages;
        uint32_t c2 = 32;
        while (c2 < (uint32_t)(p.acc_stages * p.n_tile + 2 * c2n)) c2 <<= 1;
        p.tmem_cols = c2;
        p.c2_tmem_col = (uint32_t)(p.acc_stages * p.n_tile);
    }
    L->smem = (size_t)stages * (p.b_resident ? a_stage : ab_stage) + (p.b_resident ? b_all : 0) + 1024;
    if (chain) {
        p.c2_wreg_off = (uint32_t)((size_t)stages * a_stage + b_all);
        p.c2_buf_off = (uint32_t)(p.c2_wreg_off + (chain_bytes - 2 * (size_t)p.c2_buf_bytes));
        if ((p.c2_buf_off | p.c2_buf_bytes) & 1023u) { b2_set_error("conv(chain): staged-tile buffers must be 1 KiB aligned"); return B2_ERR_UNSUPPORTED; }
        for (int i = 0; i < p.c2_nblk; ++i) p.b_res_bytes += p.c2_w_bytes[i];
        L->smem += chain_bytes;
    }
    p.out = (__nv_bfloat16*)out; p.out_cstride = out_cstride; p.out_coff = out_coff;
    p.res = (const __nv_bfloat16*)residual; p.res_cstride = res_cstride; p.res_coff = res_coff;
    p.bias = bias; p.act = act;
    p.wide = (out_cstride % 16 == 0 && out_coff % 16 == 0 && (uintptr_t)out % 32 == 0 &&
              (!residual || (res_cstride % 16 == 0 && res_coff % 16 == 0 && (uintptr_t)residual % 32 == 0))) ? 1 : 0;
    const int total_tiles = p.tiles_w * p.tiles_h * p.tiles_nb * p.n_tiles;
    {
        auto magic = [&](int d) -> uint32_t { return d == 1 ? 0u : (uint32_t)((((uint64_t)1 << 32) + (uint64_t)d - 1) / (uint64_t)d); };
        const int dmax = std::max(p.n_tiles, std::max(p.tiles_w, p.tiles_h));
        B2_REQUIRE((uint64_t)total_tiles * (uint64_t)dmax < ((uint64_t)1 << 32), "conv: %d tiles exceed the tile-index arithmetic", total_tiles);
        p.magic_nt = magic(p.n_tiles); p.magic_tw = magic(p.tiles_w); p.magic_th = magic(p.tiles_h);
    }
    const int slots = b2_num_sms() * ctas;
    L->grid = total_tiles < slots ? total_tiles : slots;
    if (const char* gv = getenv("B2_CONV_GRID")) { const int gcap = atoi(gv); if (gcap > 0 && gcap < L->grid) L->grid = gcap; }   // experiments only

    if (plan_only) return B2_OK;
    // ---- tensor maps ---------------------------------------------------------------------------------
    // L2 promotion of the activation boxes: 64 bytes.  Measured (ncu, 256 streams): with 128 B (or none) a conv that reads a 32-channel
    // slice of a 64-channel buffer (Bottleneck.cv1 inside the P2 C2f blocks) pulls the unused half of every 128-byte line from DRAM
    // (672 MB for a 336 MB input) and the single-box 64-channel layers re-fetch a third of their halo rows (64->64 + DFL at P2: 1175 MB
    // against 839 MB); the launches themselves take the same time, the power-capped step is 0.6 % shorter (tools/sustained.py)
    CUtensorMapL2promotion a_promo = CU_TENSOR_MAP_L2_PROMOTION_L2_64B;
    if (const char* pv = getenv("B2_CONV_L2PROMO")) {      // experiments only: 0 none, 1 64 B, 2 128 B, 3 256 B
        const int v = atoi(pv);
        a_promo = v == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : v == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : v == 3 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B : a_promo;
    }
    const int nmaps = stride == 1 ? 1 : 4;
    for (int si = 0; si < p.nseg; ++si) {
        Seg& s = p.seg[si];
        const B2ConvSrc& sc = srcs[src_of[si]];
        const CUtensorMapSwizzle sw = swizzle_for(s.bk);
        const char* base = (const char*)sc.ptr + (size_t)sc.coff * 2;
        const cuuint64_t cs2 = (cuuint64_t)sc.cstride * 2;
        if (sc.up == 2) {
            // (C, dup_w = 2, W/2, dup_h = 2, B*H/2) view of the half-resolution source: the two dup dims have stride 0,
            // so a box (bk, 2, TW/2, 2, TH/2) lands in shared memory as TH rows x TW pixels of the upsampled image.
            const int Wl = W / 2, Hl = H / 2;
            const cuuint64_t dims[5] = {(cuuint64_t)sc.C, 2, (cuuint64_t)Wl, 2, (cuuint64_t)B * Hl};
            const cuuint64_t strides[4] = {0, cs2, 0, (cuuint64_t)Wl * cs2};
            const cuuint32_t box[5] = {(cuuint32_t)s.bk, 2, (cuuint32_t)(p.TW / 2), 2, (cuuint32_t)(p.TH / 2)};
            const cuuint32_t es[5] = {1, 1, 1, 1, 1};
            CUresult r = encode(&s.tmA[0], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)base, dims, strides, box, es,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, a_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) { b2_set_error("cuTensorMapEncodeTiled(A upsampled, seg %d) failed with %d", si, (int)r); return B2_ERR_UNSUPPORTED; }
        } else {
            // A maps: (C, W', H', B) views of the NHWC input
            const cuuint32_t estr[4] = {1, 1, 1, 1};
            cuuint32_t box[4] = {(cuuint32_t)s.bk, (cuuint32_t)(p.halo == 2 ? p.TW + 2 : p.TW), (cuuint32_t)(p.halo == 1 || p.halo == 2 ? p.TH + 2 : p.TH), (cuuint32_t)p.NB};
            for (int m = 0; m < nmaps; ++m) {
                const int ph = m >> 1, pw_ = m & 1;
                if (p.halo == 3) { box[1] = (cuuint32_t)(p.TW + pw_); box[2] = (cuuint32_t)(p.TH + ph); }
                cuuint64_t dims[4], strides[3];
                const char* ptr = base;
                if (stride == 1) {
                    dims[0] = sc.C; dims[1] = W; dims[2] = H; dims[3] = B;
                    strides[0] = cs2; strides[1] = (cuuint64_t)W * cs2; strides[2] = (cuuint64_t)H * W * cs2;
                } else {
                    dims[0] = sc.C; dims[1] = (W - pw_ + 1) / 2; dims[2] = (H - ph + 1) / 2; dims[3] = B;
                    if (dims[1] == 0 || dims[2] == 0) { dims[1] = dims[1] ? dims[1] : 1; dims[2] = dims[2] ? dims[2] : 1; }
                    strides[0] = cs2 * 2; strides[1] = (cuuint64_t)W * cs2 * 2; strides[2] = (cuuint64_t)H * W * cs2;
                    ptr = base + ((size_t)ph * W + pw_) * cs2;
                }
                CUresult r = encode(&s.tmA[m], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)ptr, dims, strides, box, estr,
                                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw, a_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) { b2_set_error("cuTensorMapEncodeTiled(A, seg %d map %d) failed with %d", si, m, (int)r); return B2_ERR_CUDA; }
            }
        }
        // B map: weights [Cout][K] K-major
        const cuuint64_t K = (cuuint64_t)ksize * ksize * Cin;
        const cuuint64_t dimsb[2] = {K, (cuuint64_t)Cout};
        const cuuint64_t stridesb[1] = {K * 2};
        const cuuint32_t boxb[2] = {(cuuint32_t)s.bk, (cuuint32_t)p.n_tile};
        const cuuint32_t es[2] = {1, 1};
        CUresult r = encode(&s.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)w, dimsb, stridesb, boxb, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { b2_set_error("cuTensorMapEncodeTiled(B, seg %d) failed with %d", si, (int)r); return B2_ERR_CUDA; }
    }
    if (chain) {
        const cuuint64_t K2 = (cuuint64_t)((chain->xsrc ? chain->xC : 0) + Cout);
        int k0 = 0;
        for (int i = 0; i < p.c2_nblk; ++i) {
            const CUtensorMapSwizzle sw = swizzle_for(p.c2_bk[i]);
            // weights [Cout2][K2]: box (bk, c2_n) at K column k0 (columns / rows past the matrix are zero fill)
            const cuuint64_t dimsb[2] = {K2, (cuuint64_t)chain->Cout2};
            const cuuint64_t stridesb[1] = {K2 * 2};
            const cuuint32_t boxb[2] = {(cuuint32_t)p.c2_bk[i], (cuuint32_t)p.c2_n};
            const cuuint32_t es[2] = {1, 1};
            CUresult r = encode(&p.tmW2[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)chain->w2, dimsb, stridesb, boxb, es,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) { b2_set_error("cuTensorMapEncodeTiled(W2, block %d) failed with %d", i, (int)r); return B2_ERR_CUDA; }
            if (i < p.c2_nx) {
                // extra source: (C, Wo, Ho, B) view at the conv's output resolution, the tile's own pixels
                const char* base = (const char*)chain->xsrc + (size_t)chain->x_coff * 2;
                const cuuint64_t cs2 = (cuuint64_t)chain->x_cstride * 2;
                const cuuint64_t dims[4] = {(cuuint64_t)chain->xC, (cuuint64_t)p.Wo, (cuuint64_t)p.Ho, (cuuint64_t)B};
                const cuuint64_t strides[3] = {cs2, (cuuint64_t)p.Wo * cs2, (cuuint64_t)p.Ho * p.Wo * cs2};
                const cuuint32_t box[4] = {(cuuint32_t)p.c2_bk[i], (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.NB};
                const cuuint32_t estr[4] = {1, 1, 1, 1};
                r = encode(&p.tmX[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, sw, a_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) { b2_set_error("cuTensorMapEncodeTiled(X, block %d) failed with %d", i, (int)r); return B2_ERR_CUDA; }
            }
            k0 += p.c2_bk[i];
        }
        (void)k0;
    }
    return B2_OK;
}

int b2_conv_prepare(void* storage, const void* in, int B, int H, int W, int in_cstride, int in_coff, int Cin,
                    const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                    void* out, int out_cstride, int out_coff, const void* residual, int res_cstride, int res_coff) {
    B2_REQUIRE(Cin % 16 == 0 && Cin > 0, "conv: Cin=%d must be a positive multiple of 16", Cin);
    const B2ConvSrc src{in, in_cstride, in_coff, Cin, 1};
    return b2_conv_prepare_ms(storage, &src, 1, B, H, W, w, bias, Cout, ksize, stride, act, out, out_cstride, out_coff, residual, res_cstride, res_coff);
}

// Switch a prepared conv to a fused Detect-head epilogue (see ConvParams::epi).
int b2_conv_set_head_epilogue(void* storage, int epi, float* out_f32) {
    B2ConvLaunch* L = reinterpret_cast<B2ConvLaunch*>(storage);
    B2_REQUIRE(epi == 1 || epi == 2, "conv: head epilogue mode must be 1 (DFL) or 2 (classes)");
    if (L->p.chain) {          // the head epilogue runs on the chained 1x1 conv's accumulator
        B2_REQUIRE((epi != 1 || L->p.c2_cout == 64) && out_f32 && L->p.halo == 2, "conv(chain): head epilogue needs a 3x3 stride-1 main conv (DFL: exactly 64 channels)");
        L->p.epi = epi; L->p.out_f32 = out_f32;
        return B2_OK;
    }
    B2_REQUIRE(L->p.n_tiles == 1 && (epi != 1 || L->p.Cout == 64) && out_f32, "conv: head epilogue needs one N tile (DFL: exactly 64 channels)");
    B2_REQUIRE(L->p.halo == 0, "conv: head epilogues are implemented for 1x1 convs in conv_tc_kernel only");
    L->p.mma_warps = 1;
    L->p.epi = epi; L->p.out_f32 = out_f32;
    return B2_OK;
}

void b2_count_launch(int n);

int b2_conv_launch(const void* storage, cudaStream_t stream) {
    const B2ConvLaunch* L = reinterpret_cast<const B2ConvLaunch*>(storage);
    // programmatic dependent launch: this grid's prologue overlaps the tail of the previous kernel of the stream when that
    // kernel is a conv_tc_kernel too (it calls griddepcontrol.launch_dependents); otherwise the attribute changes nothing
    static const bool pdl = [] { const char* v = getenv("B2_CONV_PDL"); return !(v && atoi(v) == 0); }();
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)L->grid); cfg.dynamicSmemBytes = L->smem; cfg.stream = stream;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    auto go = [&](auto kernel, int threads) { cfg.blockDim = dim3((unsigned)threads); return cudaLaunchKernelEx(&cfg, kernel, L->p); };
    cudaError_t e;
    if (L->p.chain) {
        constexpr int kThreadsChain = kThreadsMw2 + 256;
        if (L->p.epi == 1) e = go(conv_tc_kernel<1, 2, 2, 16, 1>, kThreadsChain);
        else if (L->p.epi == 2) e = go(conv_tc_kernel<2, 2, 2, 16, 1>, kThreadsChain);
        else if (L->p.halo == 3) e = go(conv_tc_kernel<0, 3, 2, 16, 1>, kThreadsChain);
        else e = go(conv_tc_kernel<0, 2, 2, 16, 1>, kThreadsChain);
    }
    else if (L->p.epi == 1) e = go(conv_tc_kernel<1, 0, 1>, kThreadsMw1);
    else if (L->p.epi == 2) e = go(conv_tc_kernel<2, 0, 1>, kThreadsMw1);
    else if (L->p.mma_warps == 2 && L->p.halo == 3 && L->p.epi_warps == 16) e = go(conv_tc_kernel<0, 3, 2, 16>, kThreadsMw2 + 256);
    else if (L->p.mma_warps == 2 && L->p.epi_warps == 16) e = go(conv_tc_kernel<0, 2, 2, 16>, kThreadsMw2 + 256);
    else if (L->p.mma_warps == 2 && L->p.halo == 3) e = go(conv_tc_kernel<0, 3, 2>, kThreadsMw2);
    else if (L->p.mma_warps == 2) e = go(conv_tc_kernel<0, 2, 2>, kThreadsMw2);
    else if (L->p.halo == 3) e = go(conv_tc_kernel<0, 3, 1>, kThreadsMw1);
    else if (L->p.halo == 2) e = go(conv_tc_kernel<0, 2, 1>, kThreadsMw1);
    else if (L->p.halo == 1) e = go(conv_tc_kernel<0, 1, 1>, kThreadsMw1);
    else e = go(conv_tc_kernel<0, 0, 1>, kThreadsMw1);
    B2_CUDA(e);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_conv2d_bf16(const void* in, int B, int H, int W, int in_cstride, int in_coff, int Cin,
                              const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                              void* out, int out_cstride, int out_coff,
                              const void* residual, int res_cstride, int res_coff, void* stream) {
    alignas(64) unsigned char storage[sizeof(B2ConvLaunch)];
    int rc = b2_conv_prepare(storage, in, B, H, W, in_cstride, in_coff, Cin, w, bias, Cout, ksize, stride, act,
                             out, out_cstride, out_coff, residual, res_cstride, res_coff);
    if (rc != B2_OK) return rc;
    return b2_conv_launch(storage, (cudaStream_t)stream);
}

// Conv over the channel concatenation of two inputs (Concat folded into the conv; yolov8-p2.yaml:33-54):
// in1 may be stored at half resolution (up1 = 2: nn.Upsample(None, 2, 'nearest') folded into the TMA loads).
extern "C" int b2_conv2d_cat_bf16(const void* in0, int cstride0, int coff0, int C0, int up0,
                                  const void* in1, int cstride1, int coff1, int C1, int up1,
                                  int B, int H, int W, const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                                  void* out, int out_cstride, int out_coff, void* stream) {
    alignas(64) unsigned char storage[sizeof(B2ConvLaunch)];
    const B2ConvSrc srcs[2] = {{in0, cstride0, coff0, C0, up0}, {in1, cstride1, coff1, C1, up1}};
    int rc = b2_conv_prepare_ms(storage, srcs, in1 ? 2 : 1, B, H, W, w, bias, Cout, ksize, stride, act, out, out_cstride, out_coff, nullptr, 0, 0);
    if (rc != B2_OK) return rc;
    return b2_conv_launch(storage, (cudaStream_t)stream);
}

// Conv (3x3, BN folded, SiLU, optional shortcut) immediately followed by a 1x1 conv (+ SiLU) that reads the first conv's output
// -- optionally concatenated behind `xC` channels of another tensor -- as ONE launch: the intermediate tile stays in shared
// memory (ConvParams::chain).  Covers Conv -> C2f.cv1 (nn/tasks.py:172-188 + block.py:315-316), Bottleneck.cv2 -> C2f.cv2
// (block.py:317-319, :493-495) and Detect's 3x3 -> 1x1 tails (head.py:93-100).  w2: [Cout2][xC + Cout] bf16.
// Returns B2_ERR_UNSUPPORTED when the pair does not fit the chained kernel (run the two convs separately then).
extern "C" int b2_conv2d_chain_bf16(const void* in, int B, int H, int W, int in_cstride, int in_coff, int Cin,
                                    const void* w, const float* bias, int Cout, int ksize, int stride, int act,
                                    const void* residual, int res_cstride, int res_coff,
                                    const void* xsrc, int x_cstride, int x_coff, int xC,
                                    const void* w2, const float* bias2, int Cout2, int act2,
                                    void* out, int out_cstride, int out_coff, void* stream) {
    B2_REQUIRE(Cin % 16 == 0 && Cin > 0, "conv: Cin=%d must be a positive multiple of 16", Cin);
    alignas(64) unsigned char storage[sizeof(B2ConvLaunch)];
    const B2ConvSrc src{in, in_cstride, in_coff, Cin, 1};
    const B2ConvChain ch{w2, bias2, Cout2, act2, xsrc, x_cstride, x_coff, xC};
    int rc = b2_conv_prepare_chain(storage, &src, 1, B, H, W, w, bias, Cout, ksize, stride, act, out, out_cstride, out_coff,
                                   residual, res_cstride, res_coff, &ch);
    if (rc != B2_OK) return rc;
    return b2_conv_launch(storage, (cudaStream_t)stream);
}

// 1 if b2_conv2d_chain_bf16 would accept this pair (pure planning: callable without a CUDA device), else 0.
extern "C" int b2_conv_chain_plan_ok(int B, int H, int W, int Cin, int Cout, int ksize, int stride, int has_residual, int xC, int Cout2) {
    alignas(64) unsigned char storage[sizeof(B2ConvLaunch)];
    alignas(64) static unsigned char dummy[64];
    const B2ConvSrc src{dummy, ((Cin + 15) / 16) * 16, 0, Cin, 1};
    const B2ConvChain ch{dummy, (const float*)dummy, Cout2, 1, xC > 0 ? (const void*)dummy : nullptr, ((xC + 15) / 16) * 16, 0, xC};
    if (Cin <= 0 || Cin % 16 || Cout <= 0 || Cout2 <= 0 || xC < 0 || xC % 16) return 0;
    g_plan_only = true;
    const int rc = b2_conv_prepare_chain(storage, &src, 1, B, H, W, dummy, (const float*)dummy, Cout, ksize, stride, 1, dummy, ((Cout2 + 15) / 16) * 16, 0,
                                         has_residual ? dummy : nullptr, ((Cout + 15) / 16) * 16, 0, &ch);
    g_plan_only = false;
    return rc == B2_OK ? 1 : 0;
}
