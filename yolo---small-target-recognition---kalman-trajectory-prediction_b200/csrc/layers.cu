// Bandwidth-shaped layer kernels of the detect path (sm_100a): stem conv on raw uint8 frames, SPPF pooling,
// nearest-2x upsample / concat slice copy, stand-alone preprocess.  All NHWC bf16, 16-byte vector accesses.
#include "common.cuh"

#include <stdlib.h>

void b2_count_launch(int n);

namespace {

// ------------------------------------------------------------------------------------------------
// Stem: LetterBox pad (114) + BGR->RGB + /255 (engine/predictor.py:152-175, data/augment.py:1717-1728)
// fused with model.0 = Conv(3 -> C0, k3, s2) + SiLU, on the tensor cores.
//
// Implicit GEMM with K = 27 (padded to 32): each of the 128 threads of a CTA builds the im2col row of ONE output
// pixel (27 uint8 pixel values, exact in bf16) directly in shared memory in the SWIZZLE_64B K-major UMMA layout,
// one thread issues two tcgen05.mma (M=128, N=C0, K=16) against the resident bf16 weight tile, and the same 128
// threads read their accumulator row back from TMEM (thread r <-> TMEM lane r), apply 1/255 and the folded bias
// in fp32, SiLU, and store C0 bf16 channels.  Several CTAs per SM overlap load / MMA / epilogue phases.
//
// uint8 frames (Loader::kMagic): no integer -> float conversion at all.  The operand is FP16 and byte n is stored as
// 0x6400 | n == 1024 + n (exact: one PRMT makes two operands), the weights are the bf16 weights converted to FP16, and
// the constant 1024 * sum_k w[n][k] is taken out again through the bias in the fp32 epilogue.  The im2col row is laid out
// as the bytes lie in memory -- K index = kh * 10 + kw * 3 + c (c in B, G, R order, index 9 of every kh a zero weight) --
// so a row is three runs of 10 consecutive frame bytes: 3 aligned word loads, 3 funnel shifts and 5 PRMT per run.
// ------------------------------------------------------------------------------------------------
#ifndef B2_STEM_CTAS
#define B2_STEM_CTAS 8          // co-resident stem CTAs per SM the register budget is set for (experiment builds: 10, 12)
#endif
constexpr int kStemThreads = 128;
constexpr int kStemMaxC0 = 128;
constexpr int kStemPitch = 144;          // bytes between staged patch rows (16-byte multiple, not a multiple of 128: rows 2 apart hit other banks)

__device__ __forceinline__ uint32_t swz64_chunk_off(int row, int chunk) {   // byte offset of 16-byte chunk `chunk` of 64-byte row `row`
    return (uint32_t)row * 64u + (uint32_t)((chunk ^ ((row >> 1) & 3)) << 4);
}

template <typename Loader>
__global__ void __launch_bounds__(kStemThreads, B2_STEM_CTAS) stem_tc_kernel(Loader ld, int B, int H, int W, int Ho, int Wo,
                                                               const __nv_bfloat16* __restrict__ w, const float* __restrict__ bias,
                                                               float in_scale, int C0, int n_tile, uint32_t tmem_cols,
                                                               __nv_bfloat16* __restrict__ out, int out_cstride, int out_coff,
                                                               int tiles_w, int tiles_h, int total_tiles) {
    __shared__ __align__(1024) uint8_t s_a[128 * 64];
    __shared__ __align__(1024) uint8_t s_b[kStemMaxC0 * 64];
    __shared__ __align__(16) float s_bias[kStemMaxC0];
    __shared__ __align__(16) uint8_t s_in[17 * kStemPitch + 32];      // staged input patch: 17 rows x kStemPitch bytes, then the 17 row offsets (0..15)
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { mbar_init(&s_bar, 1); fence_mbar_init(); }
    if (warp == 0) { tmem_alloc(&s_tmem, tmem_cols); tmem_relinquish(); }
    // weights [C0][32] bf16 (k = (kh*3+kw)*3 + c_rgb, 27..31 zero) -> swizzled 64-byte rows; rows >= C0 zero
    constexpr bool kMagic = Loader::kMagic;
    for (int i = tid; i < n_tile * 4; i += kStemThreads) {
        const int n = i >> 2, c = i & 3;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (n < C0) {
            if (!kMagic) v = *reinterpret_cast<const uint4*>(w + (size_t)n * 32 + c * 8);
            else {
                // FP16 copy in memory-byte order: k' = kh * 10 + kw * 3 + c_mem  <-  k = (kh * 3 + kw) * 3 + (2 - c_mem)
                uint32_t h[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int kp = c * 8 + e, kh = kp / 10, j = kp - kh * 10;
                    float x = 0.f;
                    if (kp < 30 && j < 9) x = __bfloat162float(w[(size_t)n * 32 + (kh * 3 + j / 3) * 3 + (2 - j % 3)]);
                    h[e] = (uint32_t)__half_as_ushort(__float2half_rn(x));
                }
                v = make_uint4(h[0] | (h[1] << 16), h[2] | (h[3] << 16), h[4] | (h[5] << 16), h[6] | (h[7] << 16));
            }
        }
        *reinterpret_cast<uint4*>(s_b + swz64_chunk_off(n, c)) = v;
    }
    // s_bias holds HALF the effective bias (SiLU(x) = h + h tanh(h), h = x / 2 comes out of one FFMA); kMagic: the
    // 1024 carried by every operand is removed here: x = in_scale * (acc - 1024 * sum_k w16[k]) + bias
    for (int i = tid; i < n_tile; i += kStemThreads) {
        float b = 0.f;
        if (i < C0) {
            b = bias[i];
            if (kMagic) {
                float sw = 0.f;
                for (int k = 0; k < 27; ++k) sw += __half2float(__float2half_rn(__bfloat162float(w[(size_t)i * 32 + k])));
                b -= in_scale * 1024.f * sw;
            }
        }
        s_bias[i] = 0.5f * b;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    // c_format F32 (bit 4); a/b format BF16 (1 at bits 7, 10) or F16 (0)
    const uint32_t idesc = (1u << 4) | (kMagic ? 0u : (1u << 7) | (1u << 10)) | ((uint32_t)(n_tile >> 3) << 17) | ((128u >> 4) << 24);
    const float half_scale = 0.5f * in_scale;
    const uint64_t desc_hi = (uint64_t)(((512u >> 4) & 0x3FFFu) | (1u << 14) | (4u << 29)) << 32;   // SBO = 8 rows x 64 B, SWIZZLE_64B
    const uint32_t a_lo = ((smem_u32(s_a) >> 4) & 0x3FFFu) | (1u << 16), b_lo = ((smem_u32(s_b) >> 4) & 0x3FFFu) | (1u << 16);
    const int tw = tid & 15, th = tid >> 4;                 // 16 x 8 output pixels per tile
    uint32_t phase = 0;
    // tile -> (column cx, row cy, image cb) once, then advanced by the grid stride in mixed radix: no division per tile (the
    // divisions, 64-bit patch addresses and coordinate products were most of the 560 instructions a warp spent per tile -- ncu:
    // 59 % of the issue slots, 136 of them the arithmetic of the layer)
    const int tpi = tiles_w * tiles_h;
    int cb = (int)blockIdx.x / tpi, cy = ((int)blockIdx.x - cb * tpi) / tiles_w, cx = (int)blockIdx.x - cb * tpi - cy * tiles_w;
    const int sb = (int)gridDim.x / tpi, sy = ((int)gridDim.x - sb * tpi) / tiles_w, sx = (int)gridDim.x - sb * tpi - sy * tiles_w;
    auto advance = [&](int& x, int& y, int& b_) {
        x += sx; if (x >= tiles_w) { x -= tiles_w; y += 1; }
        y += sy; if (y >= tiles_h) { y -= tiles_h; b_ += 1; }
        b_ += sb;
    };
    int nx = cx, ny = cy, nb = cb;
    advance(nx, ny, nb);
    // patch of the first tile (see LoadU8::fetch)
    typename Loader::Patch pp;
    const int roff = ld.row_offset(tid);
    bool pok = false;
    if (Loader::kStaged && (int)blockIdx.x < total_tiles) pok = ld.fetch(cb, 16 * cy - 1, 32 * cx - 1, tid, roff, pp);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int wo = cx * 16 + tw, ho = cy * 8 + th, b = cb;
        // ---- im2col row of this thread's pixel ----
        bool staged = false;
        uint32_t pk[16];
        if (Loader::kStaged) {
            // Interior tiles of uint8 frames: the 17 x 33-pixel input patch (99 bytes per row) is copied into shared memory
            // with aligned 16-byte loads (<= 8 per row; one or two per thread) and each thread then takes its three runs of
            // 10 bytes from there -- 136 vector loads and no per-byte bounds checks instead of 3456 byte loads per tile.
            staged = pok;                                                                        // uniform across the CTA
            if (staged) ld.commit(s_in, tid, pp);
            {   // loads of the next tile's patch: consumed at the top of the next iteration
                pok = false;
                if (tile + (int)gridDim.x < total_tiles) pok = ld.fetch(nb, 16 * ny - 1, 32 * nx - 1, tid, roff, pp);
            }
            if (staged) {
                __syncthreads();
#pragma unroll
                for (int kh = 0; kh < 3; ++kh) {
                    const int r = 2 * th + kh;
                    const uint32_t e = (uint32_t)s_in[17 * kStemPitch + r] + 6u * (uint32_t)tw;      // first byte of the run
                    const uint32_t* q = reinterpret_cast<const uint32_t*>(s_in + r * kStemPitch + (e & ~3u));
                    const uint32_t w0 = q[0], w1 = q[1], w2 = q[2], sh = (e & 3u) * 8u;
                    const uint32_t a0 = __funnelshift_r(w0, w1, sh), a1 = __funnelshift_r(w1, w2, sh), a2 = w2 >> sh;
                    pk[kh * 5 + 0] = __byte_perm(a0, 0x64646464u, 0x4140);     // {1024 + b0, 1024 + b1} as two FP16
                    pk[kh * 5 + 1] = __byte_perm(a0, 0x64646464u, 0x4342);
                    pk[kh * 5 + 2] = __byte_perm(a1, 0x64646464u, 0x4140);
                    pk[kh * 5 + 3] = __byte_perm(a1, 0x64646464u, 0x4342);
                    pk[kh * 5 + 4] = __byte_perm(a2, 0x64646464u, 0x4140);     // b9 belongs to the next pixel: its weight is zero
                }
                pk[15] = 0u;
            }
        }
        if (!staged) {
            float v[27];
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) {
                    float rgb[3];
                    ld.load(b, 2 * ho + kh - 1, 2 * wo + kw - 1, H, W, rgb);
                    v[(kh * 3 + kw) * 3 + 0] = rgb[0]; v[(kh * 3 + kw) * 3 + 1] = rgb[1]; v[(kh * 3 + kw) * 3 + 2] = rgb[2];
                }
            if (kMagic) {
                // integer-valued 0..255 floats -> 0x6400 | n, in memory-byte order (B, G, R)
#pragma unroll
                for (int kh = 0; kh < 3; ++kh)
#pragma unroll
                    for (int i = 0; i < 5; ++i) {
                        const int j0 = 2 * i, j1 = 2 * i + 1;
                        const uint32_t lo = 0x6400u | (uint32_t)v[(kh * 3 + j0 / 3) * 3 + (2 - j0 % 3)];
                        const uint32_t hi = j1 < 9 ? 0x6400u | (uint32_t)v[(kh * 3 + j1 / 3) * 3 + (2 - j1 % 3)] : 0x6400u;
                        pk[kh * 5 + i] = lo | (hi << 16);
                    }
                pk[15] = 0u;
            } else {
#pragma unroll
                for (int i = 0; i < 13; ++i) pk[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
                pk[13] = pack_bf16x2(v[26], 0.f); pk[14] = 0u; pk[15] = 0u;
            }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
            *reinterpret_cast<uint4*>(s_a + swz64_chunk_off(tid, c)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        fence_proxy_async();                                 // generic-proxy writes -> visible to the tensor core (async proxy)
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            tc_mma_bf16(tmem, desc_hi | a_lo, desc_hi | b_lo, idesc, 0u);
            tc_mma_bf16(tmem, desc_hi | (a_lo + 2u), desc_hi | (b_lo + 2u), idesc, 1u);
            tc_commit(&s_bar);
        }
        mbar_wait(&s_bar, phase);
        phase ^= 1;
        tc_fence_after();
        const bool valid = wo < Wo && ho < Ho;
        __nv_bfloat16* op = out + (size_t)((b * Ho + ho) * Wo + wo) * out_cstride + out_coff;        // B * Ho * Wo < 2^31 (checked on the host)
        const uint32_t t_addr = tmem + ((uint32_t)(warp * 32) << 16);
        for (int j = 0; j < n_tile; j += 16) {
            uint32_t a[16];
            tmem_ld16(t_addr + j, a);
            tmem_ld_wait();
            if (valid) {
                uint32_t o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float h0 = fmaf(__uint_as_float(a[2 * i]), half_scale, s_bias[j + 2 * i]);
                    const float h1 = fmaf(__uint_as_float(a[2 * i + 1]), half_scale, s_bias[j + 2 * i + 1]);
                    o[i] = pack_bf16x2(silu_half(h0), silu_half(h1));
                }
                if (j + 16 <= C0) {
                    *reinterpret_cast<uint4*>(op + j) = make_uint4(o[0], o[1], o[2], o[3]);
                    *reinterpret_cast<uint4*>(op + j + 8) = make_uint4(o[4], o[5], o[6], o[7]);
                } else if (j + 8 <= C0) {
                    *reinterpret_cast<uint4*>(op + j) = make_uint4(o[0], o[1], o[2], o[3]);
                }
            }
        }
        tc_fence_before();
        __syncthreads();                                     // accumulator and A tile are free for the next tile
        cx = nx; cy = ny; cb = nb;
        advance(nx, ny, nb);
    }
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem, tmem_cols); }
}

struct LoadU8 {   // [B][src_h][src_w][3] uint8 BGR placed at (pad_top, pad_left) of the canvas, border 114, outside canvas 0
    static constexpr bool kStaged = true, kMagic = true;
    const uint8_t* p; int sh, sw, pt, pl;
    long long total_bytes;      // B * sh * sw * 3 (vector loads must stay inside the buffer)
    // Copy canvas rows y0 .. y0+16, columns x0 .. x0+32 into s_in (row r at r * kStemPitch + off[r], off[r] = s_in[17 * kStemPitch + r]).
    // Returns false (nothing written) unless the whole patch lies inside the frame: border tiles take the per-byte path.
    // fetch(): the loads of one patch into registers (chunk tid, and chunk 128 + tid for tid < 8); commit(): registers -> s_in.
    // The kernel fetches the patch of its NEXT tile before it works on the current one, so the global-memory latency of the
    // patch is hidden behind a whole tile of build / MMA / epilogue instead of being paid at the top of every tile.
    // Per-thread state of one patch between fetch and commit: the two vectors, the low address bits of the thread's rows (row r
    // starts lo bytes into its first 16-byte vector) and whether the thread's vectors belong to the patch at all.
    struct Patch { uint4 v0, v1; int lo0, lo1; bool p0, p1; };
    __device__ __forceinline__ int row_offset(int tid) const { return (tid >> 3) * sw * 3; }       // byte offset of the thread's patch row
    __device__ __forceinline__ bool fetch(int b, int y0, int x0, int tid, int roff, Patch& P) const {
        const int fy0 = y0 - pt, fx0 = x0 - pl;
        if (fy0 < 0 || fx0 < 0 || fy0 + 16 >= sh || fx0 + 32 >= sw) return false;
        const long long g_first = (((long long)b * sh + fy0) * sw + fx0) * 3;                       // block-uniform
        if (g_first + 16ll * sw * 3 + 99 + 16 > total_bytes) return false;
        const int c16 = (tid & 7) * 16;
        {
            const long long g0 = g_first + roff;
            P.lo0 = (int)(g0 & 15);
            P.p0 = c16 < P.lo0 + 99;
            if (P.p0) P.v0 = __ldg(reinterpret_cast<const uint4*>(p + (g0 - P.lo0) + c16));
        }
        P.p1 = false;
        if (tid < 8) {
            const long long g0 = g_first + 16ll * sw * 3;
            P.lo1 = (int)(g0 & 15);
            P.p1 = c16 < P.lo1 + 99;
            if (P.p1) P.v1 = __ldg(reinterpret_cast<const uint4*>(p + (g0 - P.lo1) + c16));
        }
        return true;
    }
    __device__ __forceinline__ void commit(uint8_t* s_in, int tid, const Patch& P) const {
        const int r = tid >> 3, c16 = (tid & 7) * 16;
        if (P.p0) *reinterpret_cast<uint4*>(s_in + r * kStemPitch + c16) = P.v0;
        if (c16 == 0) s_in[17 * kStemPitch + r] = (uint8_t)P.lo0;
        if (tid < 8) {
            if (P.p1) *reinterpret_cast<uint4*>(s_in + 16 * kStemPitch + c16) = P.v1;
            if (tid == 0) s_in[17 * kStemPitch + 16] = (uint8_t)P.lo1;
        }
    }
    __device__ __forceinline__ void load(int b, int y, int x, int H, int W, float (&rgb)[3]) const {
        if (y < 0 || x < 0 || y >= H || x >= W) { rgb[0] = rgb[1] = rgb[2] = 0.f; return; }
        const int fy = y - pt, fx = x - pl;
        if (fy < 0 || fx < 0 || fy >= sh || fx >= sw) { rgb[0] = rgb[1] = rgb[2] = 114.f; return; }
        const uint8_t* q = p + (((size_t)b * sh + fy) * sw + fx) * 3;
        rgb[2] = (float)__ldg(q); rgb[1] = (float)__ldg(q + 1); rgb[0] = (float)__ldg(q + 2);
    }
};
template <typename T>
struct LoadPlanar {   // [B][3][H][W] RGB in [0,1]; the tensor core consumes bf16(255 x) (exact for uint8-derived inputs)
    static constexpr bool kStaged = false, kMagic = false;
    const T* p;
    struct Patch {};
    __device__ __forceinline__ int row_offset(int) const { return 0; }
    __device__ __forceinline__ bool fetch(int, int, int, int, int, Patch&) const { return false; }
    __device__ __forceinline__ void commit(uint8_t*, int, const Patch&) const {}
    __device__ __forceinline__ void load(int b, int y, int x, int H, int W, float (&rgb)[3]) const {
        if (y < 0 || x < 0 || y >= H || x >= W) { rgb[0] = rgb[1] = rgb[2] = 0.f; return; }
        const size_t plane = (size_t)H * W;
        const T* q = p + (size_t)b * 3 * plane + (size_t)y * W + x;
        rgb[0] = 255.f * (float)q[0]; rgb[1] = 255.f * (float)q[plane]; rgb[2] = 255.f * (float)q[2 * plane];
    }
};

template <typename Loader>
int launch_stem(Loader ld, int B, int H, int W, const void* w, const float* bias, int C0,
                void* out, int out_cstride, int out_coff, cudaStream_t st) {
    const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
    const int n_tile = b2_ceil_div(C0, 16) * 16;
    if (n_tile > kStemMaxC0) { b2_set_error("stem: C0=%d exceeds %d", C0, kStemMaxC0); return B2_ERR_UNSUPPORTED; }
    uint32_t cols = 32;
    while (cols < (uint32_t)n_tile) cols <<= 1;
    const int tiles_w = b2_ceil_div(Wo, 16), tiles_h = b2_ceil_div(Ho, 8);
    const long long total = (long long)tiles_w * tiles_h * B;
    // (a two-role variant -- 128 builder + 128 drainer threads, two tiles in flight per CTA, four CTAs per SM -- was slower: 0.71 vs
    //  0.58 ms; the kernel is bound by instruction issue and the shared-memory pipe, not by the serial phases of a tile)
    if ((long long)B * Ho * Wo >= (1ll << 31)) { b2_set_error("stem: B * Ho * Wo exceeds 2^31"); return B2_ERR_UNSUPPORTED; }
    const int per_sm = (int)(512 / cols) < B2_STEM_CTAS ? (int)(512 / cols) : B2_STEM_CTAS;       // TMEM columns bound the co-resident CTAs
    const long long slots = (long long)b2_num_sms() * per_sm;
    const int grid = (int)(total < slots ? total : slots);
    stem_tc_kernel<Loader><<<grid, kStemThreads, 0, st>>>(ld, B, H, W, Ho, Wo, (const __nv_bfloat16*)w, bias, 1.f / 255.f, C0, n_tile, cols,
                                                          (__nv_bfloat16*)out, out_cstride, out_coff, tiles_w, tiles_h, (int)total);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

// ------------------------------------------------------------------------------------------------
// SPPF pooling: three chained MaxPool2d(5,1,2) == windows of 5, 9, 13 with -inf padding (block.py:237-241)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 max_bf16x8(uint4 a, uint4 b) {
    uint4 r;
    const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
    __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) pr[i] = __hmax2(pa[i], pb[i]);
    return r;
}

// One CTA per (image, group of CK 8-channel chunks): the whole H x W map of the group sits in shared memory, pixel-major with
// the CK chunks of a pixel adjacent (global accesses are CK * 16 contiguous bytes per pixel instead of one 16-byte piece per
// 2 KB); each MaxPool2d(5,1,2) is a row pass then a column pass (2 x 4 comparisons per pixel instead of 24), chained three times.
__global__ void __launch_bounds__(256) sppf_pool_kernel(__nv_bfloat16* __restrict__ buf, int B, int H, int W, int cstride, int coff, int C, int CK) {
    extern __shared__ uint4 s_pool[];              // [2][H*W*CK]
    const int b = blockIdx.y, HW = H * W, n = HW * CK;
    uint4* cur = s_pool;
    uint4* tmp = s_pool + n;
    __nv_bfloat16* base = buf + (size_t)b * HW * cstride + coff + blockIdx.x * CK * 8;
    for (int q = threadIdx.x; q < n; q += blockDim.x) {
        const int p = q / CK, c = q - p * CK;
        cur[q] = *reinterpret_cast<const uint4*>(base + (size_t)p * cstride + c * 8);
    }
    __syncthreads();
    const int rw = W * CK;                         // one image row in staged elements
    for (int level = 1; level <= 3; ++level) {
        for (int q = threadIdx.x; q < n; q += blockDim.x) {      // row pass: max over x-2..x+2
            const int x = (q / CK) % W;
            uint4 m = cur[q];
            if (x >= 1) m = max_bf16x8(m, cur[q - CK]);
            if (x >= 2) m = max_bf16x8(m, cur[q - 2 * CK]);
            if (x + 1 < W) m = max_bf16x8(m, cur[q + CK]);
            if (x + 2 < W) m = max_bf16x8(m, cur[q + 2 * CK]);
            tmp[q] = m;
        }
        __syncthreads();
        for (int q = threadIdx.x; q < n; q += blockDim.x) {      // column pass: max over y-2..y+2
            const int p = q / CK, c = q - p * CK, y = p / W;
            uint4 m = tmp[q];
            if (y >= 1) m = max_bf16x8(m, tmp[q - rw]);
            if (y >= 2) m = max_bf16x8(m, tmp[q - 2 * rw]);
            if (y + 1 < H) m = max_bf16x8(m, tmp[q + rw]);
            if (y + 2 < H) m = max_bf16x8(m, tmp[q + 2 * rw]);
            cur[q] = m;
            *reinterpret_cast<uint4*>(base + (size_t)p * cstride + (size_t)level * C + c * 8) = m;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// nearest upsample (x1 / x2) of a channel slice into a channel slice (Upsample + Concat)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upsample_slice_kernel(const __nv_bfloat16* __restrict__ in, int B, int H, int W, int ics, int ico,
                                                             int C, int scale, __nv_bfloat16* __restrict__ out, int ocs, int oco) {
    const int chunks = C / 8;
    const int Ho = H * scale, Wo = W * scale;
    const size_t total = (size_t)B * Ho * Wo * chunks;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int ck = (int)(idx % chunks);
    size_t pix = idx / chunks;
    const int x = (int)(pix % Wo), y = (int)((pix / Wo) % Ho), b = (int)(pix / ((size_t)Wo * Ho));
    const uint4 v = *reinterpret_cast<const uint4*>(in + (((size_t)b * H + y / scale) * W + x / scale) * ics + ico + ck * 8);
    *reinterpret_cast<uint4*>(out + (((size_t)b * Ho + y) * Wo + x) * ocs + oco + ck * 8) = v;
}

__global__ void __launch_bounds__(256) preprocess_u8_kernel(const uint8_t* __restrict__ f, int B, int sh, int sw, int H, int W, int pt, int pl,
                                                            float* __restrict__ out) {
    const size_t total = (size_t)B * H * W;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % W), y = (int)((idx / W) % H), b = (int)(idx / ((size_t)W * H));
    const int fy = y - pt, fx = x - pl;
    float r = 114.f, g = 114.f, bl = 114.f;
    if (fy >= 0 && fx >= 0 && fy < sh && fx < sw) {
        const uint8_t* q = f + (((size_t)b * sh + fy) * sw + fx) * 3;
        bl = (float)q[0]; g = (float)q[1]; r = (float)q[2];
    }
    const size_t plane = (size_t)H * W;
    float* o = out + (size_t)b * 3 * plane + (size_t)y * W + x;
    o[0] = r / 255.f; o[plane] = g / 255.f; o[2 * plane] = bl / 255.f;
}

// cv2.resize(INTER_LINEAR) for uint8, bit-exact: 11-bit fixed-point coefficients (INTER_RESIZE_COEF_BITS = 11),
// coefficients rounded with saturate_cast<short>(rint(f * 2048)), vertical pass result
// (x >> 4 * beta >> 16 ...) reproduced with the 8u formula  ((b0*(S0>>4))>>16 + (b1*(S1>>4))>>16 + 2) >> 2.
// The three functions below are the only copy of that arithmetic; every resize kernel samples through them.
struct CvTap { int i0, i1, w0, w1; };      // source indices and their 11-bit weights for one destination index

// cv::resize: f = (float)((d + 0.5) * scale - 0.5) in double, rounded once -- no fused multiply-add.  scale = 1 / (dst / src).
// Horizontal taps: an index outside [0, n-1) is clamped AND its fraction zeroed (the xofs / alpha tables of cv::resize).
__device__ __forceinline__ CvTap cv_tap_x(int d, double scale, int n) {
    float f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    int s = (int)floorf(f); f -= s;
    if (s < 0) { f = 0; s = 0; }
    if (s >= n - 1) { f = 0; s = n - 1; }
    return {s, min(s + 1, n - 1), __float2int_rn((1.f - f) * 2048.f), __float2int_rn(f * 2048.f)};
}

// Vertical taps: the two row indices are clamped, the fraction is kept (yofs / beta).
__device__ __forceinline__ CvTap cv_tap_y(int d, double scale, int n) {
    float f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    const int s = (int)floorf(f); f -= s;
    return {min(max(s, 0), n - 1), min(max(s + 1, 0), n - 1), __float2int_rn((1.f - f) * 2048.f), __float2int_rn(f * 2048.f)};
}

// One output byte from the 2 x 2 neighbourhood (p_row_col) of one channel.
__device__ __forceinline__ int cv_sample_u8(int p00, int p01, int p10, int p11, int a0, int a1, int b0, int b1) {
    const int S0 = p00 * a0 + p01 * a1;
    const int S1 = p10 * a0 + p11 * a1;
    const int v = (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2;
    return min(max(v, 0), 255);
}

__global__ void __launch_bounds__(256) resize_bilinear_u8_kernel(const uint8_t* __restrict__ src, int B, int sh, int sw,
                                                                 uint8_t* __restrict__ dst, int dh, int dw, double fy, double fx) {
    const size_t total = (size_t)B * dh * dw;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % dw), y = (int)((idx / dw) % dh), b = (int)(idx / ((size_t)dw * dh));
    const CvTap tx = cv_tap_x(x, fx, sw), ty = cv_tap_y(y, fy, sh);
    const uint8_t* r0 = src + ((size_t)b * sh + ty.i0) * sw * 3;
    const uint8_t* r1 = src + ((size_t)b * sh + ty.i1) * sw * 3;
    uint8_t* o = dst + idx * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        o[c] = (uint8_t)cv_sample_u8(r0[tx.i0 * 3 + c], r0[tx.i1 * 3 + c], r1[tx.i0 * 3 + c], r1[tx.i1 * 3 + c], tx.w0, tx.w1, ty.w0, ty.w1);
}

// LetterBox (data/augment.py:1692-1733) for a ragged batch.  Grid (bands of canvas rows, image); a thread writes 16 canvas pixels
// (48 bytes, three 16-byte stores: canvas rows are W*3 bytes with W % 16 == 0, so every group is 16-byte aligned).  Rows and
// columns outside the placed image are 114 without a read.  A resized image shares its column taps across all its rows: the CTA
// puts them in shared memory once, and the row taps of its band too.  An unresized image is copied (16-byte loads when aligned).
constexpr int kLbThreads = 256;
constexpr int kLbMaxW = 4096;        // column-tap table: 8 bytes per canvas column in static shared memory
constexpr int kLbMaxBand = 64;

__global__ void __launch_bounds__(kLbThreads) letterbox_u8_kernel(const uint8_t* __restrict__ src, const int64_t* __restrict__ src_off,
                                                                  const int32_t* __restrict__ geom, int H, int W, int band,
                                                                  uint8_t* __restrict__ canvas) {
    __shared__ int2 s_col[kLbMaxW];            // {byte offset of tap 0, (tap 1 - tap 0 in bytes: 0 or 3) << 28 | w0 << 16 | w1}
    __shared__ int4 s_row[kLbMaxBand];         // {row 0 byte offset, row 1 byte offset, b0, b1}
    const int b = blockIdx.y, y0 = blockIdx.x * band, y1 = min(H, y0 + band);
    const int* g = geom + (size_t)b * 6;
    const int sh = g[0], sw = g[1], top = g[4], left = g[5];
    int rh = g[2], rw = g[3];
    // a placement that does not fit the canvas (or an empty source) leaves the whole canvas at 114 instead of writing out of bounds
    if (sh <= 0 || sw <= 0 || top < 0 || left < 0 || rh < 0 || rw < 0 || top + rh > H || left + rw > W) rh = rw = 0;
    const uint8_t* img = src + src_off[b];
    const bool copy = rh == sh && rw == sw;
    // 16-pixel groups all inside or all outside the image, on 16-byte source addresses
    const bool copy16 = copy && left % 16 == 0 && sw % 16 == 0 && src_off[b] % 16 == 0;
    if (!copy) {
        const double fx = 1.0 / ((double)rw / sw), fy = 1.0 / ((double)rh / sh);     // scale = 1 / inv_scale as cv::resize forms it
        for (int x = threadIdx.x; x < rw; x += kLbThreads) {
            const CvTap t = cv_tap_x(x, fx, sw);
            s_col[x] = make_int2(t.i0 * 3, ((t.i1 - t.i0) * 3) << 28 | t.w0 << 16 | t.w1);
        }
        for (int r = threadIdx.x; r < y1 - y0; r += kLbThreads) {
            const int y = y0 + r - top;
            if (y >= 0 && y < rh) {
                const CvTap t = cv_tap_y(y, fy, sh);
                s_row[r] = make_int4(t.i0 * sw * 3, t.i1 * sw * 3, t.w0, t.w1);
            }
        }
        __syncthreads();
    }
    const int groups = W / 16;
    uint8_t* out = canvas + (size_t)b * H * W * 3;
    for (int it = threadIdx.x; it < (y1 - y0) * groups; it += kLbThreads) {
        const int r = it / groups, gx = (it - r * groups) * 16, y = y0 + r, sy = y - top;
        uint4* o = reinterpret_cast<uint4*>(out + ((size_t)y * W + gx) * 3);
        const bool row_in = sy >= 0 && sy < rh;
        if (!row_in || gx + 16 <= left || gx >= left + rw) {
            const uint4 fill = make_uint4(0x72727272u, 0x72727272u, 0x72727272u, 0x72727272u);
            o[0] = fill; o[1] = fill; o[2] = fill;
            continue;
        }
        if (copy16) {
            const uint4* s = reinterpret_cast<const uint4*>(img + ((size_t)sy * sw + (gx - left)) * 3);
            o[0] = s[0]; o[1] = s[1]; o[2] = s[2];
            continue;
        }
        uint32_t w[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) w[k] = 0;
        int4 rt = make_int4(sy * sw * 3, 0, 0, 0);
        if (!copy) rt = s_row[r];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int x = gx + i - left;
            int v0 = 114, v1 = 114, v2 = 114;
            if (x >= 0 && x < rw) {
                if (copy) {
                    const uint8_t* p = img + rt.x + x * 3;
                    v0 = p[0]; v1 = p[1]; v2 = p[2];
                } else {
                    const int2 c = s_col[x];
                    const int a0 = (c.y >> 16) & 0xfff, a1 = c.y & 0xffff, d = c.y >> 28;
                    const uint8_t* p0 = img + rt.x + c.x;
                    const uint8_t* p1 = img + rt.y + c.x;
                    v0 = cv_sample_u8(p0[0], p0[d], p1[0], p1[d], a0, a1, rt.z, rt.w);
                    v1 = cv_sample_u8(p0[1], p0[d + 1], p1[1], p1[d + 1], a0, a1, rt.z, rt.w);
                    v2 = cv_sample_u8(p0[2], p0[d + 2], p1[2], p1[d + 2], a0, a1, rt.z, rt.w);
                }
            }
            w[(3 * i) / 4] |= (uint32_t)v0 << (8 * ((3 * i) % 4));
            w[(3 * i + 1) / 4] |= (uint32_t)v1 << (8 * ((3 * i + 1) % 4));
            w[(3 * i + 2) / 4] |= (uint32_t)v2 << (8 * ((3 * i + 2) % 4));
        }
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
        o[2] = make_uint4(w[8], w[9], w[10], w[11]);
    }
}

}  // namespace

extern "C" int b2_stem_u8(const uint8_t* frames, int B, int src_h, int src_w, int H, int W, int pad_top, int pad_left,
                          const void* w, const float* bias, int C0, void* out, int out_cstride, int out_coff, void* stream) {
    B2_REQUIRE(frames && w && bias && out, "stem: null pointer");
    B2_REQUIRE(C0 % 8 == 0 && out_cstride % 8 == 0 && out_coff % 8 == 0, "stem: channel counts must be multiples of 8");
    B2_REQUIRE(pad_top >= 0 && pad_left >= 0 && pad_top + src_h <= H && pad_left + src_w <= W, "stem: frame does not fit the canvas");
    B2_REQUIRE((uintptr_t)w % 16 == 0 && (uintptr_t)out % 16 == 0, "stem: pointers must be 16-byte aligned");
    B2_REQUIRE((uintptr_t)frames % 16 == 0, "stem: the frame buffer must be 16-byte aligned");
    LoadU8 ld{frames, src_h, src_w, pad_top, pad_left, (long long)B * src_h * src_w * 3};
    return launch_stem(ld, B, H, W, w, bias, C0, out, out_cstride, out_coff, (cudaStream_t)stream);
}

extern "C" int b2_stem_f32(const void* bchw, int dtype, int B, int H, int W, const void* w, const float* bias, int C0,
                           void* out, int out_cstride, int out_coff, void* stream) {
    B2_REQUIRE(bchw && w && bias && out, "stem: null pointer");
    B2_REQUIRE(C0 % 8 == 0 && out_cstride % 8 == 0 && out_coff % 8 == 0, "stem: channel counts must be multiples of 8");
    if (dtype == 0) return launch_stem(LoadPlanar<float>{(const float*)bchw}, B, H, W, w, bias, C0, out, out_cstride, out_coff, (cudaStream_t)stream);
    if (dtype == 1) return launch_stem(LoadPlanar<__nv_bfloat16>{(const __nv_bfloat16*)bchw}, B, H, W, w, bias, C0, out, out_cstride, out_coff, (cudaStream_t)stream);
    b2_set_error("stem: dtype %d unsupported", dtype);
    return B2_ERR_UNSUPPORTED;
}

extern "C" int b2_sppf_pool(void* buf, int B, int H, int W, int cstride, int coff, int C, void* stream) {
    B2_REQUIRE(C % 8 == 0 && cstride % 8 == 0 && coff % 8 == 0 && coff + 4 * C <= cstride, "sppf_pool: bad channel layout");
    // chunks per CTA: 64 contiguous bytes per pixel when the map and the chunk count allow it
    int CK = 4;
    while (CK > 1 && ((C / 8) % CK != 0 || (size_t)2 * H * W * CK * sizeof(uint4) > 96 * 1024)) CK >>= 1;
    const size_t smem = (size_t)2 * H * W * CK * sizeof(uint4);
    B2_REQUIRE(smem <= 200 * 1024, "sppf_pool: %dx%d map does not fit in shared memory", H, W);
    if (smem > 48 * 1024) B2_CUDA(cudaFuncSetAttribute(sppf_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    sppf_pool_kernel<<<dim3(C / 8 / CK, B), 256, smem, (cudaStream_t)stream>>>((__nv_bfloat16*)buf, B, H, W, cstride, coff, C, CK);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_upsample_slice(const void* in, int B, int H, int W, int in_cstride, int in_coff, int C, int scale,
                                 void* out, int out_cstride, int out_coff, void* stream) {
    B2_REQUIRE(scale == 1 || scale == 2, "upsample: scale must be 1 or 2");
    B2_REQUIRE(C % 8 == 0 && in_cstride % 8 == 0 && in_coff % 8 == 0 && out_cstride % 8 == 0 && out_coff % 8 == 0, "upsample: channels must be multiples of 8");
    const size_t total = (size_t)B * H * scale * W * scale * (C / 8);
    upsample_slice_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)in, B, H, W, in_cstride, in_coff, C, scale, (__nv_bfloat16*)out, out_cstride, out_coff);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_preprocess_u8(const uint8_t* frames, int B, int src_h, int src_w, int H, int W, int pad_top, int pad_left,
                                float* out_bchw, void* stream) {
    B2_REQUIRE(pad_top >= 0 && pad_left >= 0 && pad_top + src_h <= H && pad_left + src_w <= W, "preprocess: frame does not fit the canvas");
    const size_t total = (size_t)B * H * W;
    preprocess_u8_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(frames, B, src_h, src_w, H, W, pad_top, pad_left, out_bchw);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_resize_bilinear_u8(const uint8_t* src, int B, int sh, int sw, uint8_t* dst, int dh, int dw, void* stream) {
    B2_REQUIRE(sh > 0 && sw > 0 && dh > 0 && dw > 0, "resize: bad shape");
    const size_t total = (size_t)B * dh * dw;
    resize_bilinear_u8_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        src, B, sh, sw, dst, dh, dw, 1.0 / ((double)dh / sh), 1.0 / ((double)dw / sw));   // scale = 1 / inv_scale as cv::resize forms it
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_letterbox_u8(const uint8_t* src, const int64_t* src_off, const int32_t* geom, int B, int H, int W, uint8_t* canvas,
                               void* stream) {
    B2_REQUIRE(src && src_off && geom && canvas, "letterbox: null pointer");
    B2_REQUIRE(B >= 1 && B <= 65535 && H >= 1, "letterbox: bad batch %d / height %d", B, H);
    B2_REQUIRE(W >= 16 && W <= kLbMaxW && W % 16 == 0, "letterbox: canvas width %d must be a multiple of 16 in [16, %d]", W, kLbMaxW);
    B2_REQUIRE((uintptr_t)src % 16 == 0 && (uintptr_t)canvas % 16 == 0, "letterbox: source and canvas must be 16-byte aligned");
    // a band of rows per CTA: about four 16-pixel groups per thread, so the tap tables are amortised over enough work
    const int band = min(kLbMaxBand, max(1, 4 * kLbThreads / (W / 16)));
    letterbox_u8_kernel<<<dim3((unsigned)b2_ceil_div(H, band), (unsigned)B), kLbThreads, 0, (cudaStream_t)stream>>>(
        src, src_off, geom, H, W, band, canvas);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}
