// Detect post-processing for sm_100a: DFL decode + confidence filter + compaction, and per-image NMS
// (sort, greedy suppression, scale_boxes/clip) -- HBM-bandwidth kernels with coalesced 16-byte accesses.
//
//   decode_kernel  Detect._inference (ultralytics/nn/modules/head.py:152-187), DFL (block.py:78-81),
//                  make_anchors / dist2bbox (utils/tal.py:367-391), then the candidate test of
//                  non_max_suppression (utils/nms.py:74 amax > conf, :111 best class, :120-124 classes).
//   nms_kernel     utils/nms.py:129-160 (+ torchvision.ops.nms / TorchNMS.nms :237-304) and
//                  scale_boxes / clip_boxes (utils/ops.py:105-138, :157-183).
#include "common.cuh"

#include <algorithm>

void b2_count_launch(int n);

namespace {

constexpr int kMaxLevels = 8;

struct DecodeParams {
    const __nv_bfloat16* lv[kMaxLevels];
    int h[kMaxLevels], w[kMaxLevels], stride[kMaxLevels], a_off[kMaxLevels + 1];
    int blk_off[kMaxLevels + 1];       // first block of each level: the level is block-uniform
    int n_levels, B, nc, lstride, A;
    float conf, logit_lo;              // logit_lo = logit(conf) - 0.05: below it the exact test `score > conf` cannot pass
    const uint8_t* cmask;
    float* cand; int32_t* cand_idx; int32_t* cand_count; int cand_cap;
    float* dense;
};

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
    f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}

// 8 lanes cooperate on one anchor: lane s loads 16-byte chunk s of the 64 DFL logits (side = s/2,
// bins (s&1)*8..+7), then chunks s, s+8, ... of the class logits.  A warp covers 4 consecutive anchors
// = 4 x (64+nc) x 2 contiguous bytes of the NHWC logits.
// DENSE: also write the reference-shaped (B, 4 + nc, A) tensor (every anchor decoded); the candidate-only instance keeps fewer
// registers live (6 blocks of 256 threads per SM instead of 4: the kernel is bound by bytes in flight, 32 per thread)
template <bool DENSE>
__global__ void __launch_bounds__(256, DENSE ? 4 : 6) decode_kernel(const DecodeParams p) {
    const int lane = threadIdx.x & 31, sub = lane & 7;
    const int b = blockIdx.y;
    int lvl = 0;
#pragma unroll
    for (int l = 1; l < kMaxLevels; ++l) if (l < p.n_levels && (int)blockIdx.x >= p.blk_off[l]) lvl = l;
    const int W = p.w[lvl], H = p.h[lvl];
    const int la_raw = (((int)blockIdx.x - p.blk_off[lvl]) * (int)blockDim.x + (int)threadIdx.x) >> 3;
    const bool active = la_raw < H * W;
    const int la = active ? la_raw : 0;
    const int a = p.a_off[lvl] + la;
    const __nv_bfloat16* row = p.lv[lvl] + ((size_t)b * H * W + la) * p.lstride;

    // ---- class loads first (memory-level parallelism): up to two class chunks per lane; the DFL chunk only when needed ----
    const int nchunks = (p.nc + 7) >> 3;
    const uint4 ninf4 = make_uint4(0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u);   // bf16 -inf pairs
    uint4 q0 = make_uint4(0, 0, 0, 0), q1 = ninf4, q2 = ninf4;
    if (active) {
        if (DENSE) q0 = ldg_nc_v4(row + sub * 8);
        if (sub < nchunks) q1 = ldg_nc_v4(row + 64 + sub * 8);
        if (sub + 8 < nchunks) q2 = ldg_nc_v4(row + 64 + (sub + 8) * 8);
    }

    // ---- classes: max logit / argmax over nc ----
    float best = -INFINITY; int bidx = 0x7fffffff;
    const size_t dense_base = (size_t)b * (4 + p.nc) * p.A + a;
    if (!DENSE) {
        // Pass 1: only the MAX logit of the anchor, with packed bf16x2 max instructions (exact: max of bf16 values).  The class
        // index is looked up afterwards, and only in warps that hold a candidate.
        __nv_bfloat162 m2 = __floats2bfloat162_rn(-INFINITY, -INFINITY);
        for (int ck = sub; ck < nchunks; ck += 8) {
            uint4 q = ck == sub ? q1 : ck == sub + 8 ? q2 : (active ? ldg_nc_v4(row + 64 + ck * 8) : ninf4);
            const int nvalid = p.nc - ck * 8;                       // < 8 only in the last chunk: padding channels are not classes
            if (nvalid < 8) {
                uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (2 * i >= nvalid) w[i] = 0xFF80FF80u;
                    else if (2 * i + 1 >= nvalid) w[i] = (w[i] & 0x0000FFFFu) | 0xFF800000u;
                }
                q = make_uint4(w[0], w[1], w[2], w[3]);
            }
            m2 = __hmax2(m2, *reinterpret_cast<const __nv_bfloat162*>(&q.x)); m2 = __hmax2(m2, *reinterpret_cast<const __nv_bfloat162*>(&q.y));
            m2 = __hmax2(m2, *reinterpret_cast<const __nv_bfloat162*>(&q.z)); m2 = __hmax2(m2, *reinterpret_cast<const __nv_bfloat162*>(&q.w));
        }
        best = fmaxf(__low2float(m2), __high2float(m2));
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
        const bool maybe = active && best > p.logit_lo;
        if (!__any_sync(0xffffffffu, maybe)) return;
    }
    best = -INFINITY;
    for (int ck = sub; ck < nchunks; ck += 8) {
        float c[8];
        if (ck == sub) unpack8(q1, c);
        else if (ck == sub + 8) unpack8(q2, c);
        else if (active) unpack8(ldg_nc_v4(row + 64 + ck * 8), c);
        else {
#pragma unroll
            for (int i = 0; i < 8; ++i) c[i] = -INFINITY;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int ci = ck * 8 + i;
            if (ci < p.nc) {
                if (DENSE && active) p.dense[dense_base + (size_t)(4 + ci) * p.A] = 1.f / (1.f + __expf(-c[i]));
                if (c[i] > best) { best = c[i]; bidx = ci; }
            }
        }
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
    }
    const float score = 1.f / (1.f + __expf(-best));
    // best class over ALL classes first, then the `classes=` filter drops the anchor (nms.py:111-124)
    const bool anchor_cand = active && bidx != 0x7fffffff && score > p.conf && (!p.cmask || p.cmask[bidx]);
    // Boxes are only needed for candidates (a per cent of the anchors at conf 0.15) unless the dense tensor is asked for:
    // warps without a candidate stop here -- 128 of the 288 bytes per anchor are never read, 64 exponentials never taken.
    if (!DENSE) {
        if (!__any_sync(0xffffffffu, anchor_cand)) return;
        if (active) q0 = ldg_nc_v4(row + sub * 8);
    }

    // ---- DFL: softmax expectation over 16 bins per side ----
    float f[8];
    unpack8(q0, f);
    float m = f[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) m = fmaxf(m, f[i]);
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
    float se = 0.f, sw = 0.f;
    const float bin0 = (float)((sub & 1) * 8), ml = m * kLog2e;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float e = dfl_exp(f[i], ml);
        se += e; sw = fmaf(e, bin0 + (float)i, sw);
    }
    se += __shfl_xor_sync(0xffffffffu, se, 1);
    sw += __shfl_xor_sync(0xffffffffu, sw, 1);
    const float dist = sw / se;
    const int gbase = lane & ~7;
    const float dl = __shfl_sync(0xffffffffu, dist, gbase + 0), dt = __shfl_sync(0xffffffffu, dist, gbase + 2);
    const float dr = __shfl_sync(0xffffffffu, dist, gbase + 4), db = __shfl_sync(0xffffffffu, dist, gbase + 6);

    // ---- box (tal.py:382-391 then * stride; xywh2xyxy ops.py:277-294), same fp32 operation order ----
    const float ax = (float)(la % W) + 0.5f, ay = (float)(la / W) + 0.5f, st = (float)p.stride[lvl];
    const float x1 = ax - dl, y1 = ay - dt, x2 = ax + dr, y2 = ay + db;
    const float cx = (x1 + x2) / 2.f * st, cy = (y1 + y2) / 2.f * st, bw = (x2 - x1) * st, bh = (y2 - y1) * st;
    if (DENSE && active && sub < 4) p.dense[dense_base + (size_t)sub * p.A] = sub == 0 ? cx : sub == 1 ? cy : sub == 2 ? bw : bh;

    const bool is_cand = anchor_cand && sub == 0;
    const unsigned ball = __ballot_sync(0xffffffffu, is_cand);
    if (ball) {
        int base = 0;
        const int leader = __ffs(ball) - 1;
        if (lane == leader) base = atomicAdd(p.cand_count + b, __popc(ball));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (is_cand) {
            const int pos = base + __popc(ball & ((1u << lane) - 1));
            if (pos < p.cand_cap) {
                float* o = p.cand + ((size_t)b * p.cand_cap + pos) * 6;
                const float hw = bw / 2.f, hh = bh / 2.f;
                o[0] = cx - hw; o[1] = cy - hh; o[2] = cx + hw; o[3] = cy + hh; o[4] = score; o[5] = (float)bidx;
                p.cand_idx[(size_t)b * p.cand_cap + pos] = a;
            }
        }
    }
}

// Candidate extraction from the fused Detect-head outputs (conv epilogue modes 1 / 2): per anchor 4 fp32 DFL distances
// and {best class logit, class}.  Same box arithmetic, threshold test and candidate layout as decode_kernel.
struct HeadParams {
    const float* dist[kMaxLevels]; const float* cls[kMaxLevels];
    int h[kMaxLevels], w[kMaxLevels], stride[kMaxLevels], a_off[kMaxLevels + 1];
    int blk_off[kMaxLevels + 1];       // first block of each level (blocks never straddle a level: the level is block-uniform)
    int n_levels, A, B;
    float conf, logit_lo;              // logit_lo: logit(conf) - 0.05; below it the exact score test cannot pass
    const uint8_t* cmask;
    float* cand; int32_t* cand_idx; int32_t* cand_count; int cand_cap;
};

// One thread tests kHcPer anchors of one (level, image), a block apart (coalesced 8-byte loads of {logit, class} records), all of
// them issued before any is used.  The kernel moves 8 bytes per anchor; the sigmoid, the box and the 16-byte distance record
// are touched only for the per-cent of anchors whose logit clears logit_lo (then the reference's exact test `score > conf`).
#ifndef B2_HC_PER
#define B2_HC_PER 4
#endif
#ifndef B2_HC_THREADS
#define B2_HC_THREADS 128
#endif
constexpr int kHcPer = B2_HC_PER, kHcThreads = B2_HC_THREADS;      // experiment builds: tools/build_variant.sh

__global__ void __launch_bounds__(kHcThreads) head_candidates_kernel(const HeadParams p) {
    const int lane = threadIdx.x & 31;
    int lvl = 0;
#pragma unroll
    for (int l = 1; l < kMaxLevels; ++l) if (l < p.n_levels && (int)blockIdx.x >= p.blk_off[l]) lvl = l;
    const int W = p.w[lvl], HW = p.h[lvl] * W, b = blockIdx.y;
    const float2* cp = reinterpret_cast<const float2*>(p.cls[lvl]) + (size_t)b * HW;
    const int la0 = ((int)blockIdx.x - p.blk_off[lvl]) * (kHcThreads * kHcPer) + threadIdx.x;
    float2 c[kHcPer];
#pragma unroll
    for (int k = 0; k < kHcPer; ++k) {
        const int la = la0 + k * kHcThreads;
        c[k] = la < HW ? __ldg(cp + la) : make_float2(-INFINITY, 0.f);
    }
    const float lo = p.logit_lo;
    bool any = false;
#pragma unroll
    for (int k = 0; k < kHcPer; ++k) any |= c[k].x > lo;
    if (!__any_sync(0xffffffffu, any)) return;
    const float st = (float)p.stride[lvl];
    const float4* dp = reinterpret_cast<const float4*>(p.dist[lvl]) + (size_t)b * HW;
#pragma unroll
    for (int k = 0; k < kHcPer; ++k) {
        const float logit = c[k].x;
        const int bidx = (int)c[k].y;
        const int la = la0 + k * kHcThreads;
        bool is_cand = false;
        float score = 0.f, x1 = 0.f, y1 = 0.f, x2 = 0.f, y2 = 0.f;
        if (logit > lo) {
            score = 1.f / (1.f + __expf(-logit));
            if (score > p.conf && (!p.cmask || p.cmask[bidx])) {
                const float4 d = __ldg(dp + la);
                const float ax = (float)(la % W) + 0.5f, ay = (float)(la / W) + 0.5f;
                const float u1 = ax - d.x, v1 = ay - d.y, u2 = ax + d.z, v2 = ay + d.w;
                const float cx = (u1 + u2) / 2.f * st, cy = (v1 + v2) / 2.f * st, bw = (u2 - u1) * st, bh = (v2 - v1) * st;
                const float hw = bw / 2.f, hh = bh / 2.f;
                x1 = cx - hw; y1 = cy - hh; x2 = cx + hw; y2 = cy + hh;
                is_cand = true;
            }
        }
        const unsigned ball = __ballot_sync(0xffffffffu, is_cand);
        if (!ball) continue;
        int base = 0;
        const int leader = __ffs(ball) - 1;
        if (lane == leader) base = atomicAdd(p.cand_count + b, __popc(ball));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (is_cand) {
            const int pos = base + __popc(ball & ((1u << lane) - 1));
            if (pos < p.cand_cap) {
                float* o = p.cand + ((size_t)b * p.cand_cap + pos) * 6;
                o[0] = x1; o[1] = y1; o[2] = x2; o[3] = y2; o[4] = score; o[5] = (float)bidx;
                p.cand_idx[(size_t)b * p.cand_cap + pos] = p.a_off[lvl] + la;
            }
        }
    }
}

__global__ void __launch_bounds__(256) dense_candidates_kernel(const float* __restrict__ pred, int nc, int no, int A, float conf,
                                                               const uint8_t* __restrict__ cmask, float* __restrict__ cand,
                                                               int32_t* __restrict__ cand_idx, int32_t* __restrict__ cand_count, int cand_cap) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y, lane = threadIdx.x & 31;
    const float* base = pred + (size_t)b * no * A;
    float best = -INFINITY; int bidx = -1;
    if (a < A) {
        for (int c = 0; c < nc; ++c) {
            const float v = __ldg(base + (size_t)(4 + c) * A + a);
            if (v > best) { best = v; bidx = c; }
        }
    }
    const bool is_cand = a < A && bidx >= 0 && best > conf && (!cmask || cmask[bidx]);
    const unsigned ball = __ballot_sync(0xffffffffu, is_cand);
    if (!ball) return;
    int pos0 = 0;
    const int leader = __ffs(ball) - 1;
    if (lane == leader) pos0 = atomicAdd(cand_count + b, __popc(ball));
    pos0 = __shfl_sync(0xffffffffu, pos0, leader);
    if (is_cand) {
        const int pos = pos0 + __popc(ball & ((1u << lane) - 1));
        if (pos < cand_cap) {
            const float cx = base[a], cy = base[(size_t)A + a], hw = base[(size_t)2 * A + a] / 2.f, hh = base[(size_t)3 * A + a] / 2.f;
            float* o = cand + ((size_t)b * cand_cap + pos) * 6;
            o[0] = cx - hw; o[1] = cy - hh; o[2] = cx + hw; o[3] = cy + hh; o[4] = best; o[5] = (float)bidx;
            cand_idx[(size_t)b * cand_cap + pos] = a;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// NMS: one CTA per image
// ------------------------------------------------------------------------------------------------
constexpr int kNmsThreads = 1024;
constexpr int kSmemSort = 4096;      // pairs sorted entirely in (dynamic) shared memory: one dense image among hundreds sets the kernel's time
constexpr int kMaxCand = 65536;      // alive bitmask (shared memory) covers this many sorted candidates (max_nms <= kMaxCand)
constexpr int kMaxKeep = 1024;
constexpr int kFastN = 704;          // bit-matrix path: 704 boxes (11 KB) + 704 x 22 words (62 KB) of dynamic shared memory

struct NmsParams {
    const float* cand; const int32_t* cand_idx; const int32_t* cand_count; int cand_cap, B;
    float iou_thres; int max_det, max_nms, agnostic; float max_wh; int mode;
    float gain, pad_x, pad_y, orig_w, orig_h; int do_scale;
    const float* scale;  // NULL, or [B][5] {gain, pad_x, pad_y, orig_w, orig_h} per image (b2_nms_scaled): replaces the scalars above
    float* out; int32_t* out_count; int32_t* out_idx;
    unsigned long long* ws_keys; int32_t* ws_pay; float4* ws_box; int P_max;
    int debug;          // B2_NMS_DEBUG=1: thread 0 of every CTA leaves clock64() stamps of its phases in its ws_box slice (exact mode only)
};

__device__ __forceinline__ void bitonic_exchange(unsigned long long* keys, int32_t* pay, int i, int j, bool desc_block) {
    const unsigned long long a = keys[i], b = keys[j];
    // descending overall: within a "descending" block the larger key goes first
    if ((a < b) == desc_block) {
        keys[i] = b; keys[j] = a;
        const int32_t t = pay[i]; pay[i] = pay[j]; pay[j] = t;
    }
}

// iou(bi, bj) > thr with the reference's fp32 operation order (torchvision nms / TorchNMS.nms), written so that the common case
// -- no overlap along x (always true for boxes of different classes: the class offset is 7680 px) -- costs three instructions.
// Exactly equivalent to the clamped form: iw <= 0 or ih <= 0 makes inter 0, and 0 / union is 0, -0 or NaN, never > thr >= 0.
__device__ __forceinline__ bool iou_exceeds(const float4 bi, const float area_i, const float4 bj, const float thr, bool* touches = nullptr) {
    const float iw = __fsub_rn(fminf(bi.z, bj.z), fmaxf(bi.x, bj.x));
    if (!(iw > 0.f)) return false;
    const float ih = __fsub_rn(fminf(bi.w, bj.w), fmaxf(bi.y, bj.y));
    if (!(ih > 0.f)) return false;
    const float inter = __fmul_rn(iw, ih);
    if (touches && inter != 0.f) *touches = true;
    const float area_j = __fmul_rn(__fsub_rn(bj.z, bj.x), __fsub_rn(bj.w, bj.y));
    return __fdiv_rn(inter, __fsub_rn(__fadd_rn(area_i, area_j), inter)) > thr;
}

// kScaled: the epilogue reads image b's row of p.scale (b2_nms_scaled); the scalar instance is b2_nms
template <bool kScaled>
__global__ void __launch_bounds__(kNmsThreads, 1) nms_kernel(const NmsParams p) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    unsigned long long* const s_keys = reinterpret_cast<unsigned long long*>(s_raw);          // [kSmemSort]
    int32_t* const s_pay = reinterpret_cast<int32_t*>(s_raw + (size_t)kSmemSort * 8);          // [kSmemSort]
    __shared__ int32_t s_keep[kMaxKeep];
    __shared__ uint32_t alive[kMaxCand / 32];
    __shared__ int s_cur, s_nkeep, s_any, s_done;

    // Heaviest images first: CTA r takes the image of rank r by candidate count (ties: lower index).  The kernel lasts as long
    // as its slowest image (one dense frame among hundreds has 10x the candidates), which must not start in the second wave.
    const int tid = threadIdx.x;
    int b = blockIdx.x;
    if (p.B <= kNmsThreads) {
        int* s_cnt = reinterpret_cast<int*>(alive);                       // alive[] is not in use yet
        if (tid < p.B) s_cnt[tid] = p.cand_count[tid];
        __syncthreads();
        if (tid < p.B) {
            const int mine = s_cnt[tid];
            int rank = 0;
            for (int j = 0; j < p.B; ++j) { const int c = s_cnt[j]; rank += (c > mine) || (c == mine && j < tid); }
            if (rank == (int)blockIdx.x) s_cur = tid;
        }
        __syncthreads();
        b = s_cur;
        __syncthreads();
    }
    int n = min(p.cand_count[b], p.cand_cap);
    const float* cand = p.cand + (size_t)b * p.cand_cap * 6;
    const int32_t* cidx = p.cand_idx + (size_t)b * p.cand_cap;
    float* out = p.out + (size_t)b * p.max_det * 6;
    if (n == 0) { if (tid == 0) p.out_count[b] = 0; return; }

    long long* const stamp = reinterpret_cast<long long*>(p.ws_box + (size_t)b * p.P_max);
    int n_stamp = 0;
#define NMS_STAMP() do { if (p.debug && tid == 0) stamp[n_stamp++] = clock64(); } while (0)
    NMS_STAMP();
    int P = 32;
    while (P < n) P <<= 1;
    const bool in_smem = P <= kSmemSort;
    unsigned long long* keys = in_smem ? s_keys : p.ws_keys + (size_t)b * p.P_max;
    int32_t* pay = in_smem ? s_pay : p.ws_pay + (size_t)b * p.P_max;
    for (int i = tid; i < P; i += kNmsThreads) {
        if (i < n) {
            // score > 0: its bit pattern orders like the float; ties -> lower anchor index first (stable sort of the reference)
            keys[i] = ((unsigned long long)__float_as_uint(cand[i * 6 + 4]) << 32) | (unsigned)(0x7fffffff - cidx[i]);
            pay[i] = i;
        } else { keys[i] = 0ull; pay[i] = -1; }
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (P >> 1); t += kNmsThreads) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                bitonic_exchange(keys, pay, i, i | j, (i & k) == 0);
            }
            __syncthreads();
        }
    }
    n = min(n, p.max_nms);
    NMS_STAMP();          // [1] sorted

    const int max_keep = min(p.max_det, kMaxKeep);
    if (p.mode == 0) {
        // ---- exact greedy NMS, blocked: candidates are taken in score order in blocks of kFastN.  Per block: (1) every
        //      member is tested against the boxes kept so far, (2) all pairwise tests inside the block go in parallel into
        //      an nb x nb bit matrix, (3) one warp walks the block in score order OR-ing the suppression rows of the boxes
        //      it keeps.  One block covers the usual case; dense scenes (thousands of candidates) take a few blocks instead
        //      of one block-wide pass per kept box. ----
        uint32_t* const s_dyn = reinterpret_cast<uint32_t*>(s_raw + (size_t)kSmemSort * 12);
        float4* fbox = reinterpret_cast<float4*>(s_dyn);                  // [kFastN] boxes of the block (class offset applied)
        uint32_t* mat = s_dyn + kFastN * 4;                                 // [nb][Wd]
        float4* kbox = reinterpret_cast<float4*>(mat + kFastN * ((kFastN + 31) / 32));   // [kMaxKeep] kept boxes
        uint32_t* dead = alive;                                            // [kFastN / 32] members suppressed by earlier blocks
        if (tid == 0) s_nkeep = 0;
        __syncthreads();
        for (int s0 = 0; s0 < n; s0 += kFastN) {
            const int nb = min(kFastN, n - s0), nk0 = s_nkeep;
            if (nk0 >= max_keep) break;
            const int Wd = (nb + 31) >> 5;
            for (int i = tid; i < nb; i += kNmsThreads) {
                const float* c = cand + (size_t)pay[s0 + i] * 6;
                const float off = p.agnostic ? 0.f : __fmul_rn(c[5], p.max_wh);
                fbox[i] = make_float4(__fadd_rn(c[0], off), __fadd_rn(c[1], off), __fadd_rn(c[2], off), __fadd_rn(c[3], off));
            }
            __syncthreads();
            NMS_STAMP();
            // (1) against the kept boxes of earlier blocks (warp-coalesced: lane <-> member, ballot -> one word per warp step)
            for (int i0 = (tid >> 5) * 32; i0 < Wd * 32; i0 += kNmsThreads) {
                const int i = i0 + (tid & 31);
                bool sup = false;
                if (i < nb && nk0 > 0) {
                    const float4 bi = fbox[i];
                    const float area_i = __fmul_rn(__fsub_rn(bi.z, bi.x), __fsub_rn(bi.w, bi.y));
                    for (int k = 0; k < nk0 && !sup; ++k) sup = iou_exceeds(bi, area_i, kbox[k], p.iou_thres);
                }
                const unsigned word = __ballot_sync(0xffffffffu, sup || i >= nb);
                if ((tid & 31) == 0) dead[i0 >> 5] = word;
            }
            // (2) pairwise tests inside the block, one warp per (row i, 32-column word wj >= i / 32): lane <-> column, so the
            //     box loads are consecutive (the per-thread form read fbox at a 512-byte stride: a 22-way bank conflict per
            //     load, 250 k cycles for a full block) and the word is one ballot
            {
                const int warp = tid >> 5, lane = tid & 31;
                for (int i = warp; i < nb; i += kNmsThreads / 32) {
                    const float4 bi = fbox[i];
                    const float area_i = __fmul_rn(__fsub_rn(bi.z, bi.x), __fsub_rn(bi.w, bi.y));
                    const int w0 = i >> 5;
                    if (lane < w0) mat[i * Wd + lane] = 0u;                       // below the diagonal: never set, but OR-ed by the walk
                    for (int wj = w0; wj < Wd; ++wj) {
                        const int j = wj * 32 + lane;
                        const bool sup = j > i && j < nb && iou_exceeds(bi, area_i, fbox[j], p.iou_thres);
                        const uint32_t word = __ballot_sync(0xffffffffu, sup);
                        if (lane == 0) mat[i * Wd + wj] = word;
                    }
                }
            }
            __syncthreads();
            NMS_STAMP();
            // (3) greedy walk of the block by one warp, 32 members at a time: the keep decisions inside a group need only the
            //     group's 32 x 32 diagonal block (32 broadcast loads up front: the sequential chain is register arithmetic); the rows of the kept members are then OR-ed into the other words with independent loads
            if (tid < 32) {
                uint32_t removed = tid < Wd ? dead[tid] : 0xffffffffu;        // lane l owns word l (Wd <= 32)
                int nk = nk0;
                for (int w = 0; w < Wd && nk < max_keep; ++w) {
                    const int base = w * 32, row = base + tid;
                    // the group's diagonal words and its removal word straight from shared memory (same address in every lane:
                    // broadcast loads, all independent of the decision chain; no shuffles)
                    uint32_t d[32];
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) d[jj] = mat[(base + jj) * Wd + w];
                    uint32_t cur = dead[w], kmask = 0;
                    int room = max_keep - nk;
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                        const bool keep = !((cur >> jj) & 1u) && room > 0;
                        if (keep) { kmask |= 1u << jj; cur |= d[jj]; --room; }
                    }
                    if ((kmask >> tid) & 1u) {
                        const int pos = nk + __popc(kmask & ((1u << tid) - 1u));
                        s_keep[pos] = s0 + row; kbox[pos] = fbox[row];
                    }
                    nk += __popc(kmask);
                    // branch-free (a data-dependent loop with a divergent body costs a convergence barrier per iteration, far
                    // more than 32 predicated loads): rows past nb are inside the allocation and masked by kmask
                    uint32_t acc = 0;
                    const uint32_t* mrow = mat + base * Wd + min(tid, Wd - 1);
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) acc |= mrow[jj * Wd] & (0u - ((kmask >> jj) & 1u));
                    if (tid < Wd) { removed |= acc; dead[tid] = removed; }
                    __syncwarp();
                }
                if (tid == 0) s_nkeep = nk;
            }
            __syncthreads();
            NMS_STAMP();
        }
    } else {
    // sorted, class-offset boxes (nms.py:144,150: boxes = x[:, :4] + cls * max_wh, fp32) + alive bitmask
    float4* sbox = p.ws_box + (size_t)b * p.P_max;
    for (int i = tid; i < n; i += kNmsThreads) {
        const float* c = cand + (size_t)pay[i] * 6;
        const float off = p.agnostic ? 0.f : __fmul_rn(c[5], p.max_wh);
        sbox[i] = make_float4(__fadd_rn(c[0], off), __fadd_rn(c[1], off), __fadd_rn(c[2], off), __fadd_rn(c[3], off));
    }
    for (int i = tid; i < (n + 31) / 32; i += kNmsThreads) {
        const int rem = n - i * 32;
        alive[i] = rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u);
    }
    if (tid == 0) { s_cur = 0; s_nkeep = 0; s_done = 0; }
    __syncthreads();

    while (true) {
        // -- next alive index >= s_cur (warp 0 scans the bitmask) --
        if (tid < 32) {
            int cur = s_cur, found = -1;
            const int nwords = (n + 31) / 32;
            for (int wbase = cur >> 5; wbase < nwords && found < 0; wbase += 32) {
                const int wi = wbase + tid;
                uint32_t word = wi < nwords ? alive[wi] : 0u;
                if (wi == (cur >> 5)) word &= ~((1u << (cur & 31)) - 1u);
                const unsigned has = __ballot_sync(0xffffffffu, word != 0u);
                if (has) {
                    const int src = __ffs(has) - 1;
                    const uint32_t wsel = __shfl_sync(0xffffffffu, word, src);
                    found = (wbase + src) * 32 + __ffs(wsel) - 1;
                }
            }
            if (tid == 0) {
                if (found < 0 || s_nkeep >= max_keep) s_done = 1;
                else { s_keep[s_nkeep++] = found; s_cur = found + 1; s_any = 0; }
            }
        }
        __syncthreads();
        if (s_done) break;
        const int i = s_cur - 1;
        const float4 bi = sbox[i];
        const float area_i = __fmul_rn(__fsub_rn(bi.z, bi.x), __fsub_rn(bi.w, bi.y));
        int any = 0;
        for (int j = i + 1 + tid; j < n; j += kNmsThreads) {
            if (!((alive[j >> 5] >> (j & 31)) & 1u)) continue;
            bool touches = false;
            const bool sup = iou_exceeds(bi, area_i, sbox[j], p.iou_thres, &touches);
            if (touches) any = 1;
            if (sup) atomicAnd(&alive[j >> 5], ~(1u << (j & 31)));
        }
        if (p.mode == 1) {
            if (any) s_any = 1;      // benign race: all writers store 1
            __syncthreads();
            if (!s_any) {
                // TorchNMS.nms early exit (nms.py:290-296): nothing intersects -> keep every remaining box, stop.
                // (the suppression pass above cleared nothing: iou == 0 for all of them)
                if (tid == 0) {
                    for (int j = i + 1; j < n && s_nkeep < max_keep; ++j)
                        if ((alive[j >> 5] >> (j & 31)) & 1u) s_keep[s_nkeep++] = j;
                    s_done = 1;
                }
                __syncthreads();
                break;
            }
        }
        __syncthreads();
    }
    }

    const int nk = s_nkeep;
    for (int k = tid; k < nk; k += kNmsThreads) {
        const int src = pay[s_keep[k]];
        const float* c = cand + (size_t)src * 6;
        float x1 = c[0], y1 = c[1], x2 = c[2], y2 = c[3];
        if (kScaled) {
            const float* sc = p.scale + (size_t)b * 5;
            const float gain = sc[0], pad_x = sc[1], pad_y = sc[2], orig_w = sc[3], orig_h = sc[4];
            x1 = __fdiv_rn(__fsub_rn(x1, pad_x), gain); y1 = __fdiv_rn(__fsub_rn(y1, pad_y), gain);
            x2 = __fdiv_rn(__fsub_rn(x2, pad_x), gain); y2 = __fdiv_rn(__fsub_rn(y2, pad_y), gain);
            x1 = fminf(fmaxf(x1, 0.f), orig_w); x2 = fminf(fmaxf(x2, 0.f), orig_w);
            y1 = fminf(fmaxf(y1, 0.f), orig_h); y2 = fminf(fmaxf(y2, 0.f), orig_h);
        } else if (p.do_scale) {
            x1 = __fdiv_rn(__fsub_rn(x1, p.pad_x), p.gain); y1 = __fdiv_rn(__fsub_rn(y1, p.pad_y), p.gain);
            x2 = __fdiv_rn(__fsub_rn(x2, p.pad_x), p.gain); y2 = __fdiv_rn(__fsub_rn(y2, p.pad_y), p.gain);
            x1 = fminf(fmaxf(x1, 0.f), p.orig_w); x2 = fminf(fmaxf(x2, 0.f), p.orig_w);
            y1 = fminf(fmaxf(y1, 0.f), p.orig_h); y2 = fminf(fmaxf(y2, 0.f), p.orig_h);
        }
        float* o = out + (size_t)k * 6;
        o[0] = x1; o[1] = y1; o[2] = x2; o[3] = y2; o[4] = c[4]; o[5] = c[5];
        if (p.out_idx) p.out_idx[(size_t)b * p.max_det + k] = cidx[src];
    }
    NMS_STAMP();
    if (p.debug && tid == 0) stamp[15] = n_stamp;
    if (tid == 0) p.out_count[b] = nk;
#undef NMS_STAMP
}

inline int next_pow2(int v) { int p = 32; while (p < v) p <<= 1; return p; }

}  // namespace

extern "C" int b2_decode(const void* const* level_logits, const int* level_h, const int* level_w, const int* level_stride,
                         int n_levels, int B, int nc, int lstride, float conf, const uint8_t* classes_mask,
                         float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, float* dense_out, void* stream) {
    B2_REQUIRE(n_levels >= 1 && n_levels <= kMaxLevels, "decode: n_levels=%d out of range", n_levels);
    B2_REQUIRE(nc >= 1 && lstride % 8 == 0 && lstride >= 64 + ((nc + 7) / 8) * 8, "decode: lstride=%d too small for nc=%d", lstride, nc);
    B2_REQUIRE(cand && cand_idx && cand_count && cand_cap > 0, "decode: candidate buffers required");
    DecodeParams p{};
    p.a_off[0] = 0;
    for (int l = 0; l < n_levels; ++l) {
        p.lv[l] = (const __nv_bfloat16*)level_logits[l];
        B2_REQUIRE(p.lv[l] && ((uintptr_t)p.lv[l] % 16 == 0), "decode: level %d pointer null/unaligned", l);
        p.h[l] = level_h[l]; p.w[l] = level_w[l]; p.stride[l] = level_stride[l];
        p.a_off[l + 1] = p.a_off[l] + level_h[l] * level_w[l];
    }
    p.n_levels = n_levels; p.B = B; p.nc = nc; p.lstride = lstride; p.A = p.a_off[n_levels];
    p.conf = conf; p.cmask = classes_mask; p.cand = cand; p.cand_idx = cand_idx; p.cand_count = cand_count;
    p.cand_cap = cand_cap; p.dense = dense_out;
    cudaStream_t st = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int32_t) * B, st));
    // conf outside (0, 1) (0 keeps everything, the dense-output callers use it): no pre-filter
    p.logit_lo = (conf > 0.f && conf < 1.f) ? logf(conf / (1.f - conf)) - 0.05f : -INFINITY;
    p.blk_off[0] = 0;
    for (int l = 0; l < n_levels; ++l) p.blk_off[l + 1] = p.blk_off[l] + b2_ceil_div(level_h[l] * level_w[l] * 8, 256);
    dim3 grid(p.blk_off[n_levels], B);
    if (dense_out) decode_kernel<true><<<grid, 256, 0, st>>>(p);
    else decode_kernel<false><<<grid, 256, 0, st>>>(p);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_candidates_from_head(const float* const* level_dist, const float* const* level_cls, const int* level_h, const int* level_w,
                                       const int* level_stride, int n_levels, int B, float conf, const uint8_t* classes_mask,
                                       float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, void* stream) {
    B2_REQUIRE(n_levels >= 1 && n_levels <= kMaxLevels, "candidates: n_levels=%d out of range", n_levels);
    B2_REQUIRE(cand && cand_idx && cand_count && cand_cap > 0, "candidates: candidate buffers required");
    HeadParams p{};
    p.a_off[0] = 0;
    for (int l = 0; l < n_levels; ++l) {
        B2_REQUIRE(level_dist[l] && level_cls[l], "candidates: level %d pointer null", l);
        p.dist[l] = level_dist[l]; p.cls[l] = level_cls[l];
        p.h[l] = level_h[l]; p.w[l] = level_w[l]; p.stride[l] = level_stride[l];
        p.a_off[l + 1] = p.a_off[l] + level_h[l] * level_w[l];
    }
    p.n_levels = n_levels; p.A = p.a_off[n_levels]; p.B = B; p.conf = conf; p.cmask = classes_mask;
    B2_REQUIRE(conf > 0.f && conf < 1.f, "candidates: conf must be in (0, 1)");
    p.logit_lo = logf(conf / (1.f - conf)) - 0.05f;
    p.blk_off[0] = 0;
    for (int l = 0; l < n_levels; ++l) p.blk_off[l + 1] = p.blk_off[l] + b2_ceil_div(level_h[l] * level_w[l], kHcThreads * kHcPer);
    p.cand = cand; p.cand_idx = cand_idx; p.cand_count = cand_count; p.cand_cap = cand_cap;
    cudaStream_t st = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int32_t) * B, st));
    // (one block per chunk.  Measured at the bench size, 256 images x 27 200 anchors, L2 flushed: 128 threads x 4 records 22.6 us;
    //  256 x 8 26.6; 256 x 4 and 128 x 8 24.6; 64 x 2 36.9; a one-wave grid walking several chunks per block 32; 16-byte loads of
    //  record pairs 33: the kernel is a short burst of loads, finer blocks fill and drain the SMs more evenly)
    head_candidates_kernel<<<dim3(p.blk_off[n_levels], B), kHcThreads, 0, st>>>(p);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_candidates_from_dense(const float* pred, int B, int nc, int no, int A, float conf, const uint8_t* classes_mask,
                                        float* cand, int32_t* cand_idx, int32_t* cand_count, int cand_cap, void* stream) {
    B2_REQUIRE(pred && cand && cand_idx && cand_count, "candidates: null pointer");
    B2_REQUIRE(B >= 1 && nc >= 1 && no >= 4 + nc && A >= 1 && cand_cap >= 1, "candidates: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int32_t) * B, st));
    dense_candidates_kernel<<<dim3(b2_ceil_div(A, 256), B), 256, 0, st>>>(pred, nc, no, A, conf, classes_mask, cand, cand_idx, cand_count, cand_cap);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" size_t b2_nms_workspace_bytes(int B, int cand_cap) {
    const size_t P = (size_t)next_pow2(cand_cap);
    return (size_t)B * (P * (8 + 4 + 16)) + 256;
}

static int launch_nms(const float* cand, const int32_t* cand_idx, const int32_t* cand_count, int cand_cap, int B,
                      float iou_thres, int max_det, int max_nms, int agnostic, float max_wh, int mode,
                      float gain, float pad_x, float pad_y, float orig_w, float orig_h, int do_scale, const float* scale,
                      float* out, int32_t* out_count, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream) {
    B2_REQUIRE(cand && cand_idx && cand_count && out && out_count && workspace, "nms: null pointer");
    B2_REQUIRE(max_det >= 1 && max_det <= kMaxKeep, "nms: max_det=%d out of range [1,%d]", max_det, kMaxKeep);
    B2_REQUIRE(mode == 0 || mode == 1, "nms: mode must be 0 (exact) or 1 (legacy TorchNMS)");
    // cand_cap bounds the candidate LIST (callers size it to the anchor count, so the conf filter can never overflow it and the
    // result never depends on the order candidates were appended in); the bitmask of the legacy walk covers max_nms sorted entries
    B2_REQUIRE(cand_cap >= 1 && cand_cap <= (1 << 22), "nms: cand_cap=%d out of range [1,%d]", cand_cap, 1 << 22);
    B2_REQUIRE(max_nms >= 1 && max_nms <= kMaxCand, "nms: max_nms=%d out of range [1,%d]", max_nms, kMaxCand);
    B2_REQUIRE(workspace_bytes >= b2_nms_workspace_bytes(B, cand_cap), "nms: workspace too small");
    B2_REQUIRE(iou_thres >= 0.f && iou_thres <= 1.f, "Invalid IoU %f, valid values are between 0.0 and 1.0", iou_thres);
    NmsParams p{};
    p.cand = cand; p.cand_idx = cand_idx; p.cand_count = cand_count; p.cand_cap = cand_cap; p.B = B;
    p.iou_thres = iou_thres; p.max_det = max_det; p.max_nms = max_nms; p.agnostic = agnostic; p.max_wh = max_wh; p.mode = mode;
    p.gain = gain; p.pad_x = pad_x; p.pad_y = pad_y; p.orig_w = orig_w; p.orig_h = orig_h; p.do_scale = do_scale; p.scale = scale;
    p.out = out; p.out_count = out_count; p.out_idx = out_idx;
    const size_t P = (size_t)next_pow2(cand_cap);
    char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    p.ws_box = (float4*)ws; ws += (size_t)B * P * 16;
    p.ws_keys = (unsigned long long*)ws; ws += (size_t)B * P * 8;
    p.ws_pay = (int32_t*)ws;
    p.P_max = (int)P;
    { static const bool dbg = [] { const char* v = getenv("B2_NMS_DEBUG"); return v && atoi(v) != 0; }(); p.debug = dbg ? 1 : 0; }
    const size_t dyn = (size_t)kSmemSort * 12 + (size_t)kFastN * 16 + (size_t)kFastN * ((kFastN + 31) / 32) * 4 + (size_t)kMaxKeep * 16;
    // the attribute belongs to the current device's context: set on every call (a microsecond of host time), not once per process
    auto kernel = scale ? nms_kernel<true> : nms_kernel<false>;
    B2_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    kernel<<<B, kNmsThreads, dyn, (cudaStream_t)stream>>>(p);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_nms(const float* cand, const int32_t* cand_idx, const int32_t* cand_count, int cand_cap, int B,
                      float iou_thres, int max_det, int max_nms, int agnostic, float max_wh, int mode,
                      float gain, float pad_x, float pad_y, float orig_w, float orig_h, int do_scale,
                      float* out, int32_t* out_count, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream) {
    return launch_nms(cand, cand_idx, cand_count, cand_cap, B, iou_thres, max_det, max_nms, agnostic, max_wh, mode,
                      gain, pad_x, pad_y, orig_w, orig_h, do_scale, nullptr, out, out_count, out_idx, workspace, workspace_bytes, stream);
}

extern "C" int b2_nms_scaled(const float* cand, const int32_t* cand_idx, const int32_t* cand_count, int cand_cap, int B,
                             float iou_thres, int max_det, int max_nms, int agnostic, float max_wh, int mode, const float* scale,
                             float* out, int32_t* out_count, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream) {
    B2_REQUIRE(scale, "nms_scaled: null scale table");
    return launch_nms(cand, cand_idx, cand_count, cand_cap, B, iou_thres, max_det, max_nms, agnostic, max_wh, mode,
                      1.f, 0.f, 0.f, 0.f, 0.f, 0, scale, out, out_count, out_idx, workspace, workspace_bytes, stream);
}
