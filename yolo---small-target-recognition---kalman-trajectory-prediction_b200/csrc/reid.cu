// BoT-SORT ReID on the detector's own features (botsort.yaml `with_reid: True`, `model: auto`) for sm_100a.
//
//   reid_gather_kernel  models/yolo/detect/predict.py get_obj_feats: the appearance vector of a kept detection is its anchor's
//                       row of the Detect input map of its level, averaged over groups of C_l / s consecutive channels
//                       (s = min C_l).  One warp per detection: the NHWC bf16 row (2 C_l contiguous bytes) is read with 16-byte
//                       loads, sums in fp32, one division by the group size.
//   reid_update_kernel  trackers/bot_sort.py BOTrack.update_features, batched over rows: feat /= |feat|; smooth = feat the first
//                       time, else 0.9 smooth + 0.1 feat; smooth /= |smooth| -- all float32.
#include "common.cuh"

void b2_count_launch(int n);

namespace {

constexpr int kMaxReidLevels = 8;

struct ReidLevels {
    const __nv_bfloat16* ptr[kMaxReidLevels];     // first channel of the level's slice, image 0, anchor 0
    int cstride[kMaxReidLevels];
    int C[kMaxReidLevels];
    int hw[kMaxReidLevels];
    int start[kMaxReidLevels + 1];                // first anchor id of each level (Detect order), start[n] = anchors per image
    int n;
    int vec;                                       // every slice 16-byte aligned: 8-channel vector loads
};

__device__ __forceinline__ void bf16x8_to_f32(const uint4 v, float* f) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 t = __bfloat1622float2(h[k]);
        f[2 * k] = t.x;
        f[2 * k + 1] = t.y;
    }
}

__global__ void __launch_bounds__(256) reid_gather_kernel(const ReidLevels L, const int32_t* __restrict__ det_idx, const int32_t* __restrict__ det_count,
                                                          int B, int max_det, int s, float* __restrict__ out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B * max_det) return;
    const int b = warp / max_det, k = warp - b * max_det;
    if (k >= min(det_count[b], max_det)) return;
    const int a = det_idx[warp];
    if (a < 0 || a >= L.start[L.n]) return;
    int l = 0;
    while (a >= L.start[l + 1]) ++l;
    const int C = L.C[l], g = C / s;
    const __nv_bfloat16* row = L.ptr[l] + ((size_t)b * L.hw[l] + (a - L.start[l])) * L.cstride[l];
    float* o = out + (size_t)warp * s;
    const float gf = (float)g;
    if (L.vec && g % 8 == 0) {                     // a group spans g / 8 whole vectors
        const uint4* rv = reinterpret_cast<const uint4*>(row);
        for (int f = lane; f < s; f += 32) {
            float acc = 0.f, v[8];
            for (int q = 0; q < g / 8; ++q) {
                bf16x8_to_f32(__ldg(rv + f * (g / 8) + q), v);
#pragma unroll
                for (int e = 0; e < 8; ++e) acc = __fadd_rn(acc, v[e]);
            }
            o[f] = __fdiv_rn(acc, gf);
        }
    } else if (L.vec && 8 % g == 0) {              // one vector holds 8 / g whole groups
        const uint4* rv = reinterpret_cast<const uint4*>(row);
        for (int q = lane; q < C / 8; q += 32) {
            float v[8];
            bf16x8_to_f32(__ldg(rv + q), v);
            for (int f = 0; f < 8 / g; ++f) {
                float acc = 0.f;
                for (int e = 0; e < g; ++e) acc = __fadd_rn(acc, v[f * g + e]);
                o[q * (8 / g) + f] = __fdiv_rn(acc, gf);
            }
        }
    } else {                                       // any other group size / alignment: scalar loads
        for (int f = lane; f < s; f += 32) {
            float acc = 0.f;
            for (int e = 0; e < g; ++e) acc = __fadd_rn(acc, __bfloat162float(row[f * g + e]));
            o[f] = __fdiv_rn(acc, gf);
        }
    }
}

// |x| of a float32 vector held by one warp (float64 sum of squares, rounded once to float32)
__device__ __forceinline__ float warp_norm(const float* x, int D, int lane) {
    double ss = 0.0;
    for (int k = lane; k < D; k += 32) ss += (double)x[k] * (double)x[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    return (float)sqrt(ss);
}

__global__ void __launch_bounds__(256) reid_update_kernel(float* __restrict__ curr, float* __restrict__ smooth, const uint8_t* __restrict__ has_smooth,
                                                          int N, int D) {
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= N) return;
    float* c = curr + (size_t)r * D;
    float* sm = smooth + (size_t)r * D;
    const float n1 = warp_norm(c, D, lane);
    for (int k = lane; k < D; k += 32) c[k] = __fdiv_rn(c[k], n1);          // feat /= |feat|
    __syncwarp();
    const bool prev = has_smooth && has_smooth[r];
    const float alpha = 0.9f, beta = (float)(1.0 - 0.9);                     // self.alpha * smooth + (1 - self.alpha) * feat
    for (int k = lane; k < D; k += 32) sm[k] = prev ? __fadd_rn(__fmul_rn(alpha, sm[k]), __fmul_rn(beta, c[k])) : c[k];
    __syncwarp();
    const float n2 = warp_norm(sm, D, lane);
    for (int k = lane; k < D; k += 32) {
        const float v = __fdiv_rn(sm[k], n2);
        sm[k] = v;
        if (!prev) c[k] = v;       // first call: smooth_feat IS curr_feat (same array), so the in-place renormalisation reaches both
    }
}

}  // namespace

extern "C" int b2_reid_gather(const void* const* level_ptr, const int* level_h, const int* level_w, const int* level_cstride,
                              const int* level_coff, const int* level_c, int n_levels, const int32_t* det_idx, const int32_t* det_count,
                              int B, int max_det, int s, float* out, void* stream) {
    B2_REQUIRE(n_levels >= 1 && n_levels <= kMaxReidLevels, "reid_gather: 1..%d levels", kMaxReidLevels);
    B2_REQUIRE(B >= 1 && max_det >= 0 && s >= 1, "reid_gather: bad shape");
    if (max_det == 0) return B2_OK;
    B2_REQUIRE(level_ptr && level_h && level_w && level_cstride && level_coff && level_c && det_idx && det_count && out,
               "reid_gather: null pointer");
    ReidLevels L{};
    L.n = n_levels;
    L.vec = 1;
    L.start[0] = 0;
    for (int l = 0; l < n_levels; ++l) {
        B2_REQUIRE(level_ptr[l] && level_h[l] > 0 && level_w[l] > 0, "reid_gather: level %d: empty", l);
        B2_REQUIRE(level_c[l] >= s && level_c[l] % s == 0, "reid_gather: level %d: %d channels are not a multiple of s = %d", l, level_c[l], s);
        B2_REQUIRE(level_coff[l] >= 0 && level_coff[l] + level_c[l] <= level_cstride[l], "reid_gather: level %d: channel slice outside the buffer", l);
        L.ptr[l] = reinterpret_cast<const __nv_bfloat16*>(level_ptr[l]) + level_coff[l];
        L.cstride[l] = level_cstride[l];
        L.C[l] = level_c[l];
        L.hw[l] = level_h[l] * level_w[l];
        L.start[l + 1] = L.start[l] + L.hw[l];
        if ((uintptr_t)L.ptr[l] % 16 || level_cstride[l] % 8 || level_c[l] % 8) L.vec = 0;
    }
    const long long warps = (long long)B * max_det;
    reid_gather_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(L, det_idx, det_count, B, max_det, s, out);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_reid_update(float* curr, float* smooth, const uint8_t* has_smooth, int N, int D, void* stream) {
    B2_REQUIRE(N >= 0 && D >= 1, "reid_update: bad shape");
    if (N == 0) return B2_OK;
    B2_REQUIRE(curr && smooth, "reid_update: null pointer");
    reid_update_kernel<<<b2_ceil_div(N * 32, 256), 256, 0, (cudaStream_t)stream>>>(curr, smooth, has_smooth, N, D);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}
