// Association kernels of the upstream tracker plug-in (ByteTrack / BoT-SORT) for sm_100a, batched over independent
// problems (one per video stream and association stage).
//
//   iou_cost_kernel    ultralytics/trackers/utils/matching.py:66-113 iou_distance (bbox_ioa(.., iou=True),
//                      utils/metrics.py:19-52) and :135-157 fuse_score, in the reference's float32 operation order.
//   lap_kernel         matching.py:20-63 linear_assignment on its default branch, lap.lapjv(cost, extend_cost=True,
//                      cost_limit=thresh).  `lap` (gatagat/lap, pinned "lap>=0.5.12" by the reference) is a third-party
//                      dependency that is not vendored: its published algorithm is restated.  With extend_cost and a finite
//                      cost_limit lapjv solves the square (n+m) problem [[C, L/2], [L/2, 0]] (L = cost_limit): every real
//                      pair costs c_ij, every unmatched row or column L/2.  The optimum is the partial matching that
//                      minimises sum(c_ij - L) over its pairs, so the kernel solves exactly that: the n x (m + n)
//                      assignment in which row i may also take a private zero-cost column.  The solver is the shortest-
//                      augmenting-path (Hungarian with potentials) scheme lapjv's augmentation phase uses, in float64,
//                      one CTA per problem: the scan over the columns is spread over the threads, the arg-min is a
//                      block reduction with ties to the lowest column (deterministic).  Any exact solver returns the
//                      same matching unless two candidate matchings have bit-identical float64 totals.
//                      Instantiated for float costs (b2_linear_assignment) and float64 costs (b2_linear_assignment_f64).
//   botsort_cost_kernel bot_sort.py BOTSORT.get_dists with ReID: the IoU / fused term of iou_cost_kernel, the proximity mask,
//                      the float64 cosine embedding distance with the appearance gate, their minimum in float64.
#include "common.cuh"

#include <float.h>

void b2_count_launch(int n);

namespace {

// iou_distance of one (track, detection) pair, float32 in the reference's operation order
__device__ __forceinline__ float iou_dist(const float4 p, const float4 q) {
    // bbox_ioa: (min(x2) - max(x1)).clip(0) * (min(y2) - max(y1)).clip(0); area = area2 + area1 - inter; inter / (area + eps)
    const float iw = fmaxf(__fsub_rn(fminf(p.z, q.z), fmaxf(p.x, q.x)), 0.f);
    const float ih = fmaxf(__fsub_rn(fminf(p.w, q.w), fmaxf(p.y, q.y)), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float area2 = __fmul_rn(__fsub_rn(q.z, q.x), __fsub_rn(q.w, q.y));
    const float area1 = __fmul_rn(__fsub_rn(p.z, p.x), __fsub_rn(p.w, p.y));
    const float area = __fsub_rn(__fadd_rn(area2, area1), inter);
    const float iou = __fdiv_rn(inter, __fadd_rn(area, 1e-7f));
    return __fsub_rn(1.f, iou);                          // iou_distance: 1 - ious
}

// fuse_score: 1 - (1 - cost) * score
__device__ __forceinline__ float fuse_dist(float c, float score) { return __fsub_rn(1.f, __fmul_rn(__fsub_rn(1.f, c), score)); }

__global__ void __launch_bounds__(256) iou_cost_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ score_b,
                                                       const int32_t* __restrict__ na, const int32_t* __restrict__ nb, int n_max, int m_max,
                                                       float* __restrict__ cost) {
    const int s = blockIdx.z;
    const int n = na ? min(na[s], n_max) : n_max, m = nb ? min(nb[s], m_max) : m_max;
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (i >= n || j >= m) return;
    const float4 p = reinterpret_cast<const float4*>(a)[(size_t)s * n_max + i];
    const float4 q = reinterpret_cast<const float4*>(b)[(size_t)s * m_max + j];
    float c = iou_dist(p, q);
    if (score_b) c = fuse_dist(c, score_b[(size_t)s * m_max + j]);
    cost[((size_t)s * n_max + i) * m_max + j] = c;
}

// BOTSORT.get_dists with ReID (bot_sort.py:154-232, matching.embedding_distance).  A 16 x 16 tile of (track, detection) pairs per
// CTA, one thread per pair; the feature rows of the tile are staged through shared memory kBcK floats at a time.  The cosine
// distance is scipy's cdist(.., 'cosine') in float64: row norms sqrt(sum u_k^2) (once per row, by the threads of the tile's
// first column / row), dot product summed in k order, cos = dot / (|u| |v|) clamped to [-1, 1], 1 - cos.  The products of two
// floats are exact in float64, so the sums do not depend on FMA contraction.
constexpr int kBcT = 16, kBcK = 64;

__global__ void __launch_bounds__(kBcT * kBcT) botsort_cost_kernel(
        const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ score_b, const int32_t* __restrict__ na,
        const int32_t* __restrict__ nb, const float* __restrict__ feat_a, const float* __restrict__ feat_b, int D, int n_max, int m_max,
        float prox, double app, double* __restrict__ cost) {
    __shared__ float fa[kBcT][kBcK + 1], fb[kBcT][kBcK + 1];
    __shared__ double norm_a[kBcT], norm_b[kBcT];
    const int s = blockIdx.z, tx = threadIdx.x, ty = threadIdx.y, tid = ty * kBcT + tx;
    const int n = na ? min(na[s], n_max) : n_max, m = nb ? min(nb[s], m_max) : m_max;
    const int i0 = blockIdx.y * kBcT, j0 = blockIdx.x * kBcT;
    if (i0 >= n || j0 >= m) return;                      // whole tile outside this problem (uniform over the CTA)
    const int i = i0 + ty, j = j0 + tx;
    const float* A = feat_a + (size_t)s * n_max * D;
    const float* Bf = feat_b + (size_t)s * m_max * D;
    double dot = 0.0, ssa = 0.0, ssb = 0.0;
    for (int k0 = 0; k0 < D; k0 += kBcK) {
        const int kn = min(kBcK, D - k0);
        for (int e = tid; e < kBcT * kBcK; e += kBcT * kBcT) {
            const int r = e / kBcK, k = e % kBcK;
            if (k < kn) {
                fa[r][k] = i0 + r < n ? A[(size_t)(i0 + r) * D + k0 + k] : 0.f;
                fb[r][k] = j0 + r < m ? Bf[(size_t)(j0 + r) * D + k0 + k] : 0.f;
            }
        }
        __syncthreads();
        for (int k = 0; k < kn; ++k) dot = __dadd_rn(dot, __dmul_rn((double)fa[ty][k], (double)fb[tx][k]));
        if (tx == 0)
            for (int k = 0; k < kn; ++k) ssa = __dadd_rn(ssa, __dmul_rn((double)fa[ty][k], (double)fa[ty][k]));
        if (ty == 0)
            for (int k = 0; k < kn; ++k) ssb = __dadd_rn(ssb, __dmul_rn((double)fb[tx][k], (double)fb[tx][k]));
        __syncthreads();
    }
    if (tx == 0) norm_a[ty] = sqrt(ssa);
    if (ty == 0) norm_b[tx] = sqrt(ssb);
    __syncthreads();
    if (i >= n || j >= m) return;
    const float4 p = reinterpret_cast<const float4*>(a)[(size_t)s * n_max + i];
    const float4 q = reinterpret_cast<const float4*>(b)[(size_t)s * m_max + j];
    const float d_iou = iou_dist(p, q);
    const float d = score_b ? fuse_dist(d_iou, score_b[(size_t)s * m_max + j]) : d_iou;
    double cs = dot / (norm_a[ty] * norm_b[tx]);
    if (fabs(cs) > 1.0) cs = copysign(1.0, cs);
    double emb = 1.0 - cs;
    emb = emb < 0.0 ? 0.0 : emb;                         // np.maximum(0.0, cdist) (a NaN stays NaN)
    emb = emb / 2.0;
    if (emb > app) emb = 1.0;                            // emb_dists[emb_dists > (1 - appearance_thresh)] = 1.0 (float64)
    if (d_iou > prox) emb = 1.0;                         // emb_dists[dists_mask] = 1.0, mask in float32 on the unfused IoU distance
    double c = (double)d;
    if (!(c <= emb)) c = emb;                            // np.minimum(dists, emb_dists) -> float64
    cost[((size_t)s * n_max + i) * m_max + j] = c;
}

constexpr int kLapThreads = 256;
constexpr double kBig = 1e18;

// shared memory: double v[Mc+1], minv[Mc+1], u[n+1]; int p[Mc+1], way[Mc+1]; uint8 used[Mc+1]   (Mc = m + n columns, 1-based)
// T: float (ByteTrack, BoT-SORT without ReID) or double (the BoT-SORT ReID cost); the solver itself is float64 either way.
template <typename T>
__global__ void __launch_bounds__(kLapThreads) lap_kernel(const T* __restrict__ cost, const int32_t* __restrict__ na, const int32_t* __restrict__ nb,
                                                          int n_max, int m_max, T thresh, int32_t* __restrict__ x_out, int32_t* __restrict__ y_out) {
    extern __shared__ double sm_d[];
    __shared__ double r_val[kLapThreads / 32];
    __shared__ int r_idx[kLapThreads / 32];
    __shared__ int s_j0, s_j1;
    __shared__ double s_delta;
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = na ? min(na[s], n_max) : n_max, m = nb ? min(nb[s], m_max) : m_max;
    int32_t* x = x_out + (size_t)s * n_max;
    int32_t* y = y_out + (size_t)s * m_max;
    for (int i = tid; i < n_max; i += kLapThreads) x[i] = -1;
    for (int j = tid; j < m_max; j += kLapThreads) y[j] = -1;
    if (n == 0 || m == 0) return;
    const int Mc = m + n;
    double* v = sm_d;
    double* minv = v + (Mc + 1);
    double* u = minv + (Mc + 1);
    int* p = reinterpret_cast<int*>(u + (n + 1));
    int* way = p + (Mc + 1);
    uint8_t* used = reinterpret_cast<uint8_t*>(way + (Mc + 1));
    const T* C = cost + (size_t)s * n_max * m_max;
    const double L = (double)thresh;
    for (int j = tid; j <= Mc; j += kLapThreads) { v[j] = 0.0; p[j] = 0; }
    for (int i = tid; i <= n; i += kLapThreads) u[i] = 0.0;
    __syncthreads();
    for (int i = 1; i <= n; ++i) {
        for (int j = tid; j <= Mc; j += kLapThreads) { minv[j] = kBig; used[j] = 0; way[j] = 0; }
        if (tid == 0) { p[0] = i; s_j0 = 0; }
        __syncthreads();
        while (true) {
            const int j0 = s_j0;
            const int i0 = p[j0];
            const double ui0 = u[i0];
            __syncthreads();                               // everyone has read p[j0] / s_j0 before they change
            if (tid == 0) used[j0] = 1;
            // relax the free columns from row i0, thread-local arg-min (lowest column on ties)
            double best = kBig * 4.0; int bj = 0x7fffffff;
            for (int j = 1 + tid; j <= Mc; j += kLapThreads) {
                if (used[j] || j == j0) continue;
                const double cij = j <= m ? (double)C[(size_t)(i0 - 1) * m_max + (j - 1)] - L : (j - m == i0 ? 0.0 : kBig);
                const double cur = cij - ui0 - v[j];
                double mv = minv[j];
                if (cur < mv) { mv = cur; minv[j] = cur; way[j] = j0; }
                if (mv < best || (mv == best && j < bj)) { best = mv; bj = j; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
                if (ob < best || (ob == best && oj < bj)) { best = ob; bj = oj; }
            }
            if (lane == 0) { r_val[warp] = best; r_idx[warp] = bj; }
            __syncthreads();
            if (tid == 0) {
                double b2 = r_val[0]; int j2 = r_idx[0];
                for (int w = 1; w < kLapThreads / 32; ++w)
                    if (r_val[w] < b2 || (r_val[w] == b2 && r_idx[w] < j2)) { b2 = r_val[w]; j2 = r_idx[w]; }
                s_delta = b2; s_j1 = j2;
            }
            __syncthreads();
            const double delta = s_delta;
            const int j1 = s_j1;
            for (int j = tid; j <= Mc; j += kLapThreads) {
                if (used[j]) { u[p[j]] += delta; v[j] -= delta; }     // p[j] distinct over used columns: no two threads touch one u
                else minv[j] -= delta;
            }
            if (tid == 0) s_j0 = j1;
            __syncthreads();
            if (p[j1] == 0) break;
        }
        if (tid == 0) {                                    // augment along the alternating path
            int j0 = s_j0;
            while (j0) { const int j1 = way[j0]; p[j0] = p[j1]; j0 = j1; }
        }
        __syncthreads();
    }
    for (int j = 1 + tid; j <= m; j += kLapThreads) {
        const int i = p[j];
        // a real pair in the optimum has c_ij < cost_limit (otherwise leaving both unmatched is cheaper); the guard only
        // matters for c_ij == cost_limit exactly
        if (i > 0 && (double)C[(size_t)(i - 1) * m_max + (j - 1)] < L) { x[i - 1] = j - 1; y[j - 1] = i - 1; }
    }
}

}  // namespace

extern "C" int b2_iou_cost(const float* boxes_a, const float* boxes_b, const float* scores_b, const int32_t* na, const int32_t* nb,
                           int S, int n_max, int m_max, float* cost, void* stream) {
    B2_REQUIRE(S >= 1 && n_max >= 0 && m_max >= 0, "iou_cost: bad shape");
    if (n_max == 0 || m_max == 0) return B2_OK;
    B2_REQUIRE(boxes_a && boxes_b && cost, "iou_cost: null pointer");
    B2_REQUIRE((uintptr_t)boxes_a % 16 == 0 && (uintptr_t)boxes_b % 16 == 0, "iou_cost: boxes must be 16-byte aligned");
    B2_REQUIRE(n_max <= 65535 && S <= 65535, "iou_cost: too many rows / problems");
    dim3 grid(b2_ceil_div(m_max, 256), n_max, S);
    iou_cost_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(boxes_a, boxes_b, scores_b, na, nb, n_max, m_max, cost);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_botsort_cost(const float* boxes_a, const float* boxes_b, const float* scores_b, const int32_t* na, const int32_t* nb,
                               const float* feat_a, const float* feat_b, int D, int S, int n_max, int m_max, float prox_limit,
                               double app_limit, double* cost, void* stream) {
    B2_REQUIRE(S >= 1 && n_max >= 0 && m_max >= 0 && D >= 1, "botsort_cost: bad shape");
    if (n_max == 0 || m_max == 0) return B2_OK;
    B2_REQUIRE(boxes_a && boxes_b && feat_a && feat_b && cost, "botsort_cost: null pointer");
    B2_REQUIRE((uintptr_t)boxes_a % 16 == 0 && (uintptr_t)boxes_b % 16 == 0, "botsort_cost: boxes must be 16-byte aligned");
    B2_REQUIRE(b2_ceil_div(n_max, kBcT) <= 65535 && S <= 65535, "botsort_cost: too many rows / problems");
    dim3 grid(b2_ceil_div(m_max, kBcT), b2_ceil_div(n_max, kBcT), S);
    botsort_cost_kernel<<<grid, dim3(kBcT, kBcT), 0, (cudaStream_t)stream>>>(boxes_a, boxes_b, scores_b, na, nb, feat_a, feat_b, D, n_max,
                                                                            m_max, prox_limit, app_limit, cost);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

template <typename T>
static int linear_assignment(const T* cost, const int32_t* na, const int32_t* nb, int S, int n_max, int m_max, T thresh,
                             int32_t* x_out, int32_t* y_out, void* stream) {
    B2_REQUIRE(S >= 1 && n_max >= 0 && m_max >= 0, "linear_assignment: bad shape");
    B2_REQUIRE((n_max == 0 || x_out) && (m_max == 0 || y_out), "linear_assignment: null output");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_max == 0 || m_max == 0) {
        if (n_max) B2_CUDA(cudaMemsetAsync(x_out, 0xFF, sizeof(int32_t) * (size_t)S * n_max, st));
        if (m_max) B2_CUDA(cudaMemsetAsync(y_out, 0xFF, sizeof(int32_t) * (size_t)S * m_max, st));
        return B2_OK;
    }
    B2_REQUIRE(cost, "linear_assignment: null cost matrix");
    const size_t Mc = (size_t)n_max + m_max + 1;
    const size_t smem = 8 * (2 * Mc + n_max + 1) + 4 * 2 * Mc + Mc + 16;
    B2_REQUIRE(smem <= 200 * 1024, "linear_assignment: %d x %d is too large for one CTA's shared memory", n_max, m_max);
    if (smem > 48 * 1024) B2_CUDA(cudaFuncSetAttribute(lap_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lap_kernel<T><<<S, kLapThreads, smem, st>>>(cost, na, nb, n_max, m_max, thresh, x_out, y_out);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_linear_assignment(const float* cost, const int32_t* na, const int32_t* nb, int S, int n_max, int m_max, float thresh,
                                    int32_t* x_out, int32_t* y_out, void* stream) {
    return linear_assignment<float>(cost, na, nb, S, n_max, m_max, thresh, x_out, y_out, stream);
}

extern "C" int b2_linear_assignment_f64(const double* cost, const int32_t* na, const int32_t* nb, int S, int n_max, int m_max, double thresh,
                                        int32_t* x_out, int32_t* y_out, void* stream) {
    return linear_assignment<double>(cost, na, nb, S, n_max, m_max, thresh, x_out, y_out, stream);
}
