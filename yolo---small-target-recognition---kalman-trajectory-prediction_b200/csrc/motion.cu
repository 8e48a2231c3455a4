// Global camera-motion detection for S streams on the GPU: the 'optical_flow' method of the reference's
// camera_motion_compensation/global_motion_detector.py (:113-184) and the global-reset rule of
// motion_compensated_multi_tracker.py (:75-146), restated per stream.
//
//   gray_kernel + pyrdown_kernel   cv2.cvtColor(BGR2GRAY) and three cv2.pyrDown levels, bit-exact (integer arithmetic)
//   eig_kernel                     cv2.cornerMinEigenVal(gray, blockSize=7, ksize=3), fp32 (summation order differs from cv2)
//   gftt_* kernels                 goodFeaturesToTrack(maxCorners=200, qualityLevel=0.01, minDistance=15) on that response
//   lk_kernel                      calcOpticalFlowPyrLK(winSize=21x21, maxLevel=3, COUNT|EPS 30 / 0.01), one warp per point
//   decide_kernel                  detect_motion's statistics + thresholds and _should_global_reset, one CTA per stream
//
// Frames are HWC BGR uint8 at per-stream byte offsets (the ops.pack_frames layout).  A pyramid buffer holds, per stream, the four
// gray levels back to back; b2_pyramid_layout gives the offsets.  The LK kernel computes the Scharr derivatives of the previous
// level from the image on the fly instead of storing them (DESIGN.md section 4).
#include <float.h>

#include <algorithm>
#include <new>

#include "common.cuh"

void b2_count_launch(int n);

namespace {

constexpr int kLevels = 4;          // level 0 + maxLevel 3
constexpr int kWin = 21;            // winSize
constexpr int kWinArea = kWin * kWin;
constexpr int kPerLane = (kWinArea + 31) / 32;
constexpr int kMaxCorners = 200;
constexpr int kMinDist2 = 15 * 15;
constexpr int kSortKeys = 16384;    // selection: 8192 best keys + 8192 incoming per bitonic sort (128 KiB of shared memory)
constexpr int kKeep = kSortKeys / 2;
constexpr int kSelThreads = 1024;

struct PyrView {
    uint8_t* base;
    const long long* off;   // [S][4] byte offset of each level
    const int* hw;          // [S][4][2] {h, w}
};

// BORDER_REFLECT_101 for any offset (cv2's borderInterpolate; a one-pixel side maps to 0)
__device__ __forceinline__ int reflect101(int p, int n) {
    if (n == 1) return 0;
    while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
    return p;
}

// buildOpticalFlowPyramid keeps level l + 1 only while it is larger than the window in both sides: the LK start level of a stream
__device__ __forceinline__ int lk_max_level(const int* hw) {
    int L = 0;
    while (L < kLevels - 1 && hw[2 * (L + 1)] > kWin && hw[2 * (L + 1) + 1] > kWin) ++L;
    return L;
}

// ------------------------------------------------------------------------------------------------------------------
// gray + pyramid
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gray_kernel(const uint8_t* __restrict__ frames, const long long* __restrict__ foff, PyrView p) {
    const int s = blockIdx.y;
    const int h = p.hw[s * 8], w = p.hw[s * 8 + 1];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h * w) return;
    const uint8_t* src = frames + foff[s] + (size_t)i * 3;
    // cv2 (4.13) COLOR_BGR2GRAY on uint8: B 3735, G 19235, R 9798 in 15-bit fixed point, rounded
    const int v = src[0] * 3735 + src[1] * 19235 + src[2] * 9798;
    p.base[p.off[s * 4] + i] = (uint8_t)((v + (1 << 14)) >> 15);
}

// level l -> l + 1: 5x5 binomial (1 4 6 4 1)^2 / 256 with REFLECT_101 on the source, (sum + 128) >> 8
__global__ void __launch_bounds__(256) pyrdown_kernel(PyrView p, int l) {
    const int s = blockIdx.y;
    const int sh = p.hw[s * 8 + l * 2], sw = p.hw[s * 8 + l * 2 + 1];
    const int dh = p.hw[s * 8 + (l + 1) * 2], dw = p.hw[s * 8 + (l + 1) * 2 + 1];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dh * dw) return;
    const int y = i / dw, x = i - y * dw;
    const uint8_t* src = p.base + p.off[s * 4 + l];
    int xs[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) xs[k] = reflect101(2 * x + k - 2, sw);
    const int wk[5] = {1, 4, 6, 4, 1};
    int acc = 0;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        const uint8_t* row = src + (size_t)reflect101(2 * y + r - 2, sh) * sw;
        const int t = row[xs[0]] + 4 * row[xs[1]] + 6 * row[xs[2]] + 4 * row[xs[3]] + row[xs[4]];
        acc += wk[r] * t;
    }
    p.base[p.off[s * 4 + l + 1] + i] = (uint8_t)((acc + 128) >> 8);
}

// ------------------------------------------------------------------------------------------------------------------
// cornerMinEigenVal(blockSize 7, ksize 3): Sobel * 1/(4*7*255), 7x7 unnormalised box sums of dx^2, dx dy, dy^2 (REFLECT_101 on
// the products), (a + c) - sqrt((a - c)^2 + b^2) with a, c halved.  One 32x8 output tile per block.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTX = 32, kTY = 8, kR = 3;
__global__ void __launch_bounds__(kTX * kTY) eig_kernel(PyrView p, const long long* __restrict__ pix_off, float* __restrict__ eig) {
    __shared__ float cov[3][kTY + 2 * kR][kTX + 2 * kR];
    const int s = blockIdx.z;
    const int h = p.hw[s * 8], w = p.hw[s * 8 + 1];
    const int x0 = blockIdx.x * kTX, y0 = blockIdx.y * kTY;
    if (x0 >= w || y0 >= h) return;
    const uint8_t* g = p.base + p.off[s * 4];
    const float scale = 1.f / (4.f * 7.f * 255.f);
    const int tid = threadIdx.y * kTX + threadIdx.x;
    for (int c = tid; c < (kTY + 2 * kR) * (kTX + 2 * kR); c += kTX * kTY) {
        const int cy = c / (kTX + 2 * kR), cx = c - cy * (kTX + 2 * kR);
        const int y = reflect101(y0 + cy - kR, h), x = reflect101(x0 + cx - kR, w);
        const uint8_t* r0 = g + (size_t)reflect101(y - 1, h) * w;
        const uint8_t* r1 = g + (size_t)y * w;
        const uint8_t* r2 = g + (size_t)reflect101(y + 1, h) * w;
        const int xm = reflect101(x - 1, w), xp = reflect101(x + 1, w);
        const int dx = (r0[xp] - r0[xm]) + 2 * (r1[xp] - r1[xm]) + (r2[xp] - r2[xm]);
        const int dy = (r2[xm] + 2 * r2[x] + r2[xp]) - (r0[xm] + 2 * r0[x] + r0[xp]);
        const float fx = (float)dx * scale, fy = (float)dy * scale;
        cov[0][cy][cx] = fx * fx;
        cov[1][cy][cx] = fx * fy;
        cov[2][cy][cx] = fy * fy;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= w || y >= h) return;
    float a = 0.f, b = 0.f, c = 0.f;
    for (int dy = 0; dy < 2 * kR + 1; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2 * kR + 1; ++dx) {
            a += cov[0][threadIdx.y + dy][threadIdx.x + dx];
            b += cov[1][threadIdx.y + dy][threadIdx.x + dx];
            c += cov[2][threadIdx.y + dy][threadIdx.x + dx];
        }
    a *= 0.5f; c *= 0.5f;
    eig[pix_off[s] + (size_t)y * w + x] = (a + c) - sqrtf((a - c) * (a - c) + b * b);
}

// ------------------------------------------------------------------------------------------------------------------
// goodFeaturesToTrack on the response: per-stream max, candidates = 3x3 local maxima of the thresholded response (> 0.01 max)
// off the one-pixel border, ordered by (value desc, linear index desc), greedily accepted at squared distance >= 15^2.
// A candidate is the 64-bit key (value bits << 32 | index): values are positive, so descending keys are that order.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gftt_max_kernel(const float* __restrict__ eig, const long long* __restrict__ pix_off,
                                                       const int* __restrict__ hw, unsigned* __restrict__ mx) {
    const int s = blockIdx.y;
    const int n = hw[s * 8] * hw[s * 8 + 1];
    const float* e = eig + pix_off[s];
    float m = 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = fmaxf(m, e[i]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(mx + s, __float_as_uint(m));   // non-negative floats order as their bits
}

__device__ __forceinline__ float gftt_threshold(unsigned mbits) {
    // cv2: minMaxLoc (double) * qualityLevel, compared by threshold(THRESH_TOZERO) in float
    return (float)((double)__uint_as_float(mbits) * 0.01);
}

__global__ void __launch_bounds__(256) gftt_cand_kernel(const float* __restrict__ eig, const long long* __restrict__ pix_off,
                                                        const int* __restrict__ hw, const unsigned* __restrict__ mx,
                                                        unsigned long long* __restrict__ keys, int* __restrict__ ncand) {
    const int s = blockIdx.y;
    const int h = hw[s * 8], w = hw[s * 8 + 1];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h * w) return;
    const int y = i / w, x = i - y * w;
    if (y < 1 || y >= h - 1 || x < 1 || x >= w - 1) return;
    const float t = gftt_threshold(mx[s]);
    const float* e = eig + pix_off[s];
    const float v = e[i];
    if (!(v > t)) return;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const float u = e[i + dy * w + dx];
            if (u > t && u > v) return;
        }
    const int k = atomicAdd(ncand + s, 1);
    keys[pix_off[s] + k] = ((unsigned long long)__float_as_uint(v) << 32) | (unsigned)i;
}

__device__ void bitonic_desc(unsigned long long* a) {
    for (int k = 2; k <= kSortKeys; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < kSortKeys; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long x = a[i], y = a[l];
                    if (((i & k) == 0) ? (x < y) : (x > y)) { a[i] = y; a[l] = x; }
                }
            }
            __syncthreads();
        }
}

// One CTA per stream.  Pass: the kKeep largest keys below `bound` (merged chunk by chunk through one bitonic sort), then the greedy
// test in sorted order -- every thread tests one key against the corners accepted before the batch, warp 0 resolves the survivors
// in order against those accepted within it.  Passes repeat until 200 corners or the candidates run out.
__global__ void __launch_bounds__(kSelThreads) gftt_select_kernel(const unsigned long long* __restrict__ keys, const long long* __restrict__ pix_off,
                                                                  const int* __restrict__ hw, const int* __restrict__ ncand,
                                                                  float* __restrict__ corners, int* __restrict__ ncorners) {
    extern __shared__ unsigned long long sk[];
    __shared__ int ax[kMaxCorners], ay[kMaxCorners];
    __shared__ unsigned char alive[kSelThreads];
    __shared__ int s_nacc, s_done;
    const int s = blockIdx.x;
    const int w = hw[s * 8 + 1];
    const int n = ncand[s];
    const unsigned long long* k = keys + pix_off[s];
    if (threadIdx.x == 0) { s_nacc = 0; s_done = n == 0; }
    __syncthreads();
    unsigned long long bound = ~0ull;
    while (!s_done) {
        for (int i = threadIdx.x; i < kKeep; i += blockDim.x) sk[i] = 0;
        for (int c0 = 0; c0 < n; c0 += kKeep) {
            for (int i = threadIdx.x; i < kKeep; i += blockDim.x) {
                const unsigned long long v = c0 + i < n ? k[c0 + i] : 0ull;
                sk[kKeep + i] = v < bound ? v : 0ull;
            }
            __syncthreads();
            bitonic_desc(sk);
        }
        for (int b0 = 0; b0 < kKeep && !s_done; b0 += kSelThreads) {
            const int n0 = s_nacc;
            const unsigned long long key = sk[b0 + threadIdx.x];
            bool ok = key != 0ull;
            const int idx = (int)(unsigned)key, y = idx / w, x = idx - y * w;
            for (int j = 0; ok && j < n0; ++j) {
                const int ex = x - ax[j], ey = y - ay[j];
                ok = ex * ex + ey * ey >= kMinDist2;
            }
            alive[threadIdx.x] = ok;
            __syncthreads();
            if (threadIdx.x < 32) {
                const int lane = threadIdx.x;
                int nacc = n0, stop = 0;
                for (int c = 0; c < kSelThreads && !stop; ++c) {
                    const unsigned long long kc = sk[b0 + c];
                    if (kc == 0ull) { stop = 1; break; }
                    if (!alive[c]) continue;
                    const int ic = (int)(unsigned)kc, cy = ic / w, cx = ic - cy * w;
                    bool far = true;
                    for (int j = n0 + lane; j < nacc; j += 32) {
                        const int ex = cx - ax[j], ey = cy - ay[j];
                        far = far && ex * ex + ey * ey >= kMinDist2;
                    }
                    if (__all_sync(0xffffffffu, far)) {
                        if (lane == 0) { ax[nacc] = cx; ay[nacc] = cy; }
                        __syncwarp();
                        if (++nacc == kMaxCorners) stop = 1;
                    }
                }
                if (lane == 0) { s_nacc = nacc; if (stop) s_done = 1; }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0 && !s_done) {
            if (sk[kKeep - 1] == 0ull) s_done = 1;     // every candidate below the old bound has been seen
            else bound = sk[kKeep - 1];
        }
        if (threadIdx.x == 0) sk[kSortKeys - 1] = bound;   // broadcast the new bound through the (unused) tail slot
        __syncthreads();
        bound = sk[kSortKeys - 1];
        __syncthreads();
    }
    const int na = s_nacc;
    for (int j = threadIdx.x; j < na; j += blockDim.x) {
        corners[((size_t)s * kMaxCorners + j) * 2] = (float)ax[j];
        corners[((size_t)s * kMaxCorners + j) * 2 + 1] = (float)ay[j];
    }
    if (threadIdx.x == 0) ncorners[s] = na;
}

// ------------------------------------------------------------------------------------------------------------------
// Pyramidal Lucas-Kanade, cv2's LKTrackerInvoker arithmetic: 14-bit bilinear weights, descaled integer samples of the image (<< 5)
// and of its Scharr derivatives, window sums (exact in int64 here), fp32 solve.  Images are REFLECT_101 beyond their edge and
// the derivatives 0 (buildOpticalFlowPyramid's borders).  One warp per (stream, point); each lane holds 14 of the 441 window pixels.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int px(const uint8_t* img, int h, int w, int y, int x) {
    return img[(size_t)reflect101(y, h) * w + reflect101(x, w)];
}

// calcSharrDeriv: Ix = d/dx of (3 10 3)^T, Iy = d/dy of (3 10 3), REFLECT_101 inside the image; 0 outside it
__device__ __forceinline__ void scharr(const uint8_t* img, int h, int w, int y, int x, int& ix, int& iy) {
    if (y < 0 || y >= h || x < 0 || x >= w) { ix = iy = 0; return; }
    const uint8_t* r0 = img + (size_t)reflect101(y - 1, h) * w;
    const uint8_t* r1 = img + (size_t)y * w;
    const uint8_t* r2 = img + (size_t)reflect101(y + 1, h) * w;
    const int xm = reflect101(x - 1, w), xp = reflect101(x + 1, w);
    const int t0m = (r0[xm] + r2[xm]) * 3 + r1[xm] * 10, t0p = (r0[xp] + r2[xp]) * 3 + r1[xp] * 10;
    const int t1m = r2[xm] - r0[xm], t1 = r2[x] - r0[x], t1p = r2[xp] - r0[xp];
    ix = (int)(short)(t0p - t0m);
    iy = (int)(short)((t1p + t1m) * 3 + t1 * 10);
}

__device__ __forceinline__ int descale(int v, int n) { return (v + (1 << (n - 1))) >> n; }

__device__ __forceinline__ void lk_weights(float a, float b, int& w00, int& w01, int& w10, int& w11) {
    // cvRound((1 - a)(1 - b) 2^14) ... evaluated in fp32 without contraction, rounded half to even
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), __fsub_rn(1.f, b)), 16384.f));
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, __fsub_rn(1.f, b)), 16384.f));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), b), 16384.f));
    w11 = 16384 - w00 - w01 - w10;
}

__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(256) lk_kernel(PyrView prev, PyrView next, const float* __restrict__ pts, const int* __restrict__ npts,
                                                 int P, int S, float* __restrict__ out, uint8_t* __restrict__ status) {
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int s = wid / P, pi = wid - s * P;
    if (s >= S || pi >= npts[s]) return;
    const float ptx = pts[((size_t)s * P + pi) * 2], pty = pts[((size_t)s * P + pi) * 2 + 1];
    const float FLT_SCALE = 1.f / (1 << 20);
    float nx = 0.f, ny = 0.f;
    bool st = true;
    const int maxL = lk_max_level(prev.hw + s * 8);
    for (int L = maxL; L >= 0; --L) {
        const int h = prev.hw[s * 8 + L * 2], w = prev.hw[s * 8 + L * 2 + 1];
        const uint8_t* I = prev.base + prev.off[s * 4 + L];
        const uint8_t* J = next.base + next.off[s * 4 + L];
        const float lsc = (float)(1. / (1 << L));
        float ppx = __fmul_rn(ptx, lsc), ppy = __fmul_rn(pty, lsc);
        if (L == maxL) { nx = ppx; ny = ppy; }
        else { nx = __fmul_rn(nx, 2.f); ny = __fmul_rn(ny, 2.f); }
        ppx = __fsub_rn(ppx, 10.f); ppy = __fsub_rn(ppy, 10.f);
        const int ipx = (int)floorf(ppx), ipy = (int)floorf(ppy);
        if (ipx < -kWin || ipx >= w || ipy < -kWin || ipy >= h) { if (L == 0) st = false; continue; }
        int w00, w01, w10, w11;
        lk_weights(__fsub_rn(ppx, (float)ipx), __fsub_rn(ppy, (float)ipy), w00, w01, w10, w11);
        int Iv[kPerLane], Dx[kPerLane], Dy[kPerLane];
        int a11l = 0, a12l = 0, a22l = 0;     // per lane: 14 products of |Dx|, |Dy| <= 4080 stay below 2^31
#pragma unroll
        for (int m = 0; m < kPerLane; ++m) {
            const int k = lane + 32 * m;
            Iv[m] = Dx[m] = Dy[m] = 0;
            if (k < kWinArea) {
                const int y = ipy + k / kWin, x = ipx + k % kWin;
                Iv[m] = descale(px(I, h, w, y, x) * w00 + px(I, h, w, y, x + 1) * w01 + px(I, h, w, y + 1, x) * w10 +
                                px(I, h, w, y + 1, x + 1) * w11, 9);
                int x00, y00, x01, y01, x10, y10, x11, y11;
                scharr(I, h, w, y, x, x00, y00); scharr(I, h, w, y, x + 1, x01, y01);
                scharr(I, h, w, y + 1, x, x10, y10); scharr(I, h, w, y + 1, x + 1, x11, y11);
                Dx[m] = descale(x00 * w00 + x01 * w01 + x10 * w10 + x11 * w11, 14);
                Dy[m] = descale(y00 * w00 + y01 * w01 + y10 * w10 + y11 * w11, 14);
                a11l += Dx[m] * Dx[m]; a12l += Dx[m] * Dy[m]; a22l += Dy[m] * Dy[m];
            }
        }
        const long long a11 = warp_sum(a11l), a12 = warp_sum(a12l), a22 = warp_sum(a22l);
        const float A11 = __fmul_rn((float)a11, FLT_SCALE), A12 = __fmul_rn((float)a12, FLT_SCALE), A22 = __fmul_rn((float)a22, FLT_SCALE);
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float dd = __fsub_rn(A11, A22);
        const float minEig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), __fsqrt_rn(__fadd_rn(__fmul_rn(dd, dd), __fmul_rn(__fmul_rn(4.f, A12), A12)))),
                                       (float)(2 * kWinArea));
        if (minEig < 1e-4f || D < FLT_EPSILON) { if (L == 0) st = false; continue; }
        D = __fdiv_rn(1.f, D);
        float nwx = __fsub_rn(nx, 10.f), nwy = __fsub_rn(ny, 10.f);
        float pdx = 0.f, pdy = 0.f;
        for (int j = 0; j < 30; ++j) {
            const int inx = (int)floorf(nwx), iny = (int)floorf(nwy);
            if (inx < -kWin || inx >= w || iny < -kWin || iny >= h) { if (L == 0) st = false; break; }
            lk_weights(__fsub_rn(nwx, (float)inx), __fsub_rn(nwy, (float)iny), w00, w01, w10, w11);
            int b1l = 0, b2l = 0;                 // per lane: 14 products of |diff| <= 8160 and |D| <= 4080 stay below 2^31
            if (inx >= 0 && iny >= 0 && inx + kWin < w && iny + kWin < h) {     // the window and its +1 taps inside: no border
                const uint8_t* base = J + (size_t)iny * w + inx;
#pragma unroll
                for (int m = 0; m < kPerLane; ++m) {
                    const int k = lane + 32 * m;
                    if (k < kWinArea) {
                        const uint8_t* q = base + (k / kWin) * w + k % kWin;
                        const int diff = descale(q[0] * w00 + q[1] * w01 + q[w] * w10 + q[w + 1] * w11, 9) - Iv[m];
                        b1l += diff * Dx[m]; b2l += diff * Dy[m];
                    }
                }
            } else {
#pragma unroll
                for (int m = 0; m < kPerLane; ++m) {
                    const int k = lane + 32 * m;
                    if (k < kWinArea) {
                        const int y = iny + k / kWin, x = inx + k % kWin;
                        const int diff = descale(px(J, h, w, y, x) * w00 + px(J, h, w, y, x + 1) * w01 + px(J, h, w, y + 1, x) * w10 +
                                                 px(J, h, w, y + 1, x + 1) * w11, 9) - Iv[m];
                        b1l += diff * Dx[m]; b2l += diff * Dy[m];
                    }
                }
            }
            const long long b1 = warp_sum(b1l), b2 = warp_sum(b2l);
            const float B1 = __fmul_rn((float)b1, FLT_SCALE), B2 = __fmul_rn((float)b2, FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, B2), __fmul_rn(A22, B1)), D);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, B1), __fmul_rn(A11, B2)), D);
            nwx = __fadd_rn(nwx, dx); nwy = __fadd_rn(nwy, dy);
            nx = __fadd_rn(nwx, 10.f); ny = __fadd_rn(nwy, 10.f);
            if (__dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= 0.01 * 0.01) break;
            if (j > 0 && (double)fabsf(__fadd_rn(dx, pdx)) < 0.01 && (double)fabsf(__fadd_rn(dy, pdy)) < 0.01) {
                nx = __fsub_rn(nx, __fmul_rn(dx, 0.5f)); ny = __fsub_rn(ny, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx; pdy = dy;
        }
    }
    if (lane == 0) {
        out[((size_t)s * P + pi) * 2] = nx;
        out[((size_t)s * P + pi) * 2 + 1] = ny;
        status[(size_t)s * P + pi] = st ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Decision: GlobalMotionDetector.detect_motion + MotionCompensatedMultiTracker.update's global-reset rule, per stream.
// ------------------------------------------------------------------------------------------------------------------
struct MState {
    float vec[5][2]; int nvec, vhead;           // motion_vectors (maxlen 5)
    float mag[20]; int nmag, mhead;             // global_motion_history (maxlen 20): 0.0 on frames without a vector
    int det[10]; int ndet, dhead;               // detection_stability_history (maxlen 10)
    int pad;
    double stats[8];                            // total_detections, motion_events, reset_triggers, avg_motion_magnitude,
                                                // global_motion_events, global_resets, individual-resets base, recoveries base
};

__device__ __forceinline__ void rank_sort(const float* v, float* out, int n) {
    // out[rank] = v[t], rank = #smaller + #equal before t (stable)
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        const float x = v[t];
        int r = 0;
        for (int j = 0; j < n; ++j) r += (v[j] < x) || (v[j] == x && j < t);
        out[r] = x;
    }
}

__global__ void __launch_bounds__(256) decide_kernel(MState* __restrict__ state, const float* __restrict__ corners, const int* __restrict__ ncorners,
                                                     const float* __restrict__ nextp, const uint8_t* __restrict__ status, int has_flow,
                                                     const int* __restrict__ det_counts, const long long* __restrict__ tstats,
                                                     int* __restrict__ flags, float* __restrict__ info) {
    __shared__ float fx[kMaxCorners], fy[kMaxCorners], ds[kMaxCorners], sx[kMaxCorners], sy[kMaxCorners], sd[kMaxCorners];
    __shared__ int s_n;
    __shared__ float s_med[2], s_p75;
    const int s = blockIdx.x;
    const int nc = has_flow ? ncorners[s] : 0;
    if (threadIdx.x == 0) {
        int n = 0;
        if (nc >= 20)
            for (int i = 0; i < nc; ++i)
                if (status[(size_t)s * kMaxCorners + i]) {
                    const size_t q = ((size_t)s * kMaxCorners + i) * 2;
                    fx[n] = __fsub_rn(nextp[q], corners[q]); fy[n] = __fsub_rn(nextp[q + 1], corners[q + 1]); ++n;
                }
        s_n = n;
    }
    __syncthreads();
    const int n = s_n;
    bool vec_ok = nc >= 20 && n >= 10 && n > 8;
    if (vec_ok) {
        rank_sort(fx, sx, n); rank_sort(fy, sy, n);
        __syncthreads();
        if (threadIdx.x == 0) {   // np.median: the middle value, or the float32 mean of the two middle values
            s_med[0] = n & 1 ? sx[n / 2] : __fdiv_rn(__fadd_rn(sx[n / 2 - 1], sx[n / 2]), 2.f);
            s_med[1] = n & 1 ? sy[n / 2] : __fdiv_rn(__fadd_rn(sy[n / 2 - 1], sy[n / 2]), 2.f);
        }
        __syncthreads();
        for (int t = threadIdx.x; t < n; t += blockDim.x) {
            const float ex = __fsub_rn(fx[t], s_med[0]), ey = __fsub_rn(fy[t], s_med[1]);
            ds[t] = __fsqrt_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
        }
        __syncthreads();
        rank_sort(ds, sd, n);
        __syncthreads();
        if (threadIdx.x == 0) {   // np.percentile(..., 75), linear: the fraction is a multiple of 1/4, exact in fp32
            const double vi = 0.75 * (n - 1);
            const int lo = (int)floor(vi), hi = min(lo + 1, n - 1);
            const float t = (float)(vi - lo), a = sd[lo], b = sd[hi], df = __fsub_rn(b, a);
            s_p75 = t >= 0.5f ? __fsub_rn(b, __fmul_rn(df, __fsub_rn(1.f, t))) : __fadd_rn(a, __fmul_rn(df, t));
        }
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    MState& m = state[s];
    float vx = 0.f, vy = 0.f, mag = 0.f;
    bool is_motion = false, should_reset = false;
    if (vec_ok) {
        int k = 0; float sxx = 0.f, syy = 0.f;
        for (int i = 0; i < n; ++i)
            if (ds[i] < s_p75) { sxx = __fadd_rn(sxx, fx[i]); syy = __fadd_rn(syy, fy[i]); ++k; }
        vec_ok = k > 5;
        if (vec_ok) {
            vx = __fdiv_rn(sxx, (float)k); vy = __fdiv_rn(syy, (float)k);
            mag = __fsqrt_rn(__fadd_rn(__fmul_rn(vx, vx), __fmul_rn(vy, vy)));
            m.vec[m.vhead][0] = vx; m.vec[m.vhead][1] = vy;
            m.vhead = (m.vhead + 1) % 5; m.nvec = min(m.nvec + 1, 5);
            is_motion = mag > 30.f;
            should_reset = mag > 50.f;
            if (m.nvec >= 3 && is_motion) {   // consistency of the last three vectors (:262-280)
                float ang[3];
                for (int j = 0; j < 3; ++j) {
                    const int q = (m.vhead - 3 + j + 5) % 5;
                    ang[j] = (float)atan2((double)m.vec[q][1], (double)m.vec[q][0]);
                }
                float d[2];
                for (int j = 0; j < 2; ++j) {
                    float x = fabsf(__fsub_rn(ang[j + 1], ang[j]));
                    if ((double)x > 3.141592653589793) x = (float)(2 * 3.141592653589793 - (double)x);
                    d[j] = x;
                }
                const float cons = fmaxf(0.f, (float)(1.0 - (double)__fdiv_rn(__fadd_rn(d[0], d[1]), 2.f) / 3.141592653589793));
                if (cons > 0.7f) should_reset = should_reset || mag > 45.f;
            }
        }
        if (!vec_ok) { vx = vy = mag = 0.f; }
    }
    if (has_flow) {
        double* st = m.stats;
        st[0] += 1.0; st[1] += is_motion; st[2] += should_reset;
        st[3] = (st[3] * (st[0] - 1.0) + (double)mag) / st[0];
    }
    m.mag[m.mhead] = mag; m.mhead = (m.mhead + 1) % 20; m.nmag = min(m.nmag + 1, 20);
    m.det[m.dhead] = det_counts ? det_counts[s] : 0; m.dhead = (m.dhead + 1) % 10; m.ndet = min(m.ndet + 1, 10);
    bool reset = false;
    if (should_reset) {
        m.stats[4] += 1.0;
        if (m.ndet >= 5) {    // np.std(recent) / (np.mean(recent) + 1) > 0.5 over the last five detection counts
            double sum = 0.0, var = 0.0;
            for (int j = 0; j < 5; ++j) sum += m.det[(m.dhead - 5 + j + 10) % 10];
            const double mean = sum / 5.0;
            for (int j = 0; j < 5; ++j) { const double e = m.det[(m.dhead - 5 + j + 10) % 10] - mean; var += e * e; }
            reset = sqrt(var / 5.0) / (mean + 1.0) > 0.5;
        }
        if (!reset && m.nmag >= 3) {
            double sum = 0.0;
            for (int j = 0; j < 3; ++j) sum += (double)m.mag[(m.mhead - 3 + j + 20) % 20];
            reset = sum / 3.0 > 30.0;
        }
        reset = reset || (double)mag > 60.0;
    }
    if (reset) {
        m.stats[5] += 1.0;
        if (tstats) { m.stats[6] += (double)tstats[(size_t)s * 8 + 6]; m.stats[7] += (double)tstats[(size_t)s * 8 + 7]; }
    }
    flags[s] = reset;
    float* o = info + (size_t)s * 8;
    o[0] = mag; o[1] = vx; o[2] = vy; o[3] = is_motion; o[4] = should_reset; o[5] = reset; o[6] = (float)nc; o[7] = (float)n;
}

__global__ void stats_kernel(const MState* __restrict__ state, int S, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S * 8) out[i] = state[i / 8].stats[i % 8];
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
// every stream stores four levels; the LK kernel starts at the deepest one cv2 would build (lk_max_level)
void level_dims(int h, int w, int* hw) {
    for (int l = 0; l < kLevels; ++l) {
        hw[2 * l] = h; hw[2 * l + 1] = w;
        h = (h + 1) / 2; w = (w + 1) / 2;
    }
}

struct Geometry { int S, max_h, max_w; long long* off_d; int* hw_d; long long* pix_d; long long bytes, pixels; };

int launch_pyramid(const uint8_t* frames, const long long* foff, PyrView p, int S, int max_h, int max_w, cudaStream_t st) {
    gray_kernel<<<dim3(b2_ceil_div(max_h * max_w, 256), S), 256, 0, st>>>(frames, foff, p);
    int h = max_h, w = max_w;
    for (int l = 0; l < kLevels - 1; ++l) {
        h = (h + 1) / 2; w = (w + 1) / 2;
        pyrdown_kernel<<<dim3(b2_ceil_div(h * w, 256), S), 256, 0, st>>>(p, l);
    }
    B2_CUDA(cudaGetLastError());
    b2_count_launch(kLevels);
    return B2_OK;
}

int launch_eig(PyrView p, const long long* pix_off, int S, int max_h, int max_w, float* eig, cudaStream_t st) {
    eig_kernel<<<dim3(b2_ceil_div(max_w, kTX), b2_ceil_div(max_h, kTY), S), dim3(kTX, kTY), 0, st>>>(p, pix_off, eig);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

int launch_select(const float* eig, const long long* pix_off, const int* hw, int S, int max_h, int max_w, void* ws,
                  float* corners, int* ncorners, cudaStream_t st) {
    unsigned* mx = (unsigned*)ws;
    int* ncand = (int*)ws + S;
    unsigned long long* keys = (unsigned long long*)((char*)ws + (((size_t)S * 8 + 255) & ~(size_t)255));
    const int smem = kSortKeys * 8;
    B2_CUDA(cudaFuncSetAttribute(gftt_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));   // per device: every launch
    B2_CUDA(cudaMemsetAsync(ws, 0, (size_t)S * 8, st));
    const int np = max_h * max_w;
    gftt_max_kernel<<<dim3(std::min(b2_ceil_div(np, 256), 64), S), 256, 0, st>>>(eig, pix_off, hw, mx);
    gftt_cand_kernel<<<dim3(b2_ceil_div(np, 256), S), 256, 0, st>>>(eig, pix_off, hw, mx, keys, ncand);
    gftt_select_kernel<<<S, kSelThreads, smem, st>>>(keys, pix_off, hw, ncand, corners, ncorners);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(3);
    return B2_OK;
}

size_t select_ws_bytes(int S, long long pixels) { return (((size_t)S * 8 + 255) & ~(size_t)255) + (size_t)pixels * 8; }

int launch_lk(PyrView prev, PyrView next, const float* pts, const int* npts, int P, int S, float* out, uint8_t* status, cudaStream_t st) {
    const long long warps = (long long)S * P;
    lk_kernel<<<(unsigned)b2_ceil_div((int)warps, 8), 256, 0, st>>>(prev, next, pts, npts, P, S, out, status);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

}  // namespace

extern "C" int b2_pyramid_layout(int n_streams, const int* shapes_host, long long* level_off_host, int* level_hw_host,
                                 long long* pix_off_host, long long* totals_host) {
    B2_REQUIRE(n_streams >= 1 && shapes_host && level_off_host && level_hw_host && pix_off_host && totals_host, "pyramid_layout: bad argument");
    long long bytes = 0, pixels = 0;
    for (int s = 0; s < n_streams; ++s) {
        const int h = shapes_host[2 * s], w = shapes_host[2 * s + 1];
        B2_REQUIRE(h >= 1 && w >= 1 && (long long)h * w < (1ll << 30), "pyramid_layout: stream %d has shape %dx%d", s, h, w);
        level_dims(h, w, level_hw_host + 8 * s);
        pix_off_host[s] = pixels;
        pixels += (long long)h * w;
        for (int l = 0; l < kLevels; ++l) {
            level_off_host[4 * s + l] = bytes;
            bytes += ((long long)level_hw_host[8 * s + 2 * l] * level_hw_host[8 * s + 2 * l + 1] + 15) & ~15ll;
        }
    }
    totals_host[0] = bytes; totals_host[1] = pixels;
    return B2_OK;
}

extern "C" size_t b2_good_features_workspace_bytes(int n_streams, long long total_pixels) { return select_ws_bytes(n_streams, total_pixels); }

extern "C" int b2_gray_pyramid_u8(const uint8_t* frames, const long long* frame_off_dev, int n_streams, int max_h, int max_w,
                                  uint8_t* pyr, const long long* level_off_dev, const int* level_hw_dev, void* stream) {
    B2_REQUIRE(frames && frame_off_dev && pyr && level_off_dev && level_hw_dev && n_streams >= 1 && max_h >= 1 && max_w >= 1,
               "gray_pyramid_u8: bad argument");
    return launch_pyramid(frames, frame_off_dev, PyrView{pyr, level_off_dev, level_hw_dev}, n_streams, max_h, max_w, (cudaStream_t)stream);
}

extern "C" int b2_corner_min_eig(const uint8_t* pyr, const long long* level_off_dev, const int* level_hw_dev, const long long* pix_off_dev,
                                 int n_streams, int max_h, int max_w, int block_size, int ksize, float* eig_out, void* stream) {
    B2_REQUIRE(pyr && level_off_dev && level_hw_dev && pix_off_dev && eig_out && n_streams >= 1, "corner_min_eig: bad argument");
    if (block_size != 7 || ksize != 3) { b2_set_error("corner_min_eig: only blockSize=7, ksize=3"); return B2_ERR_UNSUPPORTED; }
    return launch_eig(PyrView{(uint8_t*)pyr, level_off_dev, level_hw_dev}, pix_off_dev, n_streams, max_h, max_w, eig_out, (cudaStream_t)stream);
}

extern "C" int b2_good_features(const float* eig, const long long* pix_off_dev, const int* level_hw_dev, int n_streams, int max_h, int max_w,
                                long long total_pixels, int max_corners, double quality_level, double min_distance, void* workspace, size_t workspace_bytes,
                                float* corners_out, int* counts_out, void* stream) {
    B2_REQUIRE(eig && pix_off_dev && level_hw_dev && workspace && corners_out && counts_out && n_streams >= 1, "good_features: bad argument");
    if (max_corners != kMaxCorners || quality_level != 0.01 || min_distance != 15.0) {
        b2_set_error("good_features: only maxCorners=200, qualityLevel=0.01, minDistance=15");
        return B2_ERR_UNSUPPORTED;
    }
    B2_REQUIRE(workspace_bytes >= select_ws_bytes(n_streams, total_pixels), "good_features: workspace of %zu bytes, need %zu", workspace_bytes,
               select_ws_bytes(n_streams, total_pixels));
    return launch_select(eig, pix_off_dev, level_hw_dev, n_streams, max_h, max_w, workspace, corners_out, counts_out, (cudaStream_t)stream);
}

extern "C" int b2_lk_pyr(const uint8_t* prev_pyr, const uint8_t* next_pyr, const long long* level_off_dev, const int* level_hw_dev,
                         int n_streams, const float* pts, const int* counts, int max_pts, int win, int max_level, int max_count,
                         double epsilon, float* next_out, uint8_t* status_out, void* stream) {
    B2_REQUIRE(prev_pyr && next_pyr && level_off_dev && level_hw_dev && pts && counts && next_out && status_out && n_streams >= 1 && max_pts >= 1,
               "lk_pyr: bad argument");
    if (win != kWin || max_level != kLevels - 1 || max_count != 30 || epsilon != 0.01) {
        b2_set_error("lk_pyr: only winSize=21x21, maxLevel=3, criteria COUNT|EPS 30 / 0.01");
        return B2_ERR_UNSUPPORTED;
    }
    B2_REQUIRE((long long)n_streams * max_pts * 32 < (1ll << 31), "lk_pyr: too many points");
    return launch_lk(PyrView{(uint8_t*)prev_pyr, level_off_dev, level_hw_dev}, PyrView{(uint8_t*)next_pyr, level_off_dev, level_hw_dev},
                     pts, counts, max_pts, n_streams, next_out, status_out, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------------------------
// the per-stream motion bank
// ------------------------------------------------------------------------------------------------------------------
struct b2_motion {
    int S, max_h, max_w;
    long long frames;      // frames given to b2_motion_flow since create / reset
    int cur;               // pyramid buffer holding the newest frame
    void* arena;
    uint8_t* pyr[2];
    long long* off_d; int* hw_d; long long* pix_d;
    float* eig; void* ws; size_t ws_bytes;
    float* corners; int* ncorners; float* nextp; uint8_t* status;
    MState* state;
    size_t state_bytes;
};

extern "C" int b2_motion_create(int n_streams, const int* shapes_host, b2_motion_t** out) {
    B2_REQUIRE(out && shapes_host && n_streams >= 1, "motion_create: bad argument");
    const int S = n_streams;
    long long* off = new (std::nothrow) long long[4 * S + S];
    int* hw = new (std::nothrow) int[8 * S];
    if (!off || !hw) { delete[] off; delete[] hw; b2_set_error("out of host memory"); return B2_ERR_STATE; }
    long long tot[2];
    int rc = b2_pyramid_layout(S, shapes_host, off, hw, off + 4 * S, tot);
    if (rc != B2_OK) { delete[] off; delete[] hw; return rc; }
    b2_motion* m = new (std::nothrow) b2_motion();
    if (!m) { delete[] off; delete[] hw; b2_set_error("out of host memory"); return B2_ERR_STATE; }
    m->S = S; m->max_h = 0; m->max_w = 0;
    for (int s = 0; s < S; ++s) { m->max_h = std::max(m->max_h, shapes_host[2 * s]); m->max_w = std::max(m->max_w, shapes_host[2 * s + 1]); }
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    m->ws_bytes = select_ws_bytes(S, tot[1]);
    m->state_bytes = (size_t)S * sizeof(MState);
    const size_t sz_pyr = up((size_t)tot[0]), sz_tab = up((size_t)S * 5 * 8) + up((size_t)S * 8 * 4), sz_eig = up((size_t)tot[1] * 4);
    const size_t sz_pts = up((size_t)S * kMaxCorners * 8), sz_cnt = up((size_t)S * 4), sz_st = up((size_t)S * kMaxCorners);
    const size_t total = 2 * sz_pyr + sz_tab + sz_eig + up(m->ws_bytes) + 2 * sz_pts + sz_cnt + sz_st + up(m->state_bytes);
    cudaError_t e = cudaMalloc(&m->arena, total);
    if (e != cudaSuccess) {
        delete[] off; delete[] hw; delete m;
        b2_set_error("motion_create: cudaMalloc(%zu) failed: %s", total, cudaGetErrorString(e));
        return B2_ERR_CUDA;
    }
    char* a = (char*)m->arena;
    m->pyr[0] = (uint8_t*)a; a += sz_pyr;
    m->pyr[1] = (uint8_t*)a; a += sz_pyr;
    m->off_d = (long long*)a; m->pix_d = m->off_d + 4 * S; a += up((size_t)S * 5 * 8);
    m->hw_d = (int*)a; a += up((size_t)S * 8 * 4);
    m->eig = (float*)a; a += sz_eig;
    m->ws = a; a += up(m->ws_bytes);
    m->corners = (float*)a; a += sz_pts;
    m->nextp = (float*)a; a += sz_pts;
    m->ncorners = (int*)a; a += sz_cnt;
    m->status = (uint8_t*)a; a += sz_st;
    m->state = (MState*)a;
    e = cudaMemcpy(m->off_d, off, (size_t)S * 5 * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(m->hw_d, hw, (size_t)S * 8 * 4, cudaMemcpyHostToDevice);
    delete[] off; delete[] hw;
    if (e != cudaSuccess) { cudaFree(m->arena); delete m; b2_set_error("motion_create: %s", cudaGetErrorString(e)); return B2_ERR_CUDA; }
    *out = m;
    return b2_motion_reset(m, nullptr);
}

extern "C" int b2_motion_destroy(b2_motion_t* m) {
    if (!m) return B2_OK;
    cudaFree(m->arena);
    delete m;
    return B2_OK;
}

extern "C" int b2_motion_reset(b2_motion_t* m, void* stream) {
    B2_REQUIRE(m, "motion_reset: null handle");
    B2_CUDA(cudaMemsetAsync(m->state, 0, m->state_bytes, (cudaStream_t)stream));
    m->frames = 0; m->cur = 0;
    return B2_OK;
}

extern "C" int b2_motion_flow(b2_motion_t* m, const uint8_t* frames, const long long* frame_off_dev, void* stream) {
    B2_REQUIRE(m && frames && frame_off_dev, "motion_flow: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int nxt = m->frames ? m->cur ^ 1 : m->cur;
    PyrView pn{m->pyr[nxt], m->off_d, m->hw_d};
    int rc = launch_pyramid(frames, frame_off_dev, pn, m->S, m->max_h, m->max_w, st);
    if (rc != B2_OK) return rc;
    if (m->frames) {
        PyrView pp{m->pyr[m->cur], m->off_d, m->hw_d};
        if ((rc = launch_eig(pp, m->pix_d, m->S, m->max_h, m->max_w, m->eig, st)) != B2_OK) return rc;
        if ((rc = launch_select(m->eig, m->pix_d, m->hw_d, m->S, m->max_h, m->max_w, m->ws, m->corners, m->ncorners, st)) != B2_OK) return rc;
        if ((rc = launch_lk(pp, pn, m->corners, m->ncorners, kMaxCorners, m->S, m->nextp, m->status, st)) != B2_OK) return rc;
    }
    m->cur = nxt;
    m->frames += 1;
    return B2_OK;
}

extern "C" int b2_motion_decide(b2_motion_t* m, const int32_t* det_counts_dev, const long long* tracker_stats_dev, int32_t* flags_dev,
                                float* info_dev, void* stream) {
    B2_REQUIRE(m && flags_dev && info_dev, "motion_decide: bad argument");
    B2_REQUIRE(m->frames > 0, "motion_decide: call b2_motion_flow for the frame first");
    decide_kernel<<<m->S, 256, 0, (cudaStream_t)stream>>>(m->state, m->corners, m->ncorners, m->nextp, m->status, m->frames > 1 ? 1 : 0,
                                                          det_counts_dev, tracker_stats_dev, flags_dev, info_dev);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_motion_stats(b2_motion_t* m, double* stats_dev_out, void* stream) {
    B2_REQUIRE(m && stats_dev_out, "motion_stats: bad argument");
    stats_kernel<<<b2_ceil_div(m->S * 8, 256), 256, 0, (cudaStream_t)stream>>>(m->state, m->S, stats_dev_out);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}
