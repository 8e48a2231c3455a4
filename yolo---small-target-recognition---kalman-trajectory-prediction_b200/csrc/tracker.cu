// Structure-of-arrays Kalman track bank for sm_100a: one independent multi-target tracker per video stream.
//
// Replaces kalman/enhanced_multi_target_tracker.py:42-132 (EnhancedMultiTargetTracker.update) and
// kalman/enhanced_aircraft_kalman_tracker.py (AircraftKalmanTracker: predict :184-203, update :249-297,
// analyze_motion_pattern :137-182, mark_as_lost :299-317, enhanced_long_term_predict :205-247,
// get_track_info :335-383, should_delete :385-405).
//
// Layout: field-major SoA over S*C slots (slot g = stream*C + i), fp32 state.  With the reference's
// F, H, Q, R, P0 the 8x8 covariance keeps the pattern P[i,j] != 0 <=> i == j (mod 4); x/y share one
// (pos,vel) covariance triple and w/h another, so the bank stores 8 state floats + 2x3 covariance floats
// per track and evaluates the exact closed-form 2x2 recurrences (SURVEY.md 8a, verified in
// tests/test_oracle_vs_golden.py::test_tracker_known_answer).
//
// Per frame, TWO launches:
//   (1) sweep_kernel   -- grid-wide, one slot per thread, a block = one 256-slot chunk of one stream (HBM-bound).
//         Every live track is predicted in registers and its predicted box tested against the stream's detections
//         (staged in shared memory).  A track that NO detection overlaps with IoU >= thr cannot be matched whatever the
//         greedy order is, so its frame is finished on the spot: mark lost, delete test, the reference's extra predict on
//         the first lost frame, and the emitted row -- every field of the slot is read once and written once.  Tracks that
//         do have a candidate pair are written back predicted and listed (slot, box, id) together with their pairs
//         (IoU, detection, track).  Row / list positions come from a block scan plus the aggregates of the stream's
//         preceding chunks (published per chunk, no atomics on the data path): the output is deterministic.
//   (2) resolve_kernel -- one CTA per stream, works on the short lists only: greedy matching == repeated mutual-best rounds
//         (exactly the pairs the reference's descending-IoU walk takes, ties -> lowest (det, track id)), Kalman update +
//         motion analysis of the matched tracks, lost / delete for the rest, new tracks for unmatched detections
//         (ascending detection index -> ascending ids, k-th new track takes the k-th free slot), rows, stats.
// Row order per stream: untouched tracks in slot order, then candidate tracks in slot order, then new tracks in slot
// order.  List order of the reference (= ascending track id) is carried by the id column; slots are recycled.
#include "common.cuh"

#include <algorithm>
#include <new>

void b2_count_launch(int n);

namespace {

enum FField { X0 = 0, X1, X2, X3, X4, X5, X6, X7, PPX, PPV, PVV, PSX, PSV, PSVV, VAVGX, VAVGY, DIRN, SPEED, STAB, PCONF, NFF };
enum IField { ID = 0, AGE, HITS, STREAK, TSU, LOSTF, ISLOST, NVEL, VHEAD, TLEN, THEAD, NIF };
// mode 1 (camera_motion_compensation/motion_reset_kalman_tracker.py:16-355): per-slot reset state
//   position_history deque(maxlen=8) (:41), last bbox of bbox_history + its length (:43, only [-1] and len >= 2 are read),
//   motion_scores deque(maxlen=10) (:55), motion_consistency, reset_count, last_reset_frame (:52-53)
#ifndef B2_SWEEP_BLOCKS
#define B2_SWEEP_BLOCKS 4      // resident sweep blocks per SM the register budget is set for (experiment builds: 5, 6)
#endif
constexpr int kPosRing = 8, kScoreRing = 10;
enum MRF { MR_PH = 0, MR_BB = MR_PH + 2 * kPosRing, MR_MS = MR_BB + 4, MR_MCONS = MR_MS + kScoreRing, MR_NF };
enum MRI { MR_PHLEN = 0, MR_PHHEAD, MR_BBLEN, MR_MSLEN, MR_MSHEAD, MR_RESETS, MR_LASTRESET, MR_NI };
constexpr float kJumpThr = 40.f, kVelThr = 60.f, kSizeThr = 0.3f;      // :46-48
constexpr int kResetCooldown = 15;                                     // :49
constexpr int kVelRing = 50;       // deque(maxlen=50)  enhanced_aircraft_kalman_tracker.py:79
constexpr int kTraj = B2_TRAJ_LEN; // only the last 30 trajectory points are ever read (:377)
#ifndef B2_SWEEP_CHUNK
#define B2_SWEEP_CHUNK 256
#endif
constexpr int kChunk = B2_SWEEP_CHUNK;        // slots per sweep block (experiment builds: 128 with B2_SWEEP_BLOCKS=8)
constexpr int kMaxDetsSmem = 1024;
constexpr int kResolveThreads = 512;
constexpr int kCtSmem = 1024;      // candidate tracks whose match keys live in shared memory (more -> dense fallback)

// noise constants, enhanced_aircraft_kalman_tracker.py:44-71
constexpr float P0_POS = 50.f, P0_VEL = 100.f, P0_SVEL = 1.f;
constexpr float Q_POS = 0.1f, Q_SIZE = 0.01f, Q_VEL = 0.1f, Q_SVEL = 0.001f, R_MEAS = 10.f;

struct Bank {
    float* f;       // [NFF][N]
    int32_t* i;     // [NIF][N]
    float* vel;     // [kVelRing*2][N]
    float* traj;    // [kTraj*2][N]
    float* mrf;     // mode 1: [MR_NF][N]
    int32_t* mri;   // mode 1: [MR_NI][N]
    // ---- per-frame scratch ----
    unsigned long long* agg;   // [S][nchunks] chunk aggregates of the sweep: bit 63 valid | pairs << 32 | cand << 16 | emitted
    int32_t* chunk_free;       // [S][nchunks] free slots per chunk after the sweep
    int32_t* fcnt;             // [S][4] sweep counters: terminated, long-term rows, live after
    unsigned int* ticket;      // [1] dynamic block id of the sweep (chunk order == scheduling order)
    int32_t* ctrk_slot;        // [S][C] candidate tracks (slot order): slot
    float4* cbox;              // [S][C]   predicted box
    int32_t* cid;              // [S][C]   track id
    int32_t* cmatch;           // [S][C]   matched detection (dense fallback / > kCtSmem candidates)
    uint4* pairs;              // [S][pair_cap] {iou bits, det, candidate index, track id}
    int32_t* next_id;          // [S]
    int32_t* frame_count;      // [S]
    long long* stats;          // [S][8]: created, terminated, active, long_term, recoveries, dropped (no free slot),
                               //         mode 1: individual_resets, tracking_recoveries (motion_compensated_multi_tracker.py:58-66)
    int S, C, N, max_dets, nchunks, pair_cap;
    int mode;                  // 0: EnhancedMultiTargetTracker; 1: MotionCompensatedMultiTracker (update without a frame)
    int max_lost, min_hits; float iou_thr;
};

struct Frame {
    const float* dets; int det_cols; const int32_t* det_counts;
    float* out_rows; int32_t* out_counts; float* out_traj; int32_t* out_traj_len;
    int out_cap;   // rows per stream the output buffers hold (<= capacity); rows beyond are counted, not written
    float* out_extra;          // mode 1 (may be NULL): [S][out_cap][4] {reset_count (i32), frames_since_reset (i32), motion_consistency, 0}
};

struct b2_tracker_impl {
    Bank b;
    void* arena;
    size_t arena_bytes;
};

__device__ __forceinline__ float& FF(const Bank& b, int field, int g) { return b.f[(size_t)field * b.N + g]; }
__device__ __forceinline__ int32_t& II(const Bank& b, int field, int g) { return b.i[(size_t)field * b.N + g]; }
__device__ __forceinline__ float& RF(const Bank& b, int field, int g) { return b.mrf[(size_t)field * b.N + g]; }
__device__ __forceinline__ int32_t& RI(const Bank& b, int field, int g) { return b.mri[(size_t)field * b.N + g]; }

// MotionResetKalmanTracker.predict (:300-321): for 10 frames after a reset the box handed to the association is centred between
// the last stored position and the Kalman prediction; the state is not touched.  age: after the predict's increment.
__device__ __forceinline__ float4 blended_box(const Bank& b, int g, int age, float cx, float cy, float w, float h) {
    const int since = age - RI(b, MR_LASTRESET, g), n = RI(b, MR_PHLEN, g);
    if (since < 10 && n > 0) {
        int last = RI(b, MR_PHHEAD, g) - 1; if (last < 0) last += kPosRing;
        const float blend = fminf((float)since / 10.f, 1.f);
        cx = (1.f - blend) * RF(b, MR_PH + 2 * last, g) + blend * cx;
        cy = (1.f - blend) * RF(b, MR_PH + 2 * last + 1, g) + blend * cy;
    }
    return make_float4(cx - w / 2.f, cy - h / 2.f, cx + w / 2.f, cy + h / 2.f);
}

__device__ __forceinline__ void push_traj(const Bank& b, int g, float cx, float cy) {
    int head = II(b, THEAD, g), len = II(b, TLEN, g);
    b.traj[(size_t)(2 * head) * b.N + g] = cx;
    b.traj[(size_t)(2 * head + 1) * b.N + g] = cy;
    head = head + 1 == kTraj ? 0 : head + 1;
    II(b, THEAD, g) = head;
    II(b, TLEN, g) = min(len + 1, kTraj);
}

// x <- F x, P <- F P F^T + Q, age++, tsu++, trajectory push  (:184-203)
__device__ __forceinline__ void predict_slot(const Bank& b, int g) {
    const float cx = FF(b, X0, g) + FF(b, X4, g), cy = FF(b, X1, g) + FF(b, X5, g);
    FF(b, X0, g) = cx; FF(b, X1, g) = cy;
    FF(b, X2, g) += FF(b, X6, g); FF(b, X3, g) += FF(b, X7, g);
    {
        const float pxx = FF(b, PPX, g), pxv = FF(b, PPV, g), pvv = FF(b, PVV, g);
        FF(b, PPX, g) = pxx + 2.f * pxv + pvv + Q_POS; FF(b, PPV, g) = pxv + pvv; FF(b, PVV, g) = pvv + Q_VEL;
    }
    {
        const float pxx = FF(b, PSX, g), pxv = FF(b, PSV, g), pvv = FF(b, PSVV, g);
        FF(b, PSX, g) = pxx + 2.f * pxv + pvv + Q_SIZE; FF(b, PSV, g) = pxv + pvv; FF(b, PSVV, g) = pvv + Q_SVEL;
    }
    II(b, AGE, g) += 1; II(b, TSU, g) += 1;
    push_traj(b, g, cx, cy);
}

// Bank-only predict (b2_tracker_bank_predict): four consecutive slots per thread with 16-byte accesses (N % 4 == 0), the same
// arithmetic as predict_slot element-wise; dead slots (id == 0) are written back unchanged.
__global__ void __launch_bounds__(256) bank_predict_kernel(const Bank b) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= b.N || II(b, ID, g) == 0) return;
    predict_slot(b, g);
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float sel(bool c, float a, float b) { return c ? a : b; }

__global__ void __launch_bounds__(256) bank_predict4_kernel(const Bank b) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (g >= b.N) return;
    const size_t N = b.N;
    const int4 id = *reinterpret_cast<const int4*>(b.i + (size_t)ID * N + g);
    const bool l0 = id.x != 0, l1 = id.y != 0, l2 = id.z != 0, l3 = id.w != 0;
    if (!(l0 || l1 || l2 || l3)) return;
    float* F = b.f + g;
    float4 x0 = ld4(F + X0 * N), x1 = ld4(F + X1 * N), x2 = ld4(F + X2 * N), x3 = ld4(F + X3 * N);
    const float4 v0 = ld4(F + X4 * N), v1 = ld4(F + X5 * N), v2 = ld4(F + X6 * N), v3 = ld4(F + X7 * N);
#define B2_ADD4(a, v) a.x = sel(l0, a.x + v.x, a.x); a.y = sel(l1, a.y + v.y, a.y); a.z = sel(l2, a.z + v.z, a.z); a.w = sel(l3, a.w + v.w, a.w);
    B2_ADD4(x0, v0) B2_ADD4(x1, v1) B2_ADD4(x2, v2) B2_ADD4(x3, v3)
#undef B2_ADD4
    st4(F + X0 * N, x0); st4(F + X1 * N, x1); st4(F + X2 * N, x2); st4(F + X3 * N, x3);
#define B2_COV4(PX, PV, VV, QP, QV)                                                                                      \
    {                                                                                                                    \
        float4 pxx = ld4(F + PX * N), pxv = ld4(F + PV * N), pvv = ld4(F + VV * N);                                       \
        pxx.x = sel(l0, pxx.x + 2.f * pxv.x + pvv.x + QP, pxx.x); pxv.x = sel(l0, pxv.x + pvv.x, pxv.x); pvv.x = sel(l0, pvv.x + QV, pvv.x); \
        pxx.y = sel(l1, pxx.y + 2.f * pxv.y + pvv.y + QP, pxx.y); pxv.y = sel(l1, pxv.y + pvv.y, pxv.y); pvv.y = sel(l1, pvv.y + QV, pvv.y); \
        pxx.z = sel(l2, pxx.z + 2.f * pxv.z + pvv.z + QP, pxx.z); pxv.z = sel(l2, pxv.z + pvv.z, pxv.z); pvv.z = sel(l2, pvv.z + QV, pvv.z); \
        pxx.w = sel(l3, pxx.w + 2.f * pxv.w + pvv.w + QP, pxx.w); pxv.w = sel(l3, pxv.w + pvv.w, pxv.w); pvv.w = sel(l3, pvv.w + QV, pvv.w); \
        st4(F + PX * N, pxx); st4(F + PV * N, pxv); st4(F + VV * N, pvv);                                                 \
    }
    B2_COV4(PPX, PPV, PVV, Q_POS, Q_VEL)
    B2_COV4(PSX, PSV, PSVV, Q_SIZE, Q_SVEL)
#undef B2_COV4
    int32_t* I = b.i + g;
    int4 age = *reinterpret_cast<const int4*>(I + (size_t)AGE * N), tsu = *reinterpret_cast<const int4*>(I + (size_t)TSU * N);
    age.x += l0; age.y += l1; age.z += l2; age.w += l3;
    tsu.x += l0; tsu.y += l1; tsu.z += l2; tsu.w += l3;
    *reinterpret_cast<int4*>(I + (size_t)AGE * N) = age; *reinterpret_cast<int4*>(I + (size_t)TSU * N) = tsu;
    int4 head = *reinterpret_cast<const int4*>(I + (size_t)THEAD * N), len = *reinterpret_cast<const int4*>(I + (size_t)TLEN * N);
    const float cx[4] = {x0.x, x0.y, x0.z, x0.w}, cy[4] = {x1.x, x1.y, x1.z, x1.w};
    const bool live[4] = {l0, l1, l2, l3};
    int hd[4] = {head.x, head.y, head.z, head.w}, ln[4] = {len.x, len.y, len.z, len.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (live[k]) {
            b.traj[(size_t)(2 * hd[k]) * N + g + k] = cx[k];                       // push_traj
            b.traj[(size_t)(2 * hd[k] + 1) * N + g + k] = cy[k];
            hd[k] = hd[k] + 1 == kTraj ? 0 : hd[k] + 1;
            ln[k] = min(ln[k] + 1, kTraj);
        }
    }
    *reinterpret_cast<int4*>(I + (size_t)THEAD * N) = make_int4(hd[0], hd[1], hd[2], hd[3]);
    *reinterpret_cast<int4*>(I + (size_t)TLEN * N) = make_int4(ln[0], ln[1], ln[2], ln[3]);
}

// _calculate_iou (enhanced_multi_target_tracker.py:200-232)
__device__ __forceinline__ float iou_ref(const float4& d, const float4& t) {
    const float x1 = fmaxf(d.x, t.x), y1 = fmaxf(d.y, t.y), x2 = fminf(d.z, t.z), y2 = fminf(d.w, t.w);
    if (x2 <= x1 || y2 <= y1) return 0.f;
    const float inter = (x2 - x1) * (y2 - y1);
    const float a1 = (d.z - d.x) * (d.w - d.y), a2 = (t.z - t.x) * (t.w - t.y);
    const float uni = a1 + a2 - inter;
    return uni <= 0.f ? 0.f : inter / uni;
}

// exclusive scan over the block of a 64-bit (packed) value; *total = block sum.  s_warp: >= blockDim/32 entries
__device__ __forceinline__ unsigned long long block_exclusive_scan64(unsigned long long v, unsigned long long* s_warp, unsigned long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < nw ? s_warp[lane] : 0ull;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
        if (lane < nw) s_warp[lane] = w;   // inclusive over warps
    }
    __syncthreads();
    const unsigned long long warp_off = warp ? s_warp[warp - 1] : 0ull;
    *total = s_warp[nw - 1];
    const unsigned long long r = warp_off + inc - v;
    __syncthreads();
    return r;
}
__device__ __forceinline__ int block_exclusive_scan(int v, unsigned long long* s_warp, int* total) {
    unsigned long long t;
    const unsigned long long r = block_exclusive_scan64((unsigned long long)(unsigned)v, s_warp, &t);
    *total = (int)t;
    return (int)r;
}

constexpr unsigned long long kAggValid = 1ull << 63;
// The aggregate word IS the message (counts + valid bit in one 64-bit store): nothing else written by the publishing block is
// read through it, so relaxed gpu-scope accesses suffice -- a release store would drain every state store the thread has in
// flight (MEMBAR.ALL.GPU on the block's critical path).
__device__ __forceinline__ void agg_publish(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v | kAggValid) : "memory");
}
__device__ __forceinline__ unsigned long long agg_wait(const unsigned long long* p) {
    unsigned long long v;
    unsigned spins = 0;
    do {
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
        if (!(v & kAggValid) && ++spins > (1u << 24)) { printf("b2dt: sweep aggregate wait timed out\n"); __trap(); }
    } while (!(v & kAggValid));
    return v & ~kAggValid;
}

// ------------------------------------------------------------------------------------------------------------------
// (1) sweep
// ------------------------------------------------------------------------------------------------------------------
// 64-bit inclusive warp scan + one barrier: every thread adds the totals of the warps before its own (s_warp: [2][8], the
// caller alternates the half so that no trailing barrier is needed)
__device__ __forceinline__ unsigned long long sweep_scan(unsigned long long v, unsigned long long* s_warp, unsigned long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    unsigned long long before = 0ull, all = 0ull;
#pragma unroll
    for (int w = 0; w < kChunk / 32; ++w) { const unsigned long long t = s_warp[w]; all += t; if (w < warp) before += t; }
    *total = all;
    return before + inc - v;
}

// Block b = chunk (b % nchunks) of stream (b / nchunks).  The aggregate look-back below waits for blocks with a LOWER block
// index only; the hardware dispatches the blocks of a 1-D grid in index order, so a waiting block's predecessors are always
// resident or finished (a bounded spin traps instead of hanging should that ever not hold).
constexpr int kGrid = 8;
// cell of a coordinate: monotonic in v, clamped to the grid (float -> int conversion saturates; NaN gives cell 0)
__device__ __forceinline__ int grid_cell(float v, float lo, float cells_per_unit) {
    return min(max((int)((v - lo) * cells_per_unit), 0), kGrid - 1);
}

template <int MODE>
__global__ void __launch_bounds__(kChunk, B2_SWEEP_BLOCKS) sweep_kernel(const Bank b, const Frame fr) {
    extern __shared__ float4 s_det[];                              // [D] detections of the stream
    __shared__ __align__(16) float s_rows[kChunk * B2_TRACK_COLS];
    __shared__ unsigned long long s_warp[kChunk / 32];
    __shared__ int s_cnt[3];
    __shared__ int s_done;                                         // warps that have finished (the last one writes the chunk's counters)
    __shared__ __align__(16) unsigned long long s_cell[kGrid * kGrid * 2];   // detection grid: bit d of cell (cy, cx) = detection d touches it
    __shared__ float s_grid[4];                                    // grid origin (x, y) and cells per unit length (x, y)
    const int tid = threadIdx.x;
    pdl_launch_dependents();            // resolve_kernel's blocks may be placed as soon as every block of this grid has started and SMs free up
    const int s = (int)(blockIdx.x / (unsigned)b.nchunks), c = (int)(blockIdx.x % (unsigned)b.nchunks);
    unsigned long long* agg = b.agg + (size_t)s * b.nchunks;
    const int chunk_slots = min(kChunk, b.C - c * kChunk);
    // a chunk that was entirely free after the previous frame has nothing to predict or emit: one word read, no slot touched
    if (b.chunk_free[(size_t)s * b.nchunks + c] == chunk_slots) {
        if (tid == 0) agg_publish(agg + c, 0ull);
        return;
    }
    if (tid < 3) s_cnt[tid] = 0;
    if (tid == 3) s_done = 0;
    const int t = c * kChunk + tid;
    const bool in = tid < chunk_slots;
    const int g = s * b.C + (in ? t : c * kChunk);
    const size_t N = b.N;
    // ---- phase 1 loads: what decides the output positions -- id, state vector, age, time since update (11 coalesced 4-byte loads
    //      per thread, independent of each other; dead slots of a live chunk are read and ignored) ----
    float x[8], p[6], m[6];
    int id = II(b, ID, g);
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = b.f[(size_t)(X0 + k) * N + g];
    int age = II(b, AGE, g), tsu = II(b, TSU, g);
    if (!in) id = 0;
    const bool live = id != 0;
    // ---- the stream's detections.  Their count and the rows a thread will need (row tid for the shared copy; rows lane, lane + 32,
    //      .. for warp 0, which builds the grid) are requested together with the state loads above, BEFORE the count is known:
    //      count -> rows -> barrier was two dependent round trips that every warp of the block then sat out at the barrier (ncu:
    //      22 % of a C3 frame's stall samples).  Rows past the count are allocated (the list is [S][max_dets][cols]) and ignored ----
    const int Dn = fr.det_counts[s];
    const float* const drow = fr.dets + (size_t)s * b.max_dets * fr.det_cols;
    float4 dmine = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < b.max_dets) { const float* r = drow + (size_t)tid * fr.det_cols; dmine = make_float4(r[0], r[1], r[2], r[3]); }
    float4 q[4];
    if (tid < 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int d = tid + 32 * k;
            q[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (d < b.max_dets) { const float* r = drow + (size_t)d * fr.det_cols; q[k] = make_float4(r[0], r[1], r[2], r[3]); }
        }
    }
    const int D = min(Dn, b.max_dets);
    if (tid < D) s_det[tid] = dmine;
    for (int d = tid + kChunk; d < D; d += kChunk) {
        const float* r = drow + (size_t)d * fr.det_cols;
        s_det[d] = make_float4(r[0], r[1], r[2], r[3]);
    }
    // ---- detection grid (0 < D <= 128): kGrid x kGrid cells over the detections' bounding range, per cell the bit set of the detections
    //      that touch it.  A track then tests only the detections of the cells its predicted box touches (a handful instead of D).
    //      Exact: the cell of a coordinate is a monotonic map clamped to the grid, so two boxes that share a point share a cell; the
    //      IoU test itself is unchanged.  Built by warp 0; the barrier below publishes it.  (Tried: a private copy and grid per warp
    //      and no block barrier -- every warp then requests every row, twice the L1 sectors, coasting sweep 58 -> 84 us) ----
    const bool use_grid = D > 0 && D <= 128;
    if (use_grid && tid < 32) {
        float lo_x = INFINITY, lo_y = INFINITY, hi_x = -INFINITY, hi_y = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int d = tid + 32 * k;
            if (d < D) {
                q[k] = make_float4(fminf(q[k].x, q[k].z), fminf(q[k].y, q[k].w), fmaxf(q[k].x, q[k].z), fmaxf(q[k].y, q[k].w));
                lo_x = fminf(lo_x, q[k].x); lo_y = fminf(lo_y, q[k].y); hi_x = fmaxf(hi_x, q[k].z); hi_y = fmaxf(hi_y, q[k].w);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo_x = fminf(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, o)); lo_y = fminf(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, o));
            hi_x = fmaxf(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, o)); hi_y = fmaxf(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, o));
        }
        const float gx = hi_x > lo_x ? (float)kGrid / (hi_x - lo_x) : 0.f, gy = hi_y > lo_y ? (float)kGrid / (hi_y - lo_y) : 0.f;
        for (int i = tid; i < kGrid * kGrid * 2; i += 32) s_cell[i] = 0ull;
        if (tid == 0) { s_grid[0] = lo_x; s_grid[1] = lo_y; s_grid[2] = gx; s_grid[3] = gy; }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int d = tid + 32 * k;
            if (d < D) {
                const int cx0 = grid_cell(q[k].x, lo_x, gx), cx1 = grid_cell(q[k].z, lo_x, gx);
                const int cy0 = grid_cell(q[k].y, lo_y, gy), cy1 = grid_cell(q[k].w, lo_y, gy);
                for (int cy = cy0; cy <= cy1; ++cy)
                    for (int cx = cx0; cx <= cx1; ++cx) atomicOr(&s_cell[(cy * kGrid + cx) * 2 + (d >> 6)], 1ull << (d & 63));
            }
        }
    }
    __syncthreads();

    // ---- predict of the state vector (:184-203) and the candidate test ----
    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
    int npairs = 0;
    const float thr = b.iou_thr;
    // IoU of detection d with the predicted box when it makes the pair a candidate, else a negative number
    auto pair_iou = [&](int d) -> float {
        const float4 db = s_det[d];
        if (fminf(db.z, box.z) > fmaxf(db.x, box.x) && fminf(db.w, box.w) > fmaxf(db.y, box.y)) {
            const float v = iou_ref(db, box);
            if (MODE ? v > thr : v >= thr) return v;                // mode 1 candidates: strictly above (motion_compensated_multi_tracker.py:262)
        }
        return -1.f;
    };
    // bit sets (detections 0..63, 64..127) of the cells the predicted box touches
    auto touched = [&](unsigned long long& m0, unsigned long long& m1) {
        const float lo_x = s_grid[0], lo_y = s_grid[1], gx = s_grid[2], gy = s_grid[3];
        const int cx0 = grid_cell(fminf(box.x, box.z), lo_x, gx), cx1 = grid_cell(fmaxf(box.x, box.z), lo_x, gx);
        const int cy0 = grid_cell(fminf(box.y, box.w), lo_y, gy), cy1 = grid_cell(fmaxf(box.y, box.w), lo_y, gy);
        m0 = 0ull; m1 = 0ull;
        for (int cy = cy0; cy <= cy1; ++cy)
            for (int cx = cx0; cx <= cx1; ++cx) {
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&s_cell[(cy * kGrid + cx) * 2]);
                m0 |= v.x; m1 |= v.y;
            }
    };
    if (live) {
        x[0] += x[4]; x[1] += x[5]; x[2] += x[6]; x[3] += x[7];
        age += 1; tsu += 1;
        box = MODE ? blended_box(b, g, age, x[0], x[1], x[2], x[3])
                   : make_float4(x[0] - x[2] / 2.f, x[1] - x[3] / 2.f, x[0] + x[2] / 2.f, x[1] + x[3] / 2.f);   // state_to_bbox :121-135
        if (use_grid) {
            unsigned long long m0, m1;
            touched(m0, m1);
            while (m0) { const int d = __ffsll((long long)m0) - 1; m0 &= m0 - 1; npairs += pair_iou(d) >= 0.f ? 1 : 0; }
            while (m1) { const int d = 63 + __ffsll((long long)m1); m1 &= m1 - 1; npairs += pair_iou(d) >= 0.f ? 1 : 0; }
        } else if (D > 0) {
            for (int d = 0; d < D; ++d) npairs += pair_iou(d) >= 0.f ? 1 : 0;
        }
    }
    const bool cand = npairs > 0;
    // should_delete (:385-405) of a track no detection can match: it is reported (emitted) unless it is deleted
    const bool del = live && !cand && (tsu > b.max_lost || (age < 5 && tsu > 15) || (age < 10 && tsu > 30));
    const int emit = (live && !cand && !del) ? 1 : 0;
    // ---- phase 2 loads, issued now: covariance, motion statistics, lifecycle counters (18 loads).  Their latency runs under the
    //      block scan, the publication of the chunk's counts and the other blocks' look-back, none of which needs them ----
#pragma unroll
    for (int k = 0; k < 6; ++k) p[k] = b.f[(size_t)(PPX + k) * N + g];
#pragma unroll
    for (int k = 0; k < 6; ++k) m[k] = b.f[(size_t)(VAVGX + k) * N + g];
    int hits = II(b, HITS, g);
    int lostf = II(b, LOSTF, g), islost = II(b, ISLOST, g), tlen = II(b, TLEN, g), thead = II(b, THEAD, g);
    // ---- positions: block scan + publication of this chunk's counts (the stream's later chunks look back over them) ----
    unsigned long long total;
    const unsigned long long mine = (unsigned long long)emit | ((unsigned long long)(cand ? 1 : 0) << 16) | ((unsigned long long)npairs << 32);
    const unsigned long long off = sweep_scan(mine, s_warp, &total);
    if (tid == 0) agg_publish(agg + c, total);

    // ---- the rest of the predict: covariance, trajectory ring ----
    if (live) {
        p[0] = p[0] + 2.f * p[1] + p[2] + Q_POS; p[1] = p[1] + p[2]; p[2] = p[2] + Q_VEL;
        p[3] = p[3] + 2.f * p[4] + p[5] + Q_SIZE; p[4] = p[4] + p[5]; p[5] = p[5] + Q_SVEL;
        b.traj[(size_t)(2 * thead) * N + g] = x[0]; b.traj[(size_t)(2 * thead + 1) * N + g] = x[1];
        thead = thead + 1 == kTraj ? 0 : thead + 1; tlen = min(tlen + 1, kTraj);
    }
    int terminated = 0, long_term = 0, freed = in && !live ? 1 : 0;
    float bx = 0.f, by = 0.f, bw = 0.f, bh = 0.f, conf = 0.f;
    if (live && !cand) {
        // ---- no detection can match this track: mark_as_lost (:299-317), delete, get_track_info (:335-383) ----
        if (!islost) { islost = 1; lostf = 0; }
        lostf += 1;
        if (del) { II(b, ID, g) = 0; terminated = 1; freed = 1; if (MODE && RI(b, MR_RESETS, g) > 0) atomicAdd(b.fcnt + s * 4 + 2, 1); }
        else {
            const int k = lostf;                                 // a lost track is always reported (multi_target_tracker.py:117-126)
            if (k <= 1) {                                        // enhanced_long_term_predict(1) -> self.predict(), 1.0 (:216-217)
                x[0] += x[4]; x[1] += x[5]; x[2] += x[6]; x[3] += x[7];
                p[0] = p[0] + 2.f * p[1] + p[2] + Q_POS; p[1] = p[1] + p[2]; p[2] = p[2] + Q_VEL;
                p[3] = p[3] + 2.f * p[4] + p[5] + Q_SIZE; p[4] = p[4] + p[5]; p[5] = p[5] + Q_SVEL;
                age += 1; tsu += 1;
                b.traj[(size_t)(2 * thead) * N + g] = x[0]; b.traj[(size_t)(2 * thead + 1) * N + g] = x[1];
                thead = thead + 1 == kTraj ? 0 : thead + 1; tlen = min(tlen + 1, kTraj);
                bx = x[0]; by = x[1]; bw = x[2]; bh = x[3]; conf = 1.f;
                if (MODE) {                                      // the overridden predict() returns the blended box (:300-321)
                    const float4 bb = blended_box(b, g, age, x[0], x[1], x[2], x[3]);
                    bx = (bb.x + bb.z) / 2.f; by = (bb.y + bb.w) / 2.f;
                }
            } else if (m[PCONF - VAVGX] > 0.3f) {                // high confidence: mean-velocity extrapolation (:224-236)
                bx = x[0] + m[0] * (float)k; by = x[1] + m[1] * (float)k; bw = x[2]; bh = x[3];
                conf = m[PCONF - VAVGX] * fmaxf(0.1f, 1.f - (float)k / (float)b.max_lost);
            } else {                                             // F^k x (:238-245)
                bx = x[0] + (float)k * x[4]; by = x[1] + (float)k * x[5];
                bw = x[2] + (float)k * x[6]; bh = x[3] + (float)k * x[7];
                conf = fmaxf(0.1f, 1.f - (float)k / ((float)b.max_lost * 0.5f));
            }
            long_term = tsu > 30 ? 1 : 0;
        }
    }
    // ---- write the slot back ----
    if (live && !terminated) {
#pragma unroll
        for (int k = 0; k < 4; ++k) b.f[(size_t)(X0 + k) * N + g] = x[k];
#pragma unroll
        for (int k = 0; k < 6; ++k) b.f[(size_t)(PPX + k) * N + g] = p[k];
        II(b, AGE, g) = age; II(b, TSU, g) = tsu; II(b, TLEN, g) = tlen; II(b, THEAD, g) = thead;
        if (!cand) { II(b, STREAK, g) = 0; II(b, LOSTF, g) = lostf; II(b, ISLOST, g) = 1; }
    }
    // ---- the aggregates of the stream's preceding chunks (published long ago by now), summed by every warp for itself: from
    //      here on a warp depends on no other warp of the block -- it stages its rows, copies them out and writes its list entries
    //      as soon as ITS loads are back instead of waiting at a block barrier for the slowest warp (ncu: 30 % of the samples) ----
    unsigned long long prefix = 0ull;
    for (int i = tid & 31; i < c; i += 32) prefix += agg_wait(agg + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) prefix += __shfl_xor_sync(0xffffffffu, prefix, o);
    if (terminated) atomicAdd(&s_cnt[0], 1);
    if (long_term) atomicAdd(&s_cnt[1], 1);
    if (freed) atomicAdd(&s_cnt[2], 1);
    if (emit) {
        float4* sr = reinterpret_cast<float4*>(s_rows + (int)(off & 0xFFFFu) * B2_TRACK_COLS);
        sr[0] = make_float4(__int_as_float(id), bx - bw / 2.f, by - bh / 2.f, bx + bw / 2.f);
        sr[1] = make_float4(by + bh / 2.f, conf, __int_as_float(1), __int_as_float(age));
        sr[2] = make_float4(__int_as_float(hits), __int_as_float(0), __int_as_float(tsu), __int_as_float(tsu));
        sr[3] = make_float4(__int_as_float(1), x[4], x[5], m[PCONF - VAVGX]);
        sr[4] = make_float4(__int_as_float(m[STAB - VAVGX] > 0.5f ? 1 : 0), m[SPEED - VAVGX], m[DIRN - VAVGX], __int_as_float(t));
    }
    __syncwarp();
    const int e0 = (int)(prefix & 0xFFFFu), c0 = (int)((prefix >> 16) & 0xFFFFu);
    // the rows a warp emits are contiguous in the block's order, hence in the output: coalesced 16-byte stores, warp by warp
    {
        const int w0 = (int)__shfl_sync(0xffffffffu, (unsigned)(off & 0xFFFFu), 0);        // rows emitted by the block before this warp
        const int nw = __popc(__ballot_sync(0xffffffffu, emit != 0));
        const float4* src4 = reinterpret_cast<const float4*>(s_rows + w0 * B2_TRACK_COLS);
        float4* dst4 = reinterpret_cast<float4*>(fr.out_rows + ((size_t)s * fr.out_cap + e0 + w0) * B2_TRACK_COLS);
        const int n4 = max(min(e0 + w0 + nw, fr.out_cap) - (e0 + w0), 0) * (B2_TRACK_COLS / 4);
        for (int i = tid & 31; i < n4; i += 32) dst4[i] = src4[i];
    }
    if (MODE && emit && fr.out_extra && e0 + (int)(off & 0xFFFFu) < fr.out_cap)
        reinterpret_cast<float4*>(fr.out_extra)[(size_t)s * fr.out_cap + e0 + (int)(off & 0xFFFFu)] =
            make_float4(__int_as_float(RI(b, MR_RESETS, g)), __int_as_float(age - RI(b, MR_LASTRESET, g)), RF(b, MR_MCONS, g), 0.f);
    if (emit && fr.out_traj && e0 + (int)(off & 0xFFFFu) < fr.out_cap) {
        const int pos = e0 + (int)(off & 0xFFFFu);
        float* to = fr.out_traj + ((size_t)s * fr.out_cap + pos) * kTraj * 2;
        int start = thead - tlen; if (start < 0) start += kTraj;
        for (int k = 0; k < tlen; ++k) {
            int r = start + k; if (r >= kTraj) r -= kTraj;
            to[2 * k] = b.traj[(size_t)(2 * r) * N + g]; to[2 * k + 1] = b.traj[(size_t)(2 * r + 1) * N + g];
        }
        fr.out_traj_len[(size_t)s * fr.out_cap + pos] = tlen;
    }
    if (cand) {
        const int ci = c0 + (int)((off >> 16) & 0xFFFFu);
        const size_t cb = (size_t)s * b.C + ci;
        b.ctrk_slot[cb] = t; b.cbox[cb] = box; b.cid[cb] = id;
        unsigned long long pp = (prefix >> 32) + (off >> 32);
        // the track's pairs in detection order (bits are taken from the lowest up), as the loop over all detections listed them
        auto list_pair = [&](int d) {
            const float v = pair_iou(d);
            if (v >= 0.f) {
                if (pp < (unsigned long long)b.pair_cap)
                    b.pairs[(size_t)s * b.pair_cap + pp] = make_uint4(__float_as_uint(v), (unsigned)d, (unsigned)ci, (unsigned)id);
                ++pp;
            }
        };
        if (use_grid) {
            unsigned long long m0, m1;
            touched(m0, m1);
            while (m0) { const int d = __ffsll((long long)m0) - 1; m0 &= m0 - 1; list_pair(d); }
            while (m1) { const int d = 63 + __ffsll((long long)m1); m1 &= m1 - 1; list_pair(d); }
        } else {
            for (int d = 0; d < D; ++d) list_pair(d);
        }
    }
    // the chunk's counters go out with the LAST warp to get here (no block barrier: the other warps have left already)
    __syncwarp();
    if ((tid & 31) == 0) {
        __threadfence_block();
        if (atomicAdd(&s_done, 1) == kChunk / 32 - 1) {
            b.chunk_free[(size_t)s * b.nchunks + c] = atomicAdd(&s_cnt[2], 0);
            const int n0 = atomicAdd(&s_cnt[0], 0), n1 = atomicAdd(&s_cnt[1], 0);
            if (n0) atomicAdd(b.fcnt + s * 4 + 0, n0);
            if (n1) atomicAdd(b.fcnt + s * 4 + 1, n1);
        }
    }
}

// analyze_motion_pattern (:137-163) + _calculate_direction_consistency (:165-182) over the velocity ring, by one warp
// (lane <-> ring entry, two entries per lane).  Sums are shuffle trees in fp32: within the 2e-4 / 1e-3 gates of
// tests/test_gpu_tracker.py against the float64 reference.
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ void analyze_slot_warp(const Bank& b, int g, int lane) {
    const int n = II(b, NVEL, g);
    if (n < 5) return;                                      // uniform: every lane reads the same slot
    const int head = II(b, VHEAD, g);
    int start = head - n; if (start < 0) start += kVelRing;
    float vx[2], vy[2]; bool ok[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int k = lane + 32 * e;                        // chronological index
        ok[e] = k < n;
        int r = start + k; if (r >= kVelRing) r -= kVelRing;
        vx[e] = ok[e] ? b.vel[(size_t)(2 * r) * b.N + g] : 0.f;
        vy[e] = ok[e] ? b.vel[(size_t)(2 * r + 1) * b.N + g] : 0.f;
    }
    const float mx = warp_sum(vx[0] + vx[1]) / n, my = warp_sum(vy[0] + vy[1]) / n;
    float qx = 0.f, qy = 0.f;
#pragma unroll
    for (int e = 0; e < 2; ++e) if (ok[e]) { const float dx = vx[e] - mx, dy = vy[e] - my; qx += dx * dx; qy += dy * dy; }
    const float sdx = sqrtf(warp_sum(qx) / n), sdy = sqrtf(warp_sum(qy) / n);
    const float PI = 3.14159265358979323846f;
    float ang[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) ang[e] = ok[e] ? atan2f(vy[e], vx[e]) : 0.f;
    // angle of the chronologically previous entry: lane - 1 of the same half, or lane 31 of the first half for entry 32
    const float up0 = __shfl_up_sync(0xffffffffu, ang[0], 1), up1 = __shfl_up_sync(0xffffffffu, ang[1], 1);
    const float last0 = __shfl_sync(0xffffffffu, ang[0], 31);
    const float prev[2] = {up0, lane == 0 ? last0 : up1};
    float c[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int k = lane + 32 * e;
        float d = ang[e] - prev[e];
        if (!(fabsf(d) < PI)) d = d - 2.f * PI * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
        c[e] = (ok[e] && k > 0) ? d : 0.f;
    }
    const float dmean = warp_sum(c[0] + c[1]) / (n - 1);
    float qv = 0.f;
#pragma unroll
    for (int e = 0; e < 2; ++e) { const int k = lane + 32 * e; if (ok[e] && k > 0) { const float t = c[e] - dmean; qv += t * t; } }
    const float dstd = sqrtf(warp_sum(qv) / (n - 1));
    if (lane == 0) {
        const float speed_stab = 1.f / (1.f + (sdx + sdy) / 2.f);
        const float dir_cons = 1.f / (1.f + dstd * 10.f);
        const float stab = (speed_stab + dir_cons) / 2.f;
        FF(b, VAVGX, g) = mx; FF(b, VAVGY, g) = my;
        FF(b, SPEED, g) = sqrtf(mx * mx + my * my);
        FF(b, DIRN, g) = atan2f(my, mx);
        FF(b, STAB, g) = stab;
        FF(b, PCONF, g) = stab * fminf((float)n / 30.f, 1.f);
    }
}

// Kalman update with measurement z = bbox_to_state(det)  (:249-297); the motion analysis follows separately (one warp per track)
__device__ __forceinline__ void update_slot(const Bank& b, int g, const float4& d) {
    // Every field the update touches is loaded first, then everything is computed, then everything is stored.  Written as
    // read-modify-writes on the bank (`FF(b, X0, g) += ...`) the compiler must assume that a store to the bank may alias the next
    // load from it: ~25 global round trips one after the other, by ONE thread per matched track, with the other ~480 threads of
    // the stream's CTA waiting at the next barrier (ncu: 43 % of the kernel's samples there).
    const size_t N = b.N;
    float x[8], pp[6];
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = b.f[(size_t)(X0 + k) * N + g];
#pragma unroll
    for (int k = 0; k < 6; ++k) pp[k] = b.f[(size_t)(PPX + k) * N + g];
    const int hits = II(b, HITS, g), streak = II(b, STREAK, g), islost = II(b, ISLOST, g);
    const int head = II(b, VHEAD, g), nvel = II(b, NVEL, g), thead = II(b, THEAD, g), tlen = II(b, TLEN, g);
    const float z0 = (d.x + d.z) / 2.f, z1 = (d.y + d.w) / 2.f, z2 = d.z - d.x, z3 = d.w - d.y;
    {   // position block (x, y share the covariance triple)
        const float pxx = pp[0], pxv = pp[1], pvv = pp[2];
        // (I - K H) P with 1 - K_x evaluated as R / S: no cancellation when P_xx >> R (long coasting tracks)
        const float S = pxx + R_MEAS, kx = pxx / S, kv = pxv / S, omk = R_MEAS / S;
        const float y0 = z0 - x[0], y1 = z1 - x[1];
        x[0] += kx * y0; x[4] += kv * y0;
        x[1] += kx * y1; x[5] += kv * y1;
        pp[0] = omk * pxx; pp[1] = omk * pxv; pp[2] = pvv - kv * pxv;
    }
    {   // size block (w, h)
        const float pxx = pp[3], pxv = pp[4], pvv = pp[5];
        const float S = pxx + R_MEAS, kx = pxx / S, kv = pxv / S, omk = R_MEAS / S;
        const float y2 = z2 - x[2], y3 = z3 - x[3];
        x[2] += kx * y2; x[6] += kv * y2;
        x[3] += kx * y3; x[7] += kv * y3;
        pp[3] = omk * pxx; pp[4] = omk * pxv; pp[5] = pvv - kv * pxv;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) b.f[(size_t)(X0 + k) * N + g] = x[k];
#pragma unroll
    for (int k = 0; k < 6; ++k) b.f[(size_t)(PPX + k) * N + g] = pp[k];
    II(b, TSU, g) = 0; II(b, HITS, g) = hits + 1; II(b, STREAK, g) = streak + 1;
    if (islost) { II(b, ISLOST, g) = 0; II(b, LOSTF, g) = 0; }
    // velocity ring push, trajectory push (push_traj)
    b.vel[(size_t)(2 * head) * N + g] = x[4];
    b.vel[(size_t)(2 * head + 1) * N + g] = x[5];
    II(b, VHEAD, g) = head + 1 == kVelRing ? 0 : head + 1;
    II(b, NVEL, g) = min(nvel + 1, kVelRing);
    b.traj[(size_t)(2 * thead) * N + g] = x[0]; b.traj[(size_t)(2 * thead + 1) * N + g] = x[1];
    II(b, THEAD, g) = thead + 1 == kTraj ? 0 : thead + 1;
    II(b, TLEN, g) = min(tlen + 1, kTraj);
}

// AircraftKalmanTracker.__init__ (:23-101)
__device__ __forceinline__ void init_slot(const Bank& b, int g, const float4& d, int id) {
    const float cx = (d.x + d.z) / 2.f, cy = (d.y + d.w) / 2.f;
    FF(b, X0, g) = cx; FF(b, X1, g) = cy; FF(b, X2, g) = d.z - d.x; FF(b, X3, g) = d.w - d.y;
    FF(b, X4, g) = 0.f; FF(b, X5, g) = 0.f; FF(b, X6, g) = 0.f; FF(b, X7, g) = 0.f;
    FF(b, PPX, g) = P0_POS; FF(b, PPV, g) = 0.f; FF(b, PVV, g) = P0_VEL;
    FF(b, PSX, g) = P0_POS; FF(b, PSV, g) = 0.f; FF(b, PSVV, g) = P0_SVEL;
    FF(b, VAVGX, g) = 0.f; FF(b, VAVGY, g) = 0.f; FF(b, DIRN, g) = 0.f; FF(b, SPEED, g) = 0.f; FF(b, STAB, g) = 0.f; FF(b, PCONF, g) = 0.f;
    II(b, ID, g) = id; II(b, AGE, g) = 0; II(b, HITS, g) = 1; II(b, STREAK, g) = 1; II(b, TSU, g) = 0;
    II(b, LOSTF, g) = 0; II(b, ISLOST, g) = 0; II(b, NVEL, g) = 0; II(b, VHEAD, g) = 0; II(b, TLEN, g) = 0; II(b, THEAD, g) = 0;
    push_traj(b, g, cx, cy);
}

// ---- mode 1: MotionResetKalmanTracker (camera_motion_compensation/motion_reset_kalman_tracker.py) ----
__device__ __forceinline__ void mr_push_pos(const Bank& b, int g, float cx, float cy) {       // position_history.append
    int head = RI(b, MR_PHHEAD, g);
    RF(b, MR_PH + 2 * head, g) = cx; RF(b, MR_PH + 2 * head + 1, g) = cy;
    RI(b, MR_PHHEAD, g) = head + 1 == kPosRing ? 0 : head + 1;
    RI(b, MR_PHLEN, g) = min(RI(b, MR_PHLEN, g) + 1, kPosRing);
}
__device__ __forceinline__ void mr_init_slot(const Bank& b, int g, const float4& d) {         // __init__ :37-58
    RI(b, MR_PHLEN, g) = 0; RI(b, MR_PHHEAD, g) = 0; RI(b, MR_MSLEN, g) = 0; RI(b, MR_MSHEAD, g) = 0;
    RI(b, MR_RESETS, g) = 0; RI(b, MR_LASTRESET, g) = -999; RF(b, MR_MCONS, g) = 0.f;
    mr_push_pos(b, g, (d.x + d.z) / 2.f, (d.y + d.w) / 2.f);
    RF(b, MR_BB, g) = d.x; RF(b, MR_BB + 1, g) = d.y; RF(b, MR_BB + 2, g) = d.z; RF(b, MR_BB + 3, g) = d.w;
    RI(b, MR_BBLEN, g) = 1;
}
// the k-th most recent stored position (k = 1: last)
__device__ __forceinline__ float2 mr_pos_back(const Bank& b, int g, int k) {
    int r = RI(b, MR_PHHEAD, g) - k; if (r < 0) r += kPosRing;
    return make_float2(RF(b, MR_PH + 2 * r, g), RF(b, MR_PH + 2 * r + 1, g));
}
// should_reset (:161-244) with its side effects (a motion score is stored by the jump detector, motion_consistency is refreshed
// when a detector fires); returns the reset confidence (> 1: reset)
__device__ float mr_should_reset(const Bank& b, int g, const float4& d) {
    const int since = II(b, AGE, g) - RI(b, MR_LASTRESET, g);
    if (since < kResetCooldown) return 0.f;
    const float cx = (d.x + d.z) / 2.f, cy = (d.y + d.w) / 2.f;
    const int n = RI(b, MR_PHLEN, g);
    float fsum = 0.f; int nf = 0;
    if (n >= 2) {                                               // _detect_position_jump :78-94
        const int m = min(n, 3);
        float ax = 0.f, ay = 0.f;
        for (int k = m; k >= 1; --k) { const float2 q = mr_pos_back(b, g, k); ax += q.x; ay += q.y; }
        ax /= (float)m; ay /= (float)m;
        const float dist = sqrtf((cx - ax) * (cx - ax) + (cy - ay) * (cy - ay));
        int head = RI(b, MR_MSHEAD, g);
        RF(b, MR_MS + head, g) = fminf(dist / kJumpThr, 3.f);
        RI(b, MR_MSHEAD, g) = head + 1 == kScoreRing ? 0 : head + 1;
        RI(b, MR_MSLEN, g) = min(RI(b, MR_MSLEN, g) + 1, kScoreRing);
        if (dist > kJumpThr) { fsum += fminf(dist / kJumpThr, 2.f); ++nf; }
    }
    if (n >= 3) {                                               // _detect_velocity_change :96-121
        const float2 p0 = mr_pos_back(b, g, 3), p1 = mr_pos_back(b, g, 2), p2 = mr_pos_back(b, g, 1);
        const float v1 = sqrtf((p1.x - p0.x) * (p1.x - p0.x) + (p1.y - p0.y) * (p1.y - p0.y));
        const float v2 = sqrtf((p2.x - p1.x) * (p2.x - p1.x) + (p2.y - p1.y) * (p2.y - p1.y));
        const float v3 = sqrtf((cx - p2.x) * (cx - p2.x) + (cy - p2.y) * (cy - p2.y));
        const float change = fabsf(v3 - (v1 + v2) / 2.f);
        if (change > kVelThr) { fsum += fminf(change / kVelThr, 2.f); ++nf; }
    }
    if (RI(b, MR_BBLEN, g) >= 2) {                              // _detect_size_change :123-142
        const float pw = fmaxf(RF(b, MR_BB + 2, g) - RF(b, MR_BB, g), 1.f), ph = fmaxf(RF(b, MR_BB + 3, g) - RF(b, MR_BB + 1, g), 1.f);
        const float m = fmaxf(fabsf((d.z - d.x) / pw - 1.f), fabsf((d.w - d.y) / ph - 1.f));
        if (m > kSizeThr) { fsum += m / kSizeThr; ++nf; }
    }
    if (!nf) return 0.f;
    float conf = fsum / (float)nf;
    float mc = 0.f;                                             // _calculate_motion_consistency :144-159
    const int ns = RI(b, MR_MSLEN, g);
    if (ns >= 3) {
        float sm = 0.f;
        for (int k = 0; k < ns; ++k) sm += RF(b, MR_MS + k, g);       // mean / variance do not depend on the ring order
        const float mean = sm / (float)ns;
        float var = 0.f;
        for (int k = 0; k < ns; ++k) { const float e = RF(b, MR_MS + k, g) - mean; var += e * e; }
        var /= (float)ns;
        mc = mean > 0.f ? fmaxf(0.f, 1.f - var / (mean + 0.1f)) : 1.f;
    }
    RF(b, MR_MCONS, g) = mc;
    if (mc < 0.3f) conf *= 1.5f;
    if (RI(b, MR_RESETS, g) > 0 && since < 50) conf *= 0.8f;
    return conf;
}
// _perform_reset (:246-279): the state is overwritten by the detection, velocities zeroed, P rescaled (velocity block x100,
// position block x5, cross terms untouched), histories cleared; is_lost / lost_frames are NOT cleared
__device__ void mr_reset_slot(const Bank& b, int g, const float4& d) {
    RI(b, MR_RESETS, g) += 1; RI(b, MR_LASTRESET, g) = II(b, AGE, g);
    const float cx = (d.x + d.z) / 2.f, cy = (d.y + d.w) / 2.f;
    FF(b, X0, g) = cx; FF(b, X1, g) = cy; FF(b, X2, g) = d.z - d.x; FF(b, X3, g) = d.w - d.y;
    FF(b, X4, g) = 0.f; FF(b, X5, g) = 0.f; FF(b, X6, g) = 0.f; FF(b, X7, g) = 0.f;
    FF(b, PPX, g) *= 5.f; FF(b, PVV, g) *= 100.f; FF(b, PSX, g) *= 5.f; FF(b, PSVV, g) *= 100.f;
    II(b, TLEN, g) = 0; II(b, THEAD, g) = 0; push_traj(b, g, cx, cy);
    II(b, NVEL, g) = 0; II(b, VHEAD, g) = 0;
    RI(b, MR_PHLEN, g) = 0; RI(b, MR_PHHEAD, g) = 0; mr_push_pos(b, g, cx, cy);
    RI(b, MR_MSLEN, g) = 0; RI(b, MR_MSHEAD, g) = 0;
    II(b, HITS, g) += 1; II(b, STREAK, g) += 1; II(b, TSU, g) = 0;
}

// get_track_info (:335-383) incl. get_lost_prediction / enhanced_long_term_predict side effects; the row goes to global
// memory as five 16-byte stores
__device__ void emit_slot(const Bank& b, int g, float* out_row, float* traj_out, int32_t* traj_len_out, int slot, int* long_term) {
    float bx, by, bw, bh, conf; int predicted = II(b, TSU, g) > 0;
    if (predicted) {
        if (II(b, ISLOST, g)) {
            const int k = II(b, LOSTF, g);
            if (k <= 1) {                                   // enhanced_long_term_predict(1) -> self.predict(), 1.0 (:216-217)
                predict_slot(b, g);
                bx = FF(b, X0, g); by = FF(b, X1, g); bw = FF(b, X2, g); bh = FF(b, X3, g); conf = 1.f;
                if (b.mode) {                               // the overridden predict() returns the blended box
                    const float4 bb = blended_box(b, g, II(b, AGE, g), bx, by, bw, bh);
                    bx = (bb.x + bb.z) / 2.f; by = (bb.y + bb.w) / 2.f;
                }
            } else if (FF(b, PCONF, g) > 0.3f) {            // high confidence: mean-velocity extrapolation (:224-236)
                bx = FF(b, X0, g) + FF(b, VAVGX, g) * (float)k; by = FF(b, X1, g) + FF(b, VAVGY, g) * (float)k;
                bw = FF(b, X2, g); bh = FF(b, X3, g);
                conf = FF(b, PCONF, g) * fmaxf(0.1f, 1.f - (float)k / (float)b.max_lost);
            } else {                                        // F^k x (:238-245)
                bx = FF(b, X0, g) + (float)k * FF(b, X4, g); by = FF(b, X1, g) + (float)k * FF(b, X5, g);
                bw = FF(b, X2, g) + (float)k * FF(b, X6, g); bh = FF(b, X3, g) + (float)k * FF(b, X7, g);
                conf = fmaxf(0.1f, 1.f - (float)k / ((float)b.max_lost * 0.5f));
            }
        } else {
            bx = FF(b, X0, g); by = FF(b, X1, g); bw = FF(b, X2, g); bh = FF(b, X3, g);
            conf = fmaxf(0.3f, 1.f - (float)II(b, TSU, g) / 60.f);
        }
    } else {
        bx = FF(b, X0, g); by = FF(b, X1, g); bw = FF(b, X2, g); bh = FF(b, X3, g); conf = 1.f;
    }
    const int tsu = II(b, TSU, g);
    if (predicted && tsu > 30) *long_term += 1;
    if (!out_row) return;                                    // beyond the caller's row capacity: state side effects only
    // every field first, then the five stores: a store to the row may alias the bank as far as the compiler knows, so loads
    // written between the stores would each wait for the previous round trip
    const int rid = II(b, ID, g), rage = II(b, AGE, g), rhits = II(b, HITS, g), rstreak = II(b, STREAK, g);
    const float vx = FF(b, X4, g), vy = FF(b, X5, g), pc = FF(b, PCONF, g), stab = FF(b, STAB, g), spd = FF(b, SPEED, g), dirn = FF(b, DIRN, g);
    float4* o = reinterpret_cast<float4*>(out_row);
    o[0] = make_float4(__int_as_float(rid), bx - bw / 2.f, by - bh / 2.f, bx + bw / 2.f);
    o[1] = make_float4(by + bh / 2.f, conf, __int_as_float(predicted), __int_as_float(rage));
    o[2] = make_float4(__int_as_float(rhits), __int_as_float(rstreak), __int_as_float(tsu), __int_as_float(tsu));
    o[3] = make_float4(__int_as_float(predicted), vx, vy, pc);
    o[4] = make_float4(__int_as_float(stab > 0.5f ? 1 : 0), spd, dirn, __int_as_float(slot));
    if (traj_out) {
        const int len = II(b, TLEN, g), head = II(b, THEAD, g);
        int start = head - len; if (start < 0) start += kTraj;
        for (int k = 0; k < len; ++k) {
            int r = start + k; if (r >= kTraj) r -= kTraj;
            traj_out[2 * k] = b.traj[(size_t)(2 * r) * b.N + g];
            traj_out[2 * k + 1] = b.traj[(size_t)(2 * r + 1) * b.N + g];
        }
        *traj_len_out = len;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// (2) resolve: one CTA per stream on the candidate lists
// ------------------------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(kResolveThreads, 2) resolve_kernel(const Bank b, const Frame fr) {
    __shared__ float4 s_det[kMaxDetsSmem];
    __shared__ int s_dmatch[kMaxDetsSmem];
    __shared__ unsigned long long d_best[kMaxDetsSmem];      // sparse rounds: best key per detection; dense rounds: {best track, IoU}
    __shared__ int s_list[kMaxDetsSmem];                     // dense rounds: staged acceptances; then matched tracks; then new detections
    __shared__ unsigned long long t_best[kCtSmem];
    __shared__ int l_match[kCtSmem];
    __shared__ unsigned long long s_warp[kResolveThreads / 32];
    __shared__ unsigned long long s_tot;
    __shared__ int s_progress, s_an, s_emit_base, s_cnt[4];
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kResolveThreads / 32;
    const int g0 = s * b.C;
    const int D = min(fr.det_counts[s], b.max_dets);
    if (tid == 0) { s_tot = 0ull; s_an = 0; }
    if (tid < 4) s_cnt[tid] = 0;
    // the detections are inputs of the whole update (written before the sweep was launched): they are copied while the sweep's last
    // blocks still run.  Everything the sweep writes -- aggregates, lists, the bank, its counters -- is read after pdl_wait()
    for (int d = tid; d < D; d += kResolveThreads) {
        const float* r = fr.dets + ((size_t)s * b.max_dets + d) * fr.det_cols;
        s_det[d] = make_float4(r[0], r[1], r[2], r[3]);
        s_dmatch[d] = -1;
    }
    __syncthreads();
    pdl_wait();
    {   // totals of the sweep; the aggregates are consumed (zero = not yet published, for the next frame)
        unsigned long long* agg = b.agg + (size_t)s * b.nchunks;
        unsigned long long sum = 0ull;
        for (int i = tid; i < b.nchunks; i += kResolveThreads) { sum += agg[i] & ~kAggValid; agg[i] = 0ull; }
        if (sum) atomicAdd(&s_tot, sum);
    }
    __syncthreads();
    const int E1 = (int)(s_tot & 0xFFFFu), T = (int)((s_tot >> 16) & 0xFFFFu);
    const unsigned long long M64 = s_tot >> 32;
    const int frame = b.frame_count[s] + 1;
    // everything the last step (stats, counters) needs from global memory is requested now: on a frame with nothing to resolve the
    // kernel is a chain of dependent round trips, and these would be the last links of it
    const int id0 = b.next_id[s];
    int fc0 = 0, fc1 = 0;                                  // (fcnt[2] is also incremented by this kernel: read at the end)
    long long st_in[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (tid == 0) {
        const int32_t* fcp = b.fcnt + s * 4;
        fc0 = fcp[0]; fc1 = fcp[1];
#pragma unroll
        for (int k = 0; k < 8; ++k) st_in[k] = b.stats[(size_t)s * 8 + k];
    }
    const float thr = b.iou_thr;
    const int32_t* cslot = b.ctrk_slot + (size_t)g0;
    const float4* cbox = b.cbox + (size_t)g0;
    const int32_t* cid = b.cid + (size_t)g0;
    const bool sparse = M64 <= (unsigned long long)b.pair_cap && T <= kCtSmem;
    int* match = sparse ? l_match : b.cmatch + (size_t)g0;
    for (int i = tid; i < T; i += kResolveThreads) match[i] = -1;
    __syncthreads();

    if (T > 0 && D > 0) {
        if (sparse) {
            // ---- mutual-best rounds on the pair list.  A pair is accepted when the track is the detection's best free candidate
            //      by (IoU, lowest track id) and the detection is the track's best free candidate by (IoU, lowest detection
            //      index): exactly the pairs the reference's descending-IoU greedy walk takes
            //      (enhanced_multi_target_tracker.py:234-270).  Decisions of a round read only the state of the round's start. ----
            const int M = (int)M64;
            const uint4* pairs = b.pairs + (size_t)s * b.pair_cap;
            while (true) {
                for (int d = tid; d < D; d += kResolveThreads) { d_best[d] = 0ull; s_list[d] = -1; }
                for (int i = tid; i < T; i += kResolveThreads) t_best[i] = 0ull;
                if (tid == 0) s_progress = 0;
                __syncthreads();
                for (int e = tid; e < M; e += kResolveThreads) {
                    const uint4 pr = pairs[e];
                    const int d = (int)pr.y, i = (int)pr.z;
                    if (s_dmatch[d] >= 0 || l_match[i] >= 0) continue;
                    const unsigned long long hi = (unsigned long long)pr.x << 32;   // IoU > 0: bits order like the float
                    // ties: mode 0 lowest (detection, track id); mode 1 the reference sorts (iou, d, t) tuples descending: highest
                    atomicMax(&d_best[d], hi | (MODE ? pr.w : (unsigned)(0xFFFFFFFFu - pr.w)));
                    atomicMax(&t_best[i], hi | (MODE ? (unsigned)d : (unsigned)(0xFFFFFFFFu - (unsigned)d)));
                }
                __syncthreads();
                // an accepted pair is the unique entry whose key is the maximum of both its detection and its track; it is only
                // STAGED here (s_list[d]) and committed after a barrier, so every decision of the round reads the round-start state
                for (int e = tid; e < M; e += kResolveThreads) {
                    const uint4 pr = pairs[e];
                    const int d = (int)pr.y, i = (int)pr.z;
                    if (s_dmatch[d] >= 0 || l_match[i] >= 0) continue;
                    const unsigned long long hi = (unsigned long long)pr.x << 32;
                    if (d_best[d] == (hi | (MODE ? pr.w : (unsigned)(0xFFFFFFFFu - pr.w))) && t_best[i] == (hi | (MODE ? (unsigned)d : (unsigned)(0xFFFFFFFFu - (unsigned)d)))) {
                        s_list[d] = i; s_progress = 1;
                    }
                }
                __syncthreads();
                for (int d = tid; d < D; d += kResolveThreads)
                    if (s_list[d] >= 0) { s_dmatch[d] = s_list[d]; l_match[s_list[d]] = d; }
                const int progress = s_progress;
                __syncthreads();
                if (!progress) break;
            }
        } else {
            // ---- dense fallback (pair list overflow / very many candidate tracks): the same rounds with the IoUs recomputed ----
            int* s_bt = reinterpret_cast<int*>(d_best);
            float* s_bv = reinterpret_cast<float*>(d_best) + kMaxDetsSmem;
            while (true) {
                if (tid == 0) s_progress = 0;
                for (int d = warp; d < D; d += nwarps) {              // row pass: best free track per free detection
                    if (s_dmatch[d] >= 0) continue;
                    const float4 db = s_det[d];
                    float best = -1.f; int bt = -1, bid = MODE ? -1 : 0x7fffffff;
                    for (int i = lane; i < T; i += 32) {
                        if (match[i] >= 0) continue;
                        const float v = iou_ref(db, cbox[i]);
                        const int id = cid[i];
                        if ((MODE ? v > thr : v >= thr) && (v > best || (v == best && (MODE ? id > bid : id < bid)))) { best = v; bt = i; bid = id; }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                        const int ot = __shfl_xor_sync(0xffffffffu, bt, o), oid = __shfl_xor_sync(0xffffffffu, bid, o);
                        if (ob > best || (ob == best && (MODE ? oid > bid : oid < bid))) { best = ob; bt = ot; bid = oid; }
                    }
                    if (lane == 0) { s_bt[d] = bt; s_bv[d] = best; }
                }
                __syncthreads();
                for (int d = tid; d < D; d += kResolveThreads) {      // column check against the round-start state
                    int acc = -1;
                    if (s_dmatch[d] < 0 && s_bt[d] >= 0) {
                        const int i = s_bt[d];
                        const float v = s_bv[d];
                        const float4 tb = cbox[i];
                        bool dominated = false;
                        for (int e = 0; e < D && !dominated; ++e) {
                            if (e == d || s_dmatch[e] >= 0) continue;
                            const float ve = iou_ref(s_det[e], tb);
                            if ((MODE ? ve > thr : ve >= thr) && (ve > v || (ve == v && (MODE ? e > d : e < d)))) dominated = true;
                        }
                        if (!dominated) acc = i;
                    }
                    s_list[d] = acc;
                }
                __syncthreads();
                for (int d = tid; d < D; d += kResolveThreads)
                    if (s_list[d] >= 0) { s_dmatch[d] = s_list[d]; match[s_list[d]] = d; s_progress = 1; }
                __syncthreads();
                const int progress = s_progress;
                __syncthreads();
                if (!progress) break;
            }
        }
    }
    __syncthreads();

    // ---- candidate tracks: Kalman update (:249-297) or mark_as_lost (:299-317); should_delete (:385-405) ----
    for (int i = tid; i < T; i += kResolveThreads) {
        const int t = cslot[i], g = g0 + t;
        const int md = match[i];
        if (md >= 0) {
            if (II(b, ISLOST, g)) atomicAdd(&s_cnt[2], 1);                              // successful recovery (:73-79)
            const float4 dd = s_det[md];
            if (MODE && mr_should_reset(b, g, dd) > 1.f) {                              // MotionResetKalmanTracker.update :281-298
                mr_reset_slot(b, g, dd);
                atomicAdd(&s_cnt[3], 1);                                                // individual_resets
            } else {
                update_slot(b, g, dd);
                s_list[atomicAdd(&s_an, 1)] = t;
                if (MODE) mr_push_pos(b, g, FF(b, X0, g), FF(b, X1, g));                // the base class's append of the filtered centre
            }
            if (MODE) {
                mr_push_pos(b, g, (dd.x + dd.z) / 2.f, (dd.y + dd.w) / 2.f);
                RF(b, MR_BB, g) = dd.x; RF(b, MR_BB + 1, g) = dd.y; RF(b, MR_BB + 2, g) = dd.z; RF(b, MR_BB + 3, g) = dd.w;
                RI(b, MR_BBLEN, g) = min(RI(b, MR_BBLEN, g) + 1, 5);
            }
        } else {
            if (!II(b, ISLOST, g)) { II(b, ISLOST, g) = 1; II(b, LOSTF, g) = 0; }
            II(b, LOSTF, g) += 1; II(b, STREAK, g) = 0;
        }
        const int tsu = II(b, TSU, g), age = II(b, AGE, g), hs = II(b, STREAK, g);
        const bool del = tsu > b.max_lost || (age < 5 && hs == 0 && tsu > 15) || (age < 10 && hs <= 1 && tsu > 30);
        if (del) {
            II(b, ID, g) = 0; atomicAdd(&s_cnt[0], 1); atomicAdd(b.chunk_free + (size_t)s * b.nchunks + t / kChunk, 1);
            if (MODE && RI(b, MR_RESETS, g) > 0) atomicAdd(b.fcnt + s * 4 + 2, 1);     // tracking_recoveries
        }
    }
    __syncthreads();
    for (int i = warp; i < s_an; i += nwarps) analyze_slot_warp(b, g0 + s_list[i], lane);
    __syncthreads();
    // ---- rows of the candidate tracks, in list (= slot) order, after the sweep's rows ----
    if (tid == 0) s_emit_base = E1;
    __syncthreads();
    int long_term = 0;
    float* rows = fr.out_rows + (size_t)s * fr.out_cap * B2_TRACK_COLS;
    const size_t o0 = (size_t)s * fr.out_cap;
    for (int base = 0; base < T; base += kResolveThreads) {
        const int i = base + tid;
        int emit = 0, t = 0, g = 0;
        if (i < T) {
            t = cslot[i]; g = g0 + t;
            if (II(b, ID, g) != 0)     // mode 1 reports every live track (motion_compensated_multi_tracker.py:231-238)
                emit = (MODE || II(b, STREAK, g) >= b.min_hits || frame <= b.min_hits || II(b, ISLOST, g)) ? 1 : 0;   // multi_target_tracker.py:117-126
        }
        int total;
        const int off = block_exclusive_scan(emit, s_warp, &total);
        const int ebase = s_emit_base;
        if (emit) {
            const int pos = ebase + off;
            const bool fits = pos < fr.out_cap;
            emit_slot(b, g, fits ? rows + (size_t)pos * B2_TRACK_COLS : nullptr, fits && fr.out_traj ? fr.out_traj + (o0 + pos) * kTraj * 2 : nullptr,
                      fits && fr.out_traj_len ? fr.out_traj_len + o0 + pos : nullptr, t, &long_term);
            if (MODE && fits && fr.out_extra)
                reinterpret_cast<float4*>(fr.out_extra)[o0 + pos] =
                    make_float4(__int_as_float(RI(b, MR_RESETS, g)), __int_as_float(II(b, AGE, g) - RI(b, MR_LASTRESET, g)), RF(b, MR_MCONS, g), 0.f);
        }
        __syncthreads();
        if (tid == 0) s_emit_base = ebase + total;
        __syncthreads();
    }

    // ---- new tracks for unmatched detections, ascending detection index -> ascending ids; the k-th new track takes the k-th
    //      free slot of the stream ----
    int n_new = 0;
    for (int base = 0; base < D; base += kResolveThreads) {
        const int d = base + tid;
        const int um = (d < D && s_dmatch[d] < 0) ? 1 : 0;
        int total;
        const int off = block_exclusive_scan(um, s_warp, &total);
        if (um) s_list[n_new + off] = d;
        n_new += total;
    }
    __syncthreads();
    int created = 0;
    if (n_new > 0) {
        const bool emit_new = MODE || (1 >= b.min_hits) || (frame <= b.min_hits);     // hit_streak = 1
        int32_t* cfree = b.chunk_free + (size_t)s * b.nchunks;
        for (int base = 0; base < b.C && created < n_new; base += kResolveThreads) {
            // chunks without a free slot (the common case in a full bank) are skipped without touching the slots
            const int c0 = base / kChunk;
            int any = 0;
            for (int k = 0; k < kResolveThreads / kChunk; ++k) if (c0 + k < b.nchunks) any += cfree[c0 + k];
            if (!any) continue;
            const int t = base + tid, g = g0 + t;
            const int is_free = (t < b.C && II(b, ID, g) == 0) ? 1 : 0;
            int total;
            const int off = block_exclusive_scan(is_free, s_warp, &total);
            const int rank = created + off;
            const int ebase = s_emit_base;
            const int take = min(total, n_new - created);
            if (is_free && rank < n_new) {
                init_slot(b, g, s_det[s_list[rank]], id0 + rank);
                if (MODE) mr_init_slot(b, g, s_det[s_list[rank]]);
                atomicSub(b.chunk_free + (size_t)s * b.nchunks + t / kChunk, 1);     // the sweep skips chunks it believes empty
                if (emit_new) {
                    const int pos = ebase + off;
                    const bool fits = pos < fr.out_cap;
                    emit_slot(b, g, fits ? rows + (size_t)pos * B2_TRACK_COLS : nullptr, fits && fr.out_traj ? fr.out_traj + (o0 + pos) * kTraj * 2 : nullptr,
                              fits && fr.out_traj_len ? fr.out_traj_len + o0 + pos : nullptr, t, &long_term);
                    if (MODE && fits && fr.out_extra)
                        reinterpret_cast<float4*>(fr.out_extra)[o0 + pos] = make_float4(__int_as_float(0), __int_as_float(999), 0.f, 0.f);
                }
            }
            created += take;
            __syncthreads();
            if (tid == 0 && emit_new) s_emit_base = ebase + take;
            __syncthreads();
        }
    }
    if (long_term) atomicAdd(&s_cnt[1], long_term);
    __syncthreads();

    // ---- stats (enhanced_multi_target_tracker.py:32-38), counters ----
    if (tid == 0) {
        int32_t* fc = b.fcnt + s * 4;
        long long* st = b.stats + (size_t)s * 8;
        const int terminated = fc0 + s_cnt[0], lt = fc1 + s_cnt[1];
        st[0] = st_in[0] + created; st[1] = st_in[1] + terminated; st[2] = st_in[2] + created - terminated; st[3] = st_in[3] + lt;
        st[4] = st_in[4] + s_cnt[2]; st[5] = st_in[5] + n_new - created; st[6] = st_in[6] + s_cnt[3]; st[7] = st_in[7] + fc[2];
        fc[0] = 0; fc[1] = 0; fc[2] = 0;
        // the reference numbers every unmatched detection; ids keep advancing even if the bank overflowed
        b.next_id[s] = id0 + n_new;
        b.frame_count[s] = frame;
        fr.out_counts[s] = s_emit_base;
    }
}

__global__ void export_kernel(const Bank b, int s, float* x, float* P, int32_t* meta, int32_t* n_out) {
    // single thread block, slot order (the host orders by id)
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < b.C; t += blockDim.x) {
        const int g = s * b.C + t;
        if (II(b, ID, g) == 0) continue;
        const int k = atomicAdd(&cnt, 1);
        for (int j = 0; j < 8; ++j) x[k * 8 + j] = FF(b, X0 + j, g);
        float* Pk = P + (size_t)k * 64;
        for (int j = 0; j < 64; ++j) Pk[j] = 0.f;
        for (int j = 0; j < 2; ++j) {     // x,y then w,h
            Pk[j * 8 + j] = FF(b, PPX, g); Pk[j * 8 + j + 4] = FF(b, PPV, g); Pk[(j + 4) * 8 + j] = FF(b, PPV, g); Pk[(j + 4) * 8 + j + 4] = FF(b, PVV, g);
            const int q = j + 2;
            Pk[q * 8 + q] = FF(b, PSX, g); Pk[q * 8 + q + 4] = FF(b, PSV, g); Pk[(q + 4) * 8 + q] = FF(b, PSV, g); Pk[(q + 4) * 8 + q + 4] = FF(b, PSVV, g);
        }
        int32_t* mk = meta + (size_t)k * 8;
        mk[0] = II(b, ID, g); mk[1] = II(b, AGE, g); mk[2] = II(b, HITS, g); mk[3] = II(b, STREAK, g);
        mk[4] = II(b, TSU, g); mk[5] = II(b, LOSTF, g); mk[6] = II(b, ISLOST, g); mk[7] = II(b, NVEL, g);
    }
    __syncthreads();
    if (threadIdx.x == 0) *n_out = cnt;
}

__global__ void export_motion_kernel(const Bank b, int s, float* out, int32_t* n_out) {
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < b.C; t += blockDim.x) {
        const int g = s * b.C + t;
        if (II(b, ID, g) == 0) continue;
        float* o = out + (size_t)atomicAdd(&cnt, 1) * 8;
        o[0] = __int_as_float(II(b, ID, g));
        for (int j = 0; j < 6; ++j) o[1 + j] = FF(b, VAVGX + j, g);
        o[7] = __int_as_float(II(b, NVEL, g));
    }
    __syncthreads();
    if (threadIdx.x == 0) *n_out = cnt;
}

__global__ void export_reset_kernel(const Bank b, int s, float* out, int32_t* n_out) {
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < b.C; t += blockDim.x) {
        const int g = s * b.C + t;
        if (II(b, ID, g) == 0) continue;
        float* o = out + (size_t)atomicAdd(&cnt, 1) * 8;
        o[0] = __int_as_float(II(b, ID, g)); o[1] = __int_as_float(RI(b, MR_RESETS, g)); o[2] = __int_as_float(RI(b, MR_LASTRESET, g));
        o[3] = RF(b, MR_MCONS, g); o[4] = __int_as_float(RI(b, MR_PHLEN, g)); o[5] = __int_as_float(RI(b, MR_MSLEN, g));
        o[6] = __int_as_float(RI(b, MR_BBLEN, g)); o[7] = 0.f;
    }
    __syncthreads();
    if (threadIdx.x == 0) *n_out = cnt;
}

// bank regrid for b2_tracker_grow: rows of a field-major [rows][S*C] array move to [rows][S*C2]
__global__ void regrid_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, int rows, int S, int C, int C2) {
    const size_t n = (size_t)rows * S * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / ((size_t)S * C), rem = i % ((size_t)S * C);
        const size_t s = rem / C, t = rem % C;
        dst[(r * S + s) * C2 + t] = src[i];
    }
}
__global__ void fill_i32(int32_t* p, int n, int v) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

// b2_tracker_reset_streams: every word a flagged stream owns in the arena -- its slots of each [field][N] plane, its candidate
// lists, sweep scratch and pairs, counters and stats -- set to what b2_tracker_reset leaves (0, next_id = 1).
__device__ __forceinline__ uint32_t* stream_word(const Bank& b, int s, long long i) {
    const int n_planes = NFF + NIF + 2 * kVelRing + 2 * kTraj + (b.mode ? MR_NF + MR_NI : 0) + 3;
    const long long C = b.C, N = b.N;
    if (i < n_planes * C) {
        int q = (int)(i / C);
        const long long g = (long long)s * C + i % C;
        if (q < NFF) return (uint32_t*)b.f + q * N + g;
        q -= NFF;
        if (q < NIF) return (uint32_t*)b.i + q * N + g;
        q -= NIF;
        if (q < 2 * kVelRing) return (uint32_t*)b.vel + q * N + g;
        q -= 2 * kVelRing;
        if (q < 2 * kTraj) return (uint32_t*)b.traj + q * N + g;
        q -= 2 * kTraj;
        if (b.mode) {
            if (q < MR_NF) return (uint32_t*)b.mrf + q * N + g;
            q -= MR_NF;
            if (q < MR_NI) return (uint32_t*)b.mri + q * N + g;
            q -= MR_NI;
        }
        return (uint32_t*)(q == 0 ? b.ctrk_slot : q == 1 ? b.cid : b.cmatch) + g;
    }
    i -= n_planes * C;
    if (i < 4 * C) return (uint32_t*)b.cbox + 4 * C * s + i;
    i -= 4 * C;
    if (i < 4ll * b.pair_cap) return (uint32_t*)b.pairs + 4ll * b.pair_cap * s + i;
    i -= 4ll * b.pair_cap;
    if (i < 2ll * b.nchunks) return (uint32_t*)b.agg + 2ll * b.nchunks * s + i;
    i -= 2ll * b.nchunks;
    if (i < b.nchunks) return (uint32_t*)b.chunk_free + (long long)b.nchunks * s + i;
    i -= b.nchunks;
    if (i < 4) return (uint32_t*)b.fcnt + 4 * s + i;
    i -= 4;
    if (i < 16) return (uint32_t*)b.stats + 16 * s + i;
    i -= 16;
    return i == 0 ? (uint32_t*)b.frame_count + s : i == 1 ? (uint32_t*)b.next_id + s : nullptr;
}

long long stream_words(const Bank& b) {
    const int n_planes = NFF + NIF + 2 * kVelRing + 2 * kTraj + (b.mode ? MR_NF + MR_NI : 0) + 3;
    return (long long)(n_planes + 4) * b.C + 4ll * b.pair_cap + 3ll * b.nchunks + 4 + 16 + 2;
}

__global__ void __launch_bounds__(256) reset_streams_kernel(const Bank b, const int32_t* __restrict__ flags, long long n_words) {
    const int s = blockIdx.y;
    if (!flags[s]) return;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_words; i += (long long)gridDim.x * blockDim.x) {
        uint32_t* w = stream_word(b, s, i);
        *w = i == n_words - 1 ? 1u : 0u;     // the last word is next_id
    }
}

struct Layout { size_t f, i, v, t, rf, ri, agg, cf, fc, tk, cs, cb, ci, cm, pr, ni, fcn, st, total; };

Layout bank_layout(int S, int C, int max_dets, int nchunks, int pair_cap, int mode) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t N = (size_t)S * C;
    Layout L;
    size_t off = 0;
    L.f = off; off += up(N * NFF * 4);
    L.i = off; off += up(N * NIF * 4);
    L.v = off; off += up(N * kVelRing * 2 * 4);
    L.t = off; off += up(N * kTraj * 2 * 4);
    L.rf = off; off += mode ? up(N * MR_NF * 4) : 0;
    L.ri = off; off += mode ? up(N * MR_NI * 4) : 0;
    L.agg = off; off += up((size_t)S * nchunks * 8);
    L.cf = off; off += up((size_t)S * nchunks * 4);
    L.fc = off; off += up((size_t)S * 4 * 4);
    L.tk = off; off += up(4);
    L.cs = off; off += up(N * 4);
    L.cb = off; off += up(N * 16);
    L.ci = off; off += up(N * 4);
    L.cm = off; off += up(N * 4);
    L.pr = off; off += up((size_t)S * pair_cap * 16);
    L.ni = off; off += up((size_t)S * 4);
    L.fcn = off; off += up((size_t)S * 4);
    L.st = off; off += up((size_t)S * 8 * 8);
    L.total = off;
    (void)max_dets;
    return L;
}

void bank_bind(Bank& b, char* a, const Layout& L) {
    b.f = (float*)(a + L.f); b.i = (int32_t*)(a + L.i); b.vel = (float*)(a + L.v); b.traj = (float*)(a + L.t);
    b.mrf = (float*)(a + L.rf); b.mri = (int32_t*)(a + L.ri);
    b.agg = (unsigned long long*)(a + L.agg); b.chunk_free = (int32_t*)(a + L.cf); b.fcnt = (int32_t*)(a + L.fc);
    b.ticket = (unsigned int*)(a + L.tk); b.ctrk_slot = (int32_t*)(a + L.cs); b.cbox = (float4*)(a + L.cb);
    b.cid = (int32_t*)(a + L.ci); b.cmatch = (int32_t*)(a + L.cm); b.pairs = (uint4*)(a + L.pr);
    b.next_id = (int32_t*)(a + L.ni); b.frame_count = (int32_t*)(a + L.fcn); b.stats = (long long*)(a + L.st);
}

}  // namespace

struct b2_tracker { b2_tracker_impl impl; };

extern "C" int b2_tracker_create(int n_streams, int capacity, int max_dets, int max_lost_frames, int min_hits,
                                 float iou_threshold, b2_tracker_t** out) {
    return b2_tracker_create_ex(n_streams, capacity, max_dets, max_lost_frames, min_hits, iou_threshold, 0, out);
}

extern "C" int b2_tracker_create_ex(int n_streams, int capacity, int max_dets, int max_lost_frames, int min_hits,
                                    float iou_threshold, int mode, b2_tracker_t** out) {
    B2_REQUIRE(out, "tracker_create: out is null");
    B2_REQUIRE(mode == 0 || mode == 1, "tracker_create: mode must be 0 (EnhancedMultiTargetTracker) or 1 (MotionCompensatedMultiTracker)");
    B2_REQUIRE(n_streams >= 1 && capacity >= 1 && capacity <= 65535 && max_dets >= 1 && max_dets <= kMaxDetsSmem,
               "tracker_create: need n_streams>=1, 1<=capacity<=65535, 1<=max_dets<=%d", kMaxDetsSmem);
    B2_REQUIRE((long long)n_streams * capacity < (1ll << 31), "tracker_create: n_streams*capacity must be below 2^31");
    b2_tracker* t = new (std::nothrow) b2_tracker();
    if (!t) { b2_set_error("out of host memory"); return B2_ERR_STATE; }
    Bank& b = t->impl.b;
    b.S = n_streams; b.C = capacity; b.N = n_streams * capacity; b.max_dets = max_dets;
    b.nchunks = b2_ceil_div(capacity, kChunk);
    b.pair_cap = 16 * max_dets < 1024 ? 1024 : 16 * max_dets;
    b.max_lost = max_lost_frames; b.min_hits = min_hits; b.iou_thr = iou_threshold; b.mode = mode;
    const Layout L = bank_layout(b.S, b.C, max_dets, b.nchunks, b.pair_cap, mode);
    cudaError_t e = cudaMalloc(&t->impl.arena, L.total);
    if (e != cudaSuccess) { b2_set_error("tracker_create: cudaMalloc(%zu) failed: %s", L.total, cudaGetErrorString(e)); delete t; return B2_ERR_CUDA; }
    t->impl.arena_bytes = L.total;
    bank_bind(b, (char*)t->impl.arena, L);
    *out = t;
    return b2_tracker_reset(t, nullptr);
}

extern "C" int b2_tracker_destroy(b2_tracker_t* t) {
    if (!t) return B2_OK;
    cudaFree(t->impl.arena);
    delete t;
    return B2_OK;
}

extern "C" int b2_tracker_reset(b2_tracker_t* t, void* stream) {
    B2_REQUIRE(t, "tracker_reset: null handle");
    cudaStream_t st = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(t->impl.arena, 0, t->impl.arena_bytes, st));
    fill_i32<<<b2_ceil_div(t->impl.b.S, 256), 256, 0, st>>>(t->impl.b.next_id, t->impl.b.S, 1);   // next_track_id = 1 (:30)
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_tracker_reset_streams(b2_tracker_t* t, const int32_t* flags_dev, void* stream) {
    B2_REQUIRE(t && flags_dev, "tracker_reset_streams: null argument");
    const Bank& b = t->impl.b;
    const long long n = stream_words(b);
    const int blocks = (int)std::min<long long>(b2_ceil_div((int)std::min<long long>(n, 1ll << 30), 256), 64);
    reset_streams_kernel<<<dim3(blocks, b.S), 256, 0, (cudaStream_t)stream>>>(b, flags_dev, n);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_tracker_capacity(b2_tracker_t* t) { return t ? t->impl.b.C : 0; }

extern "C" int b2_tracker_grow(b2_tracker_t* t, int new_capacity, void* stream) {
    B2_REQUIRE(t, "tracker_grow: null handle");
    Bank& b = t->impl.b;
    B2_REQUIRE(new_capacity > b.C && new_capacity <= 65535, "tracker_grow: new capacity %d must be in (%d, 65535]", new_capacity, b.C);
    B2_REQUIRE((long long)b.S * new_capacity < (1ll << 31), "tracker_grow: n_streams*capacity must be below 2^31");
    cudaStream_t st = (cudaStream_t)stream;
    Bank nb = b;
    nb.C = new_capacity; nb.N = b.S * new_capacity; nb.nchunks = b2_ceil_div(new_capacity, kChunk);
    const Layout L = bank_layout(nb.S, nb.C, nb.max_dets, nb.nchunks, nb.pair_cap, nb.mode);
    void* arena = nullptr;
    cudaError_t e = cudaMalloc(&arena, L.total);
    if (e != cudaSuccess) { b2_set_error("tracker_grow: cudaMalloc(%zu) failed: %s", L.total, cudaGetErrorString(e)); return B2_ERR_CUDA; }
    bank_bind(nb, (char*)arena, L);
    B2_CUDA(cudaMemsetAsync(arena, 0, L.total, st));
    const int grid = b2_num_sms() * 8;
    regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.f, (uint32_t*)nb.f, NFF, b.S, b.C, nb.C);
    regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.i, (uint32_t*)nb.i, NIF, b.S, b.C, nb.C);
    regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.vel, (uint32_t*)nb.vel, kVelRing * 2, b.S, b.C, nb.C);
    regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.traj, (uint32_t*)nb.traj, kTraj * 2, b.S, b.C, nb.C);
    if (b.mode) {
        regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.mrf, (uint32_t*)nb.mrf, MR_NF, b.S, b.C, nb.C);
        regrid_kernel<<<grid, 256, 0, st>>>((const uint32_t*)b.mri, (uint32_t*)nb.mri, MR_NI, b.S, b.C, nb.C);
    }
    B2_CUDA(cudaMemcpyAsync(nb.next_id, b.next_id, (size_t)b.S * 4, cudaMemcpyDeviceToDevice, st));
    B2_CUDA(cudaMemcpyAsync(nb.frame_count, b.frame_count, (size_t)b.S * 4, cudaMemcpyDeviceToDevice, st));
    B2_CUDA(cudaMemcpyAsync(nb.stats, b.stats, (size_t)b.S * 64, cudaMemcpyDeviceToDevice, st));
    B2_CUDA(cudaGetLastError());
    B2_CUDA(cudaStreamSynchronize(st));
    b2_count_launch(4);
    cudaFree(t->impl.arena);
    t->impl.arena = arena; t->impl.arena_bytes = L.total;
    b = nb;
    return B2_OK;
}

extern "C" int b2_tracker_bank_predict(b2_tracker_t* t, void* stream) {
    B2_REQUIRE(t, "tracker: null handle");
    const Bank& b = t->impl.b;
    cudaStream_t st = (cudaStream_t)stream;
    if (b.N % 4 == 0) bank_predict4_kernel<<<b2_ceil_div(b.N / 4, 256), 256, 0, st>>>(b);
    else bank_predict_kernel<<<b2_ceil_div(b.N, 256), 256, 0, st>>>(b);
    B2_CUDA(cudaGetLastError());
    b2_count_launch(1);
    return B2_OK;
}

extern "C" int b2_tracker_update(b2_tracker_t* t, const float* dets, int det_cols, const int32_t* det_counts,
                                 float* out_rows, int32_t* out_counts, float* out_traj, int32_t* out_traj_len, int out_cap, void* stream) {
    return b2_tracker_update_ex(t, dets, det_cols, det_counts, out_rows, out_counts, out_traj, out_traj_len, nullptr, out_cap, stream);
}

extern "C" int b2_tracker_update_ex(b2_tracker_t* t, const float* dets, int det_cols, const int32_t* det_counts,
                                    float* out_rows, int32_t* out_counts, float* out_traj, int32_t* out_traj_len, float* out_extra,
                                    int out_cap, void* stream) {
    B2_REQUIRE(t && dets && det_counts && out_rows && out_counts, "tracker_update: null pointer");
    B2_REQUIRE(!out_extra || ((uintptr_t)out_extra % 16 == 0 && t->impl.b.mode == 1), "tracker_update: out_extra needs a mode-1 bank and 16-byte alignment");
    B2_REQUIRE(out_cap >= 1, "tracker_update: out_cap must be >= 1");
    B2_REQUIRE(det_cols >= 4, "tracker_update: det_cols must be >= 4");
    B2_REQUIRE((out_traj == nullptr) == (out_traj_len == nullptr), "tracker_update: out_traj and out_traj_len go together");
    const Bank& b = t->impl.b;
    cudaStream_t st = (cudaStream_t)stream;
    const Frame fr{dets, det_cols, det_counts, out_rows, out_counts, out_traj, out_traj_len, out_cap, out_extra};
    // resolve is launched as a programmatic dependent of the sweep: its blocks are placed while the sweep's last blocks run and wait
    // (griddepcontrol.wait) for the sweep's completion before they read anything it wrote -- the launch latency and the copy of the
    // detections come off the frame's critical path (B2_TRK_PDL=0: plain stream order)
    static const bool pdl = [] { const char* v = getenv("B2_TRK_PDL"); return !(v && atoi(v) == 0); }();
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)b.S); cfg.blockDim = dim3((unsigned)kResolveThreads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    if (b.mode) {
        sweep_kernel<1><<<b.S * b.nchunks, kChunk, (size_t)b.max_dets * sizeof(float4), st>>>(b, fr);
        B2_CUDA(cudaLaunchKernelEx(&cfg, resolve_kernel<1>, b, fr));
    } else {
        sweep_kernel<0><<<b.S * b.nchunks, kChunk, (size_t)b.max_dets * sizeof(float4), st>>>(b, fr);
        B2_CUDA(cudaLaunchKernelEx(&cfg, resolve_kernel<0>, b, fr));
    }
    B2_CUDA(cudaGetLastError());
    b2_count_launch(2);
    return B2_OK;
}

extern "C" int b2_tracker_export(b2_tracker_t* t, int stream_idx, float* x_host, float* P_host, int32_t* meta_host,
                                 int32_t* n_tracks_host, long long* stats_host) {
    B2_REQUIRE(t && stream_idx >= 0 && stream_idx < t->impl.b.S, "tracker_export: bad stream index");
    const Bank& b = t->impl.b;
    B2_CUDA(cudaDeviceSynchronize());
    if (x_host || P_host || meta_host || n_tracks_host) {
        float *dx = nullptr, *dP = nullptr; int32_t *dm = nullptr, *dn = nullptr;
        B2_CUDA(cudaMalloc(&dx, (size_t)b.C * 8 * 4)); B2_CUDA(cudaMalloc(&dP, (size_t)b.C * 64 * 4));
        B2_CUDA(cudaMalloc(&dm, (size_t)b.C * 8 * 4)); B2_CUDA(cudaMalloc(&dn, 4));
        export_kernel<<<1, 256>>>(b, stream_idx, dx, dP, dm, dn);
        b2_count_launch(1);
        int n = 0;
        cudaError_t e = cudaMemcpy(&n, dn, 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && x_host) e = cudaMemcpy(x_host, dx, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && P_host) e = cudaMemcpy(P_host, dP, (size_t)n * 64 * 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && meta_host) e = cudaMemcpy(meta_host, dm, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost);
        cudaFree(dx); cudaFree(dP); cudaFree(dm); cudaFree(dn);
        B2_CUDA(e);
        if (n_tracks_host) *n_tracks_host = n;
    }
    if (stats_host) {
        long long st[8];
        B2_CUDA(cudaMemcpy(st, b.stats + (size_t)stream_idx * 8, sizeof(st), cudaMemcpyDeviceToHost));
        int32_t fc = 0, nid = 0;
        B2_CUDA(cudaMemcpy(&fc, b.frame_count + stream_idx, 4, cudaMemcpyDeviceToHost));
        B2_CUDA(cudaMemcpy(&nid, b.next_id + stream_idx, 4, cudaMemcpyDeviceToHost));
        for (int k = 0; k < 5; ++k) stats_host[k] = st[k];
        stats_host[5] = fc; stats_host[6] = nid; stats_host[7] = st[5];
        if (b.mode) { stats_host[3] = st[6]; stats_host[4] = st[7]; }       // mode 1: individual_resets, tracking_recoveries
    }
    return B2_OK;
}

extern "C" int b2_tracker_export_motion(b2_tracker_t* t, int stream_idx, float* motion_host, int32_t* n_tracks_host) {
    B2_REQUIRE(t && stream_idx >= 0 && stream_idx < t->impl.b.S && motion_host && n_tracks_host, "tracker_export_motion: bad argument");
    const Bank& b = t->impl.b;
    B2_CUDA(cudaDeviceSynchronize());
    float* dm = nullptr; int32_t* dn = nullptr;
    B2_CUDA(cudaMalloc(&dm, (size_t)b.C * 8 * 4)); B2_CUDA(cudaMalloc(&dn, 4));
    export_motion_kernel<<<1, 256>>>(b, stream_idx, dm, dn);
    b2_count_launch(1);
    int n = 0;
    cudaError_t e = cudaMemcpy(&n, dn, 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(motion_host, dm, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost);
    cudaFree(dm); cudaFree(dn);
    B2_CUDA(e);
    *n_tracks_host = n;
    return B2_OK;
}

extern "C" int b2_tracker_export_reset(b2_tracker_t* t, int stream_idx, float* reset_host, int32_t* n_tracks_host) {
    B2_REQUIRE(t && stream_idx >= 0 && stream_idx < t->impl.b.S && reset_host && n_tracks_host && t->impl.b.mode == 1, "tracker_export_reset: bad argument (mode-1 bank required)");
    const Bank& b = t->impl.b;
    B2_CUDA(cudaDeviceSynchronize());
    float* dm = nullptr; int32_t* dn = nullptr;
    B2_CUDA(cudaMalloc(&dm, (size_t)b.C * 8 * 4)); B2_CUDA(cudaMalloc(&dn, 4));
    export_reset_kernel<<<1, 256>>>(b, stream_idx, dm, dn);
    b2_count_launch(1);
    int n = 0;
    cudaError_t e = cudaMemcpy(&n, dn, 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(reset_host, dm, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost);
    cudaFree(dm); cudaFree(dn);
    B2_CUDA(e);
    *n_tracks_host = n;
    return B2_OK;
}

extern "C" int b2_tracker_stats(b2_tracker_t* t, long long* stats_dev_out, void* stream) {
    // device-to-device snapshot of the [S][8] counters (created, terminated, active, long_term, recoveries, dropped, -, -):
    // lets a pipeline download them with its rows instead of synchronising on b2_tracker_export
    B2_REQUIRE(t && stats_dev_out, "tracker_stats: null pointer");
    B2_CUDA(cudaMemcpyAsync(stats_dev_out, t->impl.b.stats, (size_t)t->impl.b.S * 64, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return B2_OK;
}

extern "C" int b2_tracker_bytes_per_track(int* predict_bytes, int* update_bytes) {
    // sweep, per coasting (unmatched, reported) track: read id x[8] P[6] motion[6] age hits tsu lostf islost tlen thead
    // (28 words), write x[4] P[6] age tsu tlen thead streak lostf islost + 2 trajectory floats + the 20-word row (39 words)
    if (predict_bytes) *predict_bytes = (28 + 39) * 4;
    // update (matched): the candidate lists (slot, box, id, pair 16 B), the Kalman update of x[8] P[6], counters, ring and
    // trajectory pushes, the ring re-scan of the motion analysis (up to 100 floats) and the row
    if (update_bytes) *update_bytes = (6 + 4) * 4 + (14 + 14 + 8 + 4) * 4 + 100 * 4 + 6 * 4 + 20 * 4;
    return B2_OK;
}

extern "C" int b2_tracker_seed(b2_tracker_t* t, const float* boxes, const int32_t* counts, int max_rows, void* stream) {
    // Seeding == one update on an empty bank with min-hits semantics untouched: every row creates a track.
    (void)t; (void)boxes; (void)counts; (void)max_rows; (void)stream;
    b2_set_error("b2_tracker_seed: use b2_tracker_update on a reset bank (every detection creates a track)");
    return B2_ERR_UNSUPPORTED;
}
