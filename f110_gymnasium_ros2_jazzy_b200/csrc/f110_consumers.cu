// f110_consumers.cu -- device-side forms of the consumers that sit directly around the env in the reference's
// training loop (SURVEY 8f), so a rollout never leaves the GPU.  Paths are relative to /root/reference/.
//
//   gap_follow_kernel : rl_training/utils/gap_follow.py:3-58, the rule-based opponent train_ddpg.py:168 drives
//                       from info["scans"][1].  One CTA per scan; float32 arithmetic in numpy's order, so the
//                       chosen beam index -- and with it (steer, speed) -- is identical to the reference's.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "f110_b200.h"

int f110_set_error(int code, const char* msg);   // f110_capi.cu

namespace {

constexpr int GF_WARPS = 8;     // scans per CTA (one warp each); fewer when the scans are too long for that much shared memory

// Summary of a stretch of the boolean sequence proc > threshold, in the form find_max_gap :21-38 needs: runs touching
// the stretch's ends and the FIRST longest run closed inside it (metric end - start, as the reference's max(key=...)).
// Summaries of adjacent stretches combine associatively, so a warp reduces 32 of them in five shuffles.
struct RunSummary { int start, len, all_true, prefix, suffix, best_len, best_start; };

__device__ __forceinline__ RunSummary combine_runs(const RunSummary& L, const RunSummary& R) {
    if (L.len == 0) return R;
    if (R.len == 0) return L;
    RunSummary o;
    o.start = L.start;
    o.len = L.len + R.len;
    o.all_true = L.all_true && R.all_true;
    o.prefix = L.all_true ? L.len + R.prefix : L.prefix;
    o.suffix = R.all_true ? R.len + L.suffix : R.suffix;
    o.best_len = L.best_len; o.best_start = L.best_start;
    // the run across the boundary is closed on both sides only if neither stretch is all true
    if (!L.all_true && !R.all_true && L.suffix + R.prefix > 0) {
        const int m = L.suffix + R.prefix - 1;
        if (m > o.best_len) { o.best_len = m; o.best_start = L.start + L.len - L.suffix; }
    }
    if (R.best_len > o.best_len) { o.best_len = R.best_len; o.best_start = R.best_start; }
    return o;
}

// the summary of `len` (1..32) consecutive beams starting at beam `base`, bit b of `w` = beam base + b is above the threshold
__device__ __forceinline__ RunSummary word_runs(unsigned w, int len, int base) {
    RunSummary r;
    const unsigned full = len == 32 ? 0xffffffffu : (1u << len) - 1u;
    w &= full;
    r.start = base; r.len = len; r.best_len = -1; r.best_start = 0;
    r.all_true = w == full;
    if (r.all_true) { r.prefix = len; r.suffix = len; return r; }
    r.prefix = __ffs((int)~w) - 1;                                 // ones from bit 0 up (~w != 0 here)
    r.suffix = __clz((int)~(w << (32 - len)));                     // ones from bit len - 1 down
    unsigned x = w;
    if (r.prefix > 0) x &= ~((1u << r.prefix) - 1u);
    if (r.suffix > 0) x &= (1u << (len - r.suffix)) - 1u;
    while (x) {                                                    // the runs closed inside the word, lowest first
        const int s0 = __ffs((int)x) - 1;
        const unsigned y = ~(x >> s0);
        const int run = y ? __ffs((int)y) - 1 : 32 - s0;
        if (run - 1 > r.best_len) { r.best_len = run - 1; r.best_start = base + s0; }
        x &= run + s0 >= 32 ? (1u << s0) - 1u : ~(((1u << run) - 1u) << s0);
    }
    return r;
}

__device__ __forceinline__ float lds_f32(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

// preprocess_lidar :3-12 for beam i: mean of the clipped ranges over [i - w/2, i + w/2] cut at the ends, summed in numpy's
// order: fewer than 8 float32 elements in sequence, 8 to 15 as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) over the first eight and
// the rest in sequence (np.add.reduce's pairwise sum; a window holds at most 15 beams).  `clipped` is the array's 32-bit shared-memory address (formed once: indexed as a
// C array, every access re-derived the shared window's base); W > 0 = the window size as a compile-time constant, whose
// interior beams divide by a constant.
template <int W>
__device__ __forceinline__ float window_mean(unsigned clipped, int i, int n, int window_size) {
    const int half = (W > 0 ? W : window_size) / 2;
    if (W > 0 && i >= half && i + half <= n - 1) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < 2 * (W / 2) + 1; ++k) acc += lds_f32(clipped + 4u * (unsigned)(i - half + k));
        return __fdiv_rn(acc, (float)(2 * (W / 2) + 1));
    }
    const int s = max(0, i - half), e = min(n - 1, i + half);
    float acc = 0.f;
    int k = s;
    if (W == 0 && e - s + 1 >= 8) {                             // W = 5 windows never reach 8 beams
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = lds_f32(clipped + 4u * (unsigned)(s + j));
        acc = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        k = s + 8;
    }
    for (; k <= e; ++k) acc += lds_f32(clipped + 4u * (unsigned)k);
    return __fdiv_rn(acc, (float)(e - s + 1));
}

// np.argmin's order: (v, i) comes before (bv, bi) if v is the first NaN, or neither is NaN and v is smaller, or ties earlier
__device__ __forceinline__ bool argmin_before(float v, int i, float bv, int bi) {
    const bool vn = v != v, bn = bv != bv;
    if (vn != bn) return vn;
    return (vn || v == bv) ? i < bi : v < bv;
}

// One WARP per scan, beam i = 32 k + lane in round k: every access coalesced, no barrier (round 1: a CTA per scan with five
// barriers and a 128-step serial stitch by thread 0, 67 us per 8192 scans; timing under profiles/).
template <int W>
__global__ void __launch_bounds__(GF_WARPS * 32) gap_follow_kernel(const float* __restrict__ scans, long long scan_stride, int n,
                                                                  long long num_scans, float* __restrict__ actions, long long action_stride,
                                                                  double angle_min, double angle_increment, float max_distance,
                                                                  int window_size, int bubble_radius, float threshold) {
    extern __shared__ float sm[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long scan_id = (long long)blockIdx.x * (blockDim.x >> 5) + wid;
    if (scan_id >= num_scans) return;
    const int groups = (n + 31) / 32;
    float* clipped = sm + (size_t)wid * (2 * n + groups);      // [n]
    float* proc = clipped + n;                                   // [n] the window means
    unsigned* words = reinterpret_cast<unsigned*>(proc + n);     // [groups]: bit b of word k = beam 32 k + b is above the threshold
    const float* scan = scans + (size_t)scan_id * scan_stride;

    // the scan comes from DRAM (the lidar kernel wrote it with streaming stores): seventeen loads in flight per lane -- one
    // at a time, a warp waited 34 DRAM round trips in a row and the kernel ran at a ninth of the memory's speed
    constexpr int U = 17;     // 1080 beams = two batches
    for (int base = 0; base < n; base += 32 * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + 32 * u + lane;
            v[u] = i < n ? __ldcs(scan + i) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + 32 * u + lane;
            float c = v[u] < 0.f ? 0.f : v[u];
            c = c > max_distance ? max_distance : c;
            if (i < n) clipped[i] = c;
        }
    }
    __syncwarp();
    // create_bubble :14-19: np.argmin = the first NaN if any, else the first minimum over the whole scan
    const unsigned clipped_addr = (unsigned)__cvta_generic_to_shared(clipped);
    float best_v = INFINITY;
    int best_i = 0x7fffffff;
    for (int i = lane; i < n; i += 32) {
        const float m = window_mean<W>(clipped_addr, i, n, window_size);
        proc[i] = m;
        if (argmin_before(m, i, best_v, best_i)) { best_v = m; best_i = i; }    // the lane's first NaN / minimum
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float v2 = __shfl_down_sync(0xffffffffu, best_v, o);
        const int i2 = __shfl_down_sync(0xffffffffu, best_i, o);
        if (argmin_before(v2, i2, best_v, best_i)) { best_v = v2; best_i = i2; }
    }
    int closest = __shfl_sync(0xffffffffu, best_i, 0);
    closest = closest == 0x7fffffff ? 0 : closest;
    const int b0 = max(closest - bubble_radius, 0), b1 = min(closest + bubble_radius, n - 1);
    // find_max_gap :21-38: the mask, 32 beams per word (the bubble's beams hold 0)
    for (int k = 0; k < groups; ++k) {
        const int i = 32 * k + lane;
        bool val = false;
        if (i < n) val = ((i >= b0 && i <= b1) ? 0.f : proc[i]) > threshold;      // own store: no sync needed
        const unsigned w = __ballot_sync(0xffffffffu, val);
        if (lane == 0) words[k] = w;
    }
    __syncwarp();
    // lane l summarises words [l * wc, (l + 1) * wc) in order, the warp joins the 32 summaries
    const int wc = (groups + 31) / 32;
    RunSummary r;
    r.start = 0; r.len = 0; r.all_true = 1; r.prefix = 0; r.suffix = 0; r.best_len = -1; r.best_start = 0;
    for (int j = lane * wc; j < min((lane + 1) * wc, groups); ++j)
        r = combine_runs(r, word_runs(words[j], min(32, n - 32 * j), 32 * j));
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        RunSummary t;
        t.start = __shfl_down_sync(0xffffffffu, r.start, o);
        t.len = __shfl_down_sync(0xffffffffu, r.len, o);
        t.all_true = __shfl_down_sync(0xffffffffu, r.all_true, o);
        t.prefix = __shfl_down_sync(0xffffffffu, r.prefix, o);
        t.suffix = __shfl_down_sync(0xffffffffu, r.suffix, o);
        t.best_len = __shfl_down_sync(0xffffffffu, r.best_len, o);
        t.best_start = __shfl_down_sync(0xffffffffu, r.best_start, o);
        // lane l holds [l, l + o) and receives [l + o, l + 2 o): only lanes that are multiples of 2 o matter from here on
        if ((lane & (2 * o - 1)) == 0) r = combine_runs(r, t);
    }
    if (lane == 0) {
        // the runs of the whole scan in order: the one touching beam 0, the first longest closed one, the one touching
        // beam n - 1; max(key = end - start) keeps the first of equals
        int best_s = 0, best_e = n - 1, best_len = -1;
        if (r.all_true) { best_len = n - 1; }
        else {
            if (r.prefix > 0) { best_len = r.prefix - 1; best_s = 0; best_e = r.prefix - 1; }
            if (r.best_len > best_len) { best_len = r.best_len; best_s = r.best_start; best_e = r.best_start + r.best_len; }
            if (r.suffix > 0 && r.suffix - 1 > best_len) { best_len = r.suffix - 1; best_s = n - r.suffix; best_e = n - 1; }
        }
        const int best = (best_s + best_e) / 2;                                   // find_best_point :40-41
        const double steering = angle_min + best * angle_increment;               // :49
        const double d10 = 10 * (3.141592653589793 / 180.0), d20 = 20 * (3.141592653589793 / 180.0);
        const double speed = fabs(steering) < d10 ? 2.5 : (fabs(steering) < d20 ? 2.0 : 1.5);
        float* out = actions + (size_t)scan_id * action_stride;
        out[0] = (float)steering;
        out[1] = (float)speed;
    }
}

}  // namespace

extern "C" int f110_gap_follow(const float* scans, int64_t num_scans, int64_t scan_stride, int32_t num_beams,
                               float* actions, int64_t action_stride, double angle_min, double angle_increment,
                               float max_distance, int32_t window_size, int32_t bubble_radius, float threshold, void* stream) {
    if (!scans || !actions || num_scans < 0 || num_beams < 1 || num_beams > 8192 || window_size < 1 || window_size > 15 ||
        bubble_radius < 0)
        return f110_set_error(F110_ERR_INVALID, "f110_gap_follow: need non-null buffers, 1 <= num_beams <= 8192, 1 <= window_size <= 15, "
                                                "bubble_radius >= 0");
    if (num_scans == 0) return F110_OK;
    if (bubble_radius > num_beams) bubble_radius = num_beams;      // the same bubble (the whole scan), and closest + radius cannot overflow
    const size_t per_warp = sizeof(float) * (2 * (size_t)num_beams + (size_t)(num_beams + 31) / 32);
    int warps = (int)((48 * 1024) / per_warp);          // stay within the 48 KB that need no opt-in where a scan allows it
    warps = warps > GF_WARPS ? GF_WARPS : (warps < 1 ? 1 : warps);
    const size_t gf_smem = per_warp * warps;
    void (*kernel)(const float*, long long, int, long long, float*, long long, double, double, float, int, int, float) =
        window_size == 5 ? gap_follow_kernel<5> : gap_follow_kernel<0>;
    if (gf_smem > 48 * 1024) {   // one scan of more than 6 000 beams: the kernel has to opt in to its dynamic shared memory
        static size_t opted_in[64][2] = {};      // per device (the attribute is a per-device property of the function)
        int dev = 0;
        cudaGetDevice(&dev);
        size_t& have = opted_in[dev & 63][window_size == 5 ? 0 : 1];
        if (gf_smem > have) {
            if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gf_smem) != cudaSuccess) {
                cudaGetLastError();
                return f110_set_error(F110_ERR_CUDA, "f110_gap_follow: cannot reserve the shared memory these scans need");
            }
            have = gf_smem;
        }
    }
    kernel<<<(unsigned)((num_scans + warps - 1) / warps), warps * 32, gf_smem, (cudaStream_t)stream>>>(
        scans, scan_stride, num_beams, num_scans, actions, action_stride, angle_min, angle_increment, max_distance, window_size,
        bubble_radius, threshold);
    return cudaPeekAtLastError() == cudaSuccess ? F110_OK : f110_set_error(F110_ERR_CUDA, "f110_gap_follow: kernel launch failed");
}

// =====================================================================================================================
//   shaped_reward_kernel : rl_training/utils/rewards.py:185-355 (CenterlineSafetyProgressReward, with _Prog :86-180 and
//                          parse_flat_obs :11-39) over rl_training/utils/track_progress.py (CenterlineProgress.project_xy
//                          :58-95, delta_s :97-104) -- the reward train_ddpg.py:179 computes from the flat observation.
//                          One CTA per env: brute-force 5-nearest segment midpoints for both cars (the reference's
//                          cKDTree.query(k=5)), radix select for numpy's float32 quantile of the lidar, then one thread runs
//                          the per-env progress state machine.  fp64 in the reference's order; results agree to ~1e-15.
// =====================================================================================================================
struct F110Reward {
    F110RewardConfig cfg;
    int n;
    double L;
    double *xy, *s, *tan, *nrm, *mid, *wR, *wL;   // device
    double* blk;                                  // device [nblk][3]: centre x, y and radius of 64 consecutive midpoints
    int nblk;
    void* state;                                  // device RewardState[N]
    int device;
};

namespace {

struct RewardState {
    int has_s_prev[2], has_p_prev[2];
    double s_prev[2], p_prev[2][2], cum[2], ema_abs, t_last[2], flip, buf_sum;
    int buf_n, steps;
};

struct RewardView {
    F110RewardConfig p;
    int n;
    double L;
    const double *xy, *s, *tan, *nrm, *mid, *wR, *wL, *blk;
    int nblk;
    RewardState* st;
};

constexpr int RW_THREADS = 128;
constexpr int KNN = 5;
constexpr int MID_BLOCK = 64;   // midpoints per pruning block

struct Cand { double d2; int idx; };
__device__ __forceinline__ bool cand_less(const Cand& a, const Cand& b) { return a.d2 < b.d2 || (a.d2 == b.d2 && a.idx < b.idx); }

// sorted insertion into a register-resident top-5, ordered by (distance, index).  A midpoint at an infinite (or NaN)
// distance is no neighbour, as in cKDTree.query and the oracle: a car that far off falls back to the nearest node.
__device__ __forceinline__ void topk_insert(Cand (&best)[KNN], double d2, int idx) {
    if (!(d2 < INFINITY)) return;
    Cand c;
    c.d2 = d2; c.idx = idx;
    if (!cand_less(c, best[KNN - 1])) return;
    best[KNN - 1] = c;
#pragma unroll
    for (int j = KNN - 1; j > 0; --j) {
        if (cand_less(best[j], best[j - 1])) { const Cand t = best[j]; best[j] = best[j - 1]; best[j - 1] = t; }
    }
}

// The KNN smallest (d2, idx) over the whole CTA.  Each warp pops its KNN best with shuffles (no barrier), the four
// warps' lists meet in shared memory, thread 0 merges them.  `best` is this thread's sorted private list.
__device__ void block_topk(const Cand (&best)[KNN], Cand* s_cand /*[4][KNN]*/, int* s_out /*[KNN]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int head = 0;
    for (int round = 0; round < KNN; ++round) {
        Cand c;
        c.d2 = INFINITY; c.idx = 0x7fffffff;
#pragma unroll
        for (int k = 0; k < KNN; ++k) if (k == head) c = best[k];
        // warp-wide lexicographic min of (d2, idx) with three REDUX: d2 >= 0, so its bit pattern orders like the value
        const unsigned long long bits = (unsigned long long)__double_as_longlong(c.d2);
        const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
        const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
        const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xFFFFFFFFu);
        const unsigned midx = __reduce_min_sync(0xffffffffu, (hi == mhi && lo == mlo) ? (unsigned)c.idx : 0x7FFFFFFFu);
        Cand w;
        w.d2 = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
        w.idx = (int)midx;
        if (w.idx == c.idx && c.idx != 0x7fffffff) ++head;      // a midpoint index belongs to exactly one thread
        if (lane == 0) s_cand[warp * KNN + round] = w;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int h[RW_THREADS / 32] = { 0, 0, 0, 0 };
        for (int round = 0; round < KNN; ++round) {
            int bw = -1;
            Cand bc;
            bc.d2 = INFINITY; bc.idx = 0x7fffffff;
            for (int w = 0; w < RW_THREADS / 32; ++w) {
                if (h[w] < KNN && cand_less(s_cand[w * KNN + h[w]], bc)) { bc = s_cand[w * KNN + h[w]]; bw = w; }
            }
            if (bw >= 0) ++h[bw];
            s_out[round] = bc.idx == 0x7fffffff ? -1 : bc.idx;
        }
    }
    __syncthreads();
}

// np.searchsorted(P.s, s, side="right") - 1 clamped to [0, n-2] (rewards.py:108-110, :272-274).  s is non-decreasing and the
// caller knows the segment the point was projected on, so the answer is found by walking from that hint (0-1 steps)
// instead of a 13-step binary search of dependent loads.
__device__ int seg_index_at_s(const RewardView& v, double s, int hint) {
    int idx = hint < 0 ? 0 : (hint > v.n - 1 ? v.n - 1 : hint);
    while (idx + 1 <= v.n - 1 && v.s[idx + 1] <= s) ++idx;     // largest idx with s[idx] <= s ...
    while (idx > 0 && v.s[idx] > s) --idx;                     // ... from either side
    if (idx == 0 && v.s[0] > s) idx = -1;                      // searchsorted(...) - 1 == -1 below the first knot
    idx = idx < 0 ? 0 : idx;
    idx = idx > v.n - 2 ? v.n - 2 : idx;
    return idx;
}

// project_xy (track_progress.py:58-95) on the K nearest midpoints, in ascending midpoint distance
__device__ int project_on_candidates(const RewardView& v, const int* idx, int K, double x, double y, double& s_out, double& t_out) {
    bool have = false;
    int best_i = 0;
    double best_d = 0., best_s = 0., best_t = 0.;
    for (int k = 0; k < K; ++k) {
        const int i = idx[k];
        if (i < 0) continue;
        const double ax = v.xy[2 * i], ay = v.xy[2 * i + 1];
        const double abx = v.xy[2 * i + 2] - ax, aby = v.xy[2 * i + 3] - ay;
        const double L2 = abx * abx + aby * aby;
        if (L2 <= 1e-12) continue;
        const double apx = x - ax, apy = y - ay;
        double tp = (apx * abx + apy * aby) / L2;
        tp = tp < 0.0 ? 0.0 : (tp > 1.0 ? 1.0 : tp);
        const double px = ax + tp * abx, py = ay + tp * aby;
        const double s_proj = v.s[i] + tp * sqrt(abx * abx + aby * aby);
        const double t_signed = (x - px) * v.nrm[2 * i] + (y - py) * v.nrm[2 * i + 1];
        const double dist = sqrt((x - px) * (x - px) + (y - py) * (y - py));
        if (!have || dist < best_d) { have = true; best_d = dist; best_s = s_proj; best_t = t_signed; best_i = i; }
    }
    if (!have) {   // degenerate fallback :90-93: snap to the nearest node
        int j = 0;
        double bd = INFINITY;
        for (int i = 0; i < v.n; ++i) {
            const double dx = v.xy[2 * i] - x, dy = v.xy[2 * i + 1] - y;
            const double d = sqrt(dx * dx + dy * dy);
            if (d < bd) { bd = d; j = i; }
        }
        s_out = v.s[j]; t_out = 0.0;
        return j;
    }
    s_out = best_s; t_out = best_t;
    return best_i;
}

__device__ double signed_step(const RewardView& v, RewardState& r, int who, double x, double y, double s_curr, double s_prev, int seg_hint) {
    double ds_geom = s_curr - s_prev;                                   // delta_s, track_progress.py:97-104
    if (v.p.closed) { if (ds_geom > 0.5 * v.L) ds_geom -= v.L; if (ds_geom < -0.5 * v.L) ds_geom += v.L; }
    if (!r.has_p_prev[who]) { r.has_p_prev[who] = 1; r.p_prev[who][0] = x; r.p_prev[who][1] = y; return 0.0; }
    const double dx = x - r.p_prev[who][0], dy = y - r.p_prev[who][1];
    r.p_prev[who][0] = x; r.p_prev[who][1] = y;
    const int idx = seg_index_at_s(v, s_curr, seg_hint);
    const double ds_sign = dx * v.tan[2 * idx] + dy * v.tan[2 * idx + 1];
    return copysign(fabs(ds_geom), fabs(ds_sign) > 1e-6 ? ds_sign : ds_geom);
}

__global__ void __launch_bounds__(RW_THREADS) shaped_reward_kernel(RewardView v, const float* __restrict__ obs,
                                                                   const uint8_t* __restrict__ reset_mask,
                                                                   double* __restrict__ out64, float* __restrict__ out32) {
    const int env = blockIdx.x, tid = threadIdx.x;
    const int B = v.p.num_beams;
    const float* ob = obs + (size_t)env * (B + 8);
    extern __shared__ unsigned s_bits[];            // [B] lidar as order-preserving unsigned
    __shared__ Cand s_cand[(RW_THREADS / 32) * KNN];
    __shared__ double s_lb[256];                    // lower bound of every midpoint block (nblk <= 256)
    __shared__ double s_tau[RW_THREADS / 32];
    __shared__ int s_cblk[256];
    __shared__ int s_ncand;
    __shared__ int s_knn[2][KNN];
    __shared__ double s_pose[5];                    // ex, ey, ox, oy, oth
    __shared__ double s_proj[4];                    // e_s, e_t, o_s, o_t
    __shared__ int s_flag[3];                       // early-out, steps, do-wall
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_sel[4];                   // prefix, remaining rank, count<=, min>
    __shared__ float s_q[2];
    __shared__ int s_seg[2];                        // segment each car was projected on (hint for the arclength lookups)
    RewardState& r = v.st[env];

    if (tid == 0) {
        if (reset_mask && reset_mask[env]) {        // reward_fn.reset() (rewards.py:262-264, _Prog.reset :98-106)
            RewardState z;
            memset(&z, 0, sizeof(z));
            z.flip = +1.0;
            r = z;
        }
        // parse_flat_obs :11-39 (the float32 fields are widened by float())
        s_pose[0] = (double)ob[B + 0]; s_pose[1] = (double)ob[B + 1];
        s_pose[2] = (double)ob[B + 4]; s_pose[3] = (double)ob[B + 5];
        double th = (double)ob[B + 6] + 3.141592653589793;
        double m = fmod(th, 2 * 3.141592653589793);
        if (m != 0.0) { if (m < 0.0) m += 2 * 3.141592653589793; } else m = 0.0;
        s_pose[4] = m - 3.141592653589793;
        const bool ego_col = ob[B + 3] != 0.0f, opp_col = ob[B + 7] != 0.0f;
        r.steps += 1;                                                   // :299
        s_flag[1] = r.steps;
        s_flag[0] = 0;
        if (ego_col) { s_flag[0] = 1; if (out64) out64[env] = -v.p.ego_crash_penalty; if (out32) out32[env] = (float)-v.p.ego_crash_penalty; }
        else if (opp_col && v.p.opp_crash_bonus > 0.0) { s_flag[0] = 1; if (out64) out64[env] = v.p.opp_crash_bonus; if (out32) out32[env] = (float)v.p.opp_crash_bonus; }
        s_flag[2] = r.steps >= v.p.grace_steps_wall;
    }
    __syncthreads();
    if (s_flag[0]) return;

    // ---- 5 nearest midpoints of both cars (cKDTree.query(p, k=5)), exactly, without visiting all of them: the
    // midpoints are grouped in blocks of 64 consecutive ones with a bounding circle (centre, R).  Any block holds >= 5
    // points within |p - c| + R of p, so tau = min over blocks of that bound is an upper bound on the 5th-nearest
    // distance, and only blocks with |p - c| - R <= tau can contain one of the 5.  On a race track that is 1-3 blocks.
    for (int who = 0; who < 2; ++who) {
        const double px = s_pose[2 * who], py = s_pose[2 * who + 1];
        double ub = INFINITY;
        for (int k = tid; k < v.nblk; k += RW_THREADS) {
            const double dx = v.blk[3 * k] - px, dy = v.blk[3 * k + 1] - py, R = v.blk[3 * k + 2];
            const double d = sqrt(dx * dx + dy * dy);
            s_lb[k] = d - R;
            const int cnt = min(MID_BLOCK, v.n - 1 - k * MID_BLOCK);
            if (cnt >= KNN) ub = fmin(ub, d + R);
        }
        for (int o = 16; o > 0; o >>= 1) ub = fmin(ub, __shfl_xor_sync(0xffffffffu, ub, o));
        if ((tid & 31) == 0) s_tau[tid >> 5] = ub;
        __syncthreads();
        double tau = fmin(fmin(s_tau[0], s_tau[1]), fmin(s_tau[2], s_tau[3]));
        tau = tau * (1.0 + 1e-12) + 1e-12;                              // slack for the rounding of the bounds
        Cand best[KNN];
#pragma unroll
        for (int k = 0; k < KNN; ++k) { best[k].d2 = INFINITY; best[k].idx = 0x7fffffff; }
        // compact the blocks that can hold one of the 5 (all of them if no block has 5 points)
        if (tid == 0) s_ncand = 0;
        __syncthreads();
        for (int k = tid; k < v.nblk; k += RW_THREADS)
            if (!(tau < INFINITY) || s_lb[k] <= tau) s_cblk[atomicAdd(&s_ncand, 1)] = k;
        __syncthreads();
        const int ncand = s_ncand;
        for (int j0 = 0; j0 < ncand; j0 += RW_THREADS / MID_BLOCK) {
            const int j = j0 + tid / MID_BLOCK;                         // two blocks per pass
            if (j < ncand) {
                const int i = s_cblk[j] * MID_BLOCK + (tid % MID_BLOCK);
                if (i < v.n - 1) {
                    const double dx = v.mid[2 * i] - px, dy = v.mid[2 * i + 1] - py;
                    topk_insert(best, dx * dx + dy * dy, i);
                }
            }
        }
        block_topk(best, s_cand, s_knn[who]);
    }
    if (tid == 0) s_seg[0] = project_on_candidates(v, s_knn[0], KNN, s_pose[0], s_pose[1], s_proj[0], s_proj[1]);
    if (tid == 32) s_seg[1] = project_on_candidates(v, s_knn[1], KNN, s_pose[2], s_pose[3], s_proj[2], s_proj[3]);

    // ---- np.quantile(rng, wall_q) of the float32 lidar (rewards.py:335-339): radix select of the two order statistics
    if (s_flag[2]) {
        const float lm = (float)v.p.lidar_max;
        for (int i = tid; i < B; i += RW_THREADS) {
            float x = ob[i];
            if (x <= 0.0f || !isfinite(x)) x = lm;                      // zeros / NaNs count as far
            x = x < 0.0f ? 0.0f : (x > lm ? lm : x);
            s_bits[i] = __float_as_uint(x);                             // x >= 0: unsigned order == float order
        }
        const float vi = (float)(B - 1) * (float)v.p.wall_quantile;     // numpy forms the virtual index in float32
        const int lo = (int)floorf(vi);
        if (tid == 0) { s_sel[0] = 0u; s_sel[1] = (unsigned)lo; }
        __syncthreads();
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int b = tid; b < 256; b += RW_THREADS) s_hist[b] = 0u;
            __syncthreads();
            const unsigned prefix = s_sel[0];
            const unsigned himask = shift == 24 ? 0u : (0xFFFFFFFFu << (shift + 8));
            for (int i = tid; i < B; i += RW_THREADS) {
                const unsigned u = s_bits[i];
                if ((u & himask) == prefix) atomicAdd(&s_hist[(u >> shift) & 0xFFu], 1u);
            }
            __syncthreads();
            if (tid < 32) {
                // which of the 256 bins holds rank s_sel[1]?  lane l owns bins 8l..8l+7: warp scan of the lane sums, then
                // the owning lane walks its own 8 bins
                unsigned c[8], sum = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) { c[j] = s_hist[8 * tid + j]; sum += c[j]; }
                unsigned incl = sum;
                for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (tid >= o) incl += t; }
                const unsigned rank = s_sel[1];
                const unsigned excl = incl - sum;
                const bool mine = rank >= excl && rank < incl;
                const unsigned owner = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;   // counts sum to >= rank + 1: exists
                __syncwarp();
                if (tid == (int)owner) {
                    unsigned rem = rank - excl, b = 0;
#pragma unroll
                    for (int j = 0; j < 7; ++j) if (b == (unsigned)j && rem >= c[j]) { rem -= c[j]; ++b; }
                    s_sel[0] = prefix | ((8u * tid + b) << shift);
                    s_sel[1] = rem;
                }
            }
            __syncthreads();
        }
        const unsigned vk = s_sel[0];                                   // bits of sorted[lo]
        if (tid == 0) { s_sel[2] = 0u; s_sel[3] = 0xFFFFFFFFu; }
        __syncthreads();
        unsigned cnt = 0, mn = 0xFFFFFFFFu;
        for (int i = tid; i < B; i += RW_THREADS) {
            const unsigned u = s_bits[i];
            if (u <= vk) ++cnt; else mn = u < mn ? u : mn;
        }
        atomicAdd(&s_sel[2], cnt);
        atomicMin(&s_sel[3], mn);
        __syncthreads();
        if (tid == 0) {
            const int hi = lo + 1 < B ? lo + 1 : B - 1;
            const float a = __uint_as_float(vk);
            const float b = (hi == lo || s_sel[2] >= (unsigned)(lo + 2)) ? a : __uint_as_float(s_sel[3]);
            const float g = __fsub_rn(vi, (float)lo);
            const float d = __fsub_rn(b, a);
            // _lerp in float32: b - (b-a)*(1-g) for g >= 0.5, else a + (b-a)*g
            s_q[0] = g >= 0.5f ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g))) : __fadd_rn(a, __fmul_rn(d, g));
        }
    }
    __syncthreads();

    if (tid == 0) {
        const double ex = s_pose[0], ey = s_pose[1], ox = s_pose[2], oy = s_pose[3], oth = s_pose[4];
        const double e_s = s_proj[0], e_t = s_proj[1], o_s = s_proj[2], o_t = s_proj[3];
        // _Prog.update :129-167
        if (!r.has_s_prev[0]) { r.has_s_prev[0] = 1; r.s_prev[0] = e_s; }
        if (!r.has_s_prev[1]) { r.has_s_prev[1] = 1; r.s_prev[1] = o_s; }
        double de = signed_step(v, r, 0, ex, ey, e_s, r.s_prev[0], s_seg[0]);
        double dop = signed_step(v, r, 1, ox, oy, o_s, r.s_prev[1], s_seg[1]);
        r.s_prev[0] = e_s; r.s_prev[1] = o_s;
        if (r.buf_n < 20) {
            r.buf_sum += de; r.buf_n += 1;
            if (r.buf_n == 20 && r.buf_sum / 20 < 0.0) r.flip = -1.0;
        }
        de *= r.flip; dop *= r.flip;
        r.cum[0] += de; r.cum[1] += dop;
        r.ema_abs = 0.8 * r.ema_abs + (1.0 - 0.8) * fabs(de);
        r.t_last[0] = e_t; r.t_last[1] = o_t;
        const int steps = s_flag[1];
        double dego = de;
        if (steps < 10 && dego < 0.0) dego = 0.0;                        // :311-312
        const double r_prog = v.p.w_prog * v.p.forward_sign * dego;
        const double r_alive = v.p.alive_bonus;
        double r_lead = 0.0;
        if (v.p.w_rel_lead != 0.0) {
            double lead = r.cum[0] - r.cum[1];
            lead = lead < -v.p.lead_clip ? -v.p.lead_clip : (lead > v.p.lead_clip ? v.p.lead_clip : lead);
            r_lead = v.p.w_rel_lead * (lead / v.p.lead_clip);
        }
        const int idx = seg_index_at_s(v, e_s, s_seg[0]);                // lateral :323-333
        double wR = v.p.default_half_width, wL = v.p.default_half_width;
        if (v.wR && v.wL) { wR = v.wR[idx]; wL = v.wL[idx]; }
        double w_eff = e_t >= 0.0 ? wL : wR;
        w_eff = w_eff < 0.2 ? 0.2 : w_eff;
        const double lat_norm = fabs(e_t) / w_eff;
        const double lat_sq = lat_norm * lat_norm;
        const double r_lat = -v.p.w_lat * (lat_sq < v.p.lat_cap ? lat_sq : v.p.lat_cap);
        double r_wall = 0.0;                                             // :335-343
        if (s_flag[2]) {
            const double dmin = (double)s_q[0];
            if (dmin < v.p.near_wall_dist) {
                const double x = (v.p.near_wall_dist - dmin) / (v.p.near_wall_dist > 1e-6 ? v.p.near_wall_dist : 1e-6);
                r_wall = -v.p.w_wall * (x * x);
            }
        }
        double r_opp = 0.0;                                              // :345-352
        if (steps >= v.p.grace_steps_opp) {
            const double rho = hypot(ex - ox, ey - oy);
            if (rho < v.p.opp_safe_dist) {
                const double y = (v.p.opp_safe_dist - rho) / (v.p.opp_safe_dist > 1e-6 ? v.p.opp_safe_dist : 1e-6);
                r_opp = -v.p.w_opp * (y * y);
            }
        }
        double r_flank = 0.0;                                            // :353-358
        {
            const double dx = ex - ox, dy = ey - oy;
            double sn, cs;
            sincos(-oth, &sn, &cs);
            const double x_rel = cs * dx - sn * dy, y_rel = sn * dx + cs * dy;
            if (0.2 <= x_rel && x_rel <= 1.8 && 0.25 <= fabs(y_rel) && fabs(y_rel) <= 0.8) {
                double yb = 0.8 - fabs(fabs(y_rel) - 0.525);
                yb = yb < 0.0 ? 0.0 : yb;
                r_flank = 0.1 * (x_rel / 1.8) * (yb / 0.8);
            }
        }
        const double total = r_prog + r_alive + r_lead + r_lat + r_wall + r_opp + r_flank;
        if (out64) out64[env] = total;
        if (out32) out32[env] = (float)total;
    }
}


// The same reward with ONE WARP per env (round 2; the CTA-per-env kernel above stays as the form for scans too long for a
// warp's share of shared memory).  Nothing about the arithmetic changes: the one-thread sections (observation parsing,
// projections, the progress state machine) are the same statements run by lane 0 (lanes 0 and 1 for the two projections),
// the 5-nearest search and the quantile's radix select produce the same discrete answers with warp-wide instead of
// CTA-wide steps -- and no barrier: a third of the CTA kernel's stall samples were barriers around one-thread sections.
constexpr int RWW_MAX = 4;      // envs per CTA

__device__ __forceinline__ size_t reward_warp_smem_bytes(int B) { return sizeof(unsigned) * ((size_t)B + 256) + sizeof(double) * 256 + sizeof(int) * (256 + 2 * KNN + 2); }

__global__ void __launch_bounds__(RWW_MAX * 32) shaped_reward_warp_kernel(RewardView v, const float* __restrict__ obs,
                                                                          const uint8_t* __restrict__ reset_mask,
                                                                          double* __restrict__ out64, float* __restrict__ out32) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int env = blockIdx.x * (blockDim.x >> 5) + wid;
    if (env >= v.p.num_envs) return;
    const int B = v.p.num_beams;
    extern __shared__ __align__(16) unsigned char s_raw[];
    unsigned char* mine = s_raw + (size_t)wid * ((reward_warp_smem_bytes(B) + 15) & ~size_t(15));
    double* s_lb = reinterpret_cast<double*>(mine);                       // [256] lower bound of every midpoint block
    unsigned* s_bits = reinterpret_cast<unsigned*>(s_lb + 256);           // [B] lidar as order-preserving unsigned
    unsigned* s_hist = s_bits + B;                                        // [256]
    int* s_cblk = reinterpret_cast<int*>(s_hist + 256);                   // [256]
    int* s_knn = s_cblk + 256;                                            // [2][KNN]
    const float* ob = obs + (size_t)env * (B + 8);
    // the env's progress state lives in lane 0's registers for the duration of the kernel: one load of the record and one
    // store, instead of a dependent global access per field of the state machine
    RewardState r;
    memset(&r, 0, sizeof(r));

    double pose[5] = {0., 0., 0., 0., 0.};                                // ex, ey, ox, oy, oth
    int early = 0, steps = 0, do_wall = 0;
    if (lane == 0) {
        if (reset_mask && reset_mask[env]) {        // reward_fn.reset() (rewards.py:262-264, _Prog.reset :98-106)
            r.flip = +1.0;                          // everything else zero
        } else {
            r = v.st[env];
        }
        // parse_flat_obs :11-39 (the float32 fields are widened by float())
        pose[0] = (double)ob[B + 0]; pose[1] = (double)ob[B + 1];
        pose[2] = (double)ob[B + 4]; pose[3] = (double)ob[B + 5];
        double th = (double)ob[B + 6] + 3.141592653589793;
        double m = fmod(th, 2 * 3.141592653589793);
        if (m != 0.0) { if (m < 0.0) m += 2 * 3.141592653589793; } else m = 0.0;
        pose[4] = m - 3.141592653589793;
        const bool ego_col = ob[B + 3] != 0.0f, opp_col = ob[B + 7] != 0.0f;
        r.steps += 1;                                                   // :299
        steps = r.steps;
        if (ego_col) { early = 1; if (out64) out64[env] = -v.p.ego_crash_penalty; if (out32) out32[env] = (float)-v.p.ego_crash_penalty; }
        else if (opp_col && v.p.opp_crash_bonus > 0.0) { early = 1; if (out64) out64[env] = v.p.opp_crash_bonus; if (out32) out32[env] = (float)v.p.opp_crash_bonus; }
        do_wall = r.steps >= v.p.grace_steps_wall;
        if (early) v.st[env] = r;
    }
    early = __shfl_sync(0xffffffffu, early, 0);
    if (early) return;
    steps = __shfl_sync(0xffffffffu, steps, 0);
    do_wall = __shfl_sync(0xffffffffu, do_wall, 0);
#pragma unroll
    for (int k = 0; k < 5; ++k) pose[k] = __shfl_sync(0xffffffffu, pose[k], 0);

    // ---- 5 nearest midpoints of both cars, exactly (see the CTA kernel for the bounding-circle argument)
    for (int who = 0; who < 2; ++who) {
        const double px = pose[2 * who], py = pose[2 * who + 1];
        double ub = INFINITY;
        for (int k = lane; k < v.nblk; k += 32) {
            const double dx = v.blk[3 * k] - px, dy = v.blk[3 * k + 1] - py, R = v.blk[3 * k + 2];
            const double d = sqrt(dx * dx + dy * dy);
            s_lb[k] = d - R;
            const int cnt = min(MID_BLOCK, v.n - 1 - k * MID_BLOCK);
            if (cnt >= KNN) ub = fmin(ub, d + R);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ub = fmin(ub, __shfl_xor_sync(0xffffffffu, ub, o));
        const double tau = ub * (1.0 + 1e-12) + 1e-12;                  // slack for the rounding of the bounds
        __syncwarp();
        int ncand = 0;
        for (int k0 = 0; k0 < v.nblk; k0 += 32) {
            const int k = k0 + lane;
            const bool keep = k < v.nblk && (!(tau < INFINITY) || s_lb[k] <= tau);
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) s_cblk[ncand + __popc(m & ((1u << lane) - 1u))] = k;
            ncand += __popc(m);
        }
        __syncwarp();
        Cand best[KNN];
#pragma unroll
        for (int k = 0; k < KNN; ++k) { best[k].d2 = INFINITY; best[k].idx = 0x7fffffff; }
        for (int j = 0; j < ncand; ++j) {
            const int base = s_cblk[j] * MID_BLOCK;
#pragma unroll
            for (int t = 0; t < MID_BLOCK / 32; ++t) {
                const int i = base + 32 * t + lane;
                if (i < v.n - 1) {
                    const double dx = v.mid[2 * i] - px, dy = v.mid[2 * i + 1] - py;
                    topk_insert(best, dx * dx + dy * dy, i);
                }
            }
        }
        // the warp's KNN smallest (d2, idx): every round the lanes offer the head of their sorted private lists
        int head = 0;
        for (int round = 0; round < KNN; ++round) {
            Cand cnd;
            cnd.d2 = INFINITY; cnd.idx = 0x7fffffff;
#pragma unroll
            for (int k = 0; k < KNN; ++k) if (k == head) cnd = best[k];
            const unsigned long long bits = (unsigned long long)__double_as_longlong(cnd.d2);     // d2 >= 0: bits order like the value
            const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
            const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
            const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xFFFFFFFFu);
            const unsigned midx = __reduce_min_sync(0xffffffffu, (hi == mhi && lo == mlo) ? (unsigned)cnd.idx : 0x7FFFFFFFu);
            if ((int)midx == cnd.idx && cnd.idx != 0x7fffffff) ++head;      // a midpoint index belongs to exactly one lane
            if (lane == 0) s_knn[who * KNN + round] = midx == 0x7FFFFFFFu ? -1 : (int)midx;
        }
        __syncwarp();
    }
    // projections: lane 0 the ego, lane 1 the opponent (same code, different data: no divergence)
    double p_s = 0., p_t = 0.;
    int p_seg = 0;
    if (lane < 2) p_seg = project_on_candidates(v, s_knn + lane * KNN, KNN, pose[2 * lane], pose[2 * lane + 1], p_s, p_t);
    const double o_s = __shfl_sync(0xffffffffu, p_s, 1), o_t = __shfl_sync(0xffffffffu, p_t, 1);
    const int seg1 = __shfl_sync(0xffffffffu, p_seg, 1);

    // ---- np.quantile(rng, wall_q) of the float32 lidar (rewards.py:335-339): radix select of the two order statistics
    float q_wall = 0.f;
    if (do_wall) {
        const float lm = (float)v.p.lidar_max;
        for (int i = lane; i < B; i += 32) {
            float x = ob[i];
            if (x <= 0.0f || !isfinite(x)) x = lm;                      // zeros / NaNs count as far
            x = x < 0.0f ? 0.0f : (x > lm ? lm : x);
            s_bits[i] = __float_as_uint(x);                             // x >= 0: unsigned order == float order
        }
        const float vi = (float)(B - 1) * (float)v.p.wall_quantile;     // numpy forms the virtual index in float32
        const int lo = (int)floorf(vi);
        unsigned prefix = 0u, rank = (unsigned)lo;
        for (int shift = 24; shift >= 0; shift -= 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) s_hist[8 * lane + j] = 0u;
            __syncwarp();
            const unsigned himask = shift == 24 ? 0u : (0xFFFFFFFFu << (shift + 8));
            for (int i = lane; i < B; i += 32) {
                const unsigned u = s_bits[i];
                if ((u & himask) == prefix) atomicAdd(&s_hist[(u >> shift) & 0xFFu], 1u);
            }
            __syncwarp();
            // which of the 256 bins holds the rank?  lane l owns bins 8l..8l+7: warp scan of the lane sums, then the owning
            // lane walks its own 8 bins
            unsigned c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = s_hist[8 * lane + j]; sum += c[j]; }
            unsigned incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            const unsigned excl = incl - sum;
            const bool own = rank >= excl && rank < incl;
            const int owner = __ffs(__ballot_sync(0xffffffffu, own)) - 1;    // counts sum to >= rank + 1: exists
            unsigned np = 0, nr = 0;
            if (lane == owner) {
                unsigned rem = rank - excl, b = 0;
#pragma unroll
                for (int j = 0; j < 7; ++j) if (b == (unsigned)j && rem >= c[j]) { rem -= c[j]; ++b; }
                np = prefix | ((8u * lane + b) << shift);
                nr = rem;
            }
            prefix = __shfl_sync(0xffffffffu, np, owner);
            rank = __shfl_sync(0xffffffffu, nr, owner);
            __syncwarp();
        }
        const unsigned vk = prefix;                                     // bits of sorted[lo]
        unsigned cnt = 0, mn = 0xFFFFFFFFu;
        for (int i = lane; i < B; i += 32) {
            const unsigned u = s_bits[i];
            if (u <= vk) ++cnt; else mn = u < mn ? u : mn;
        }
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        mn = __reduce_min_sync(0xffffffffu, mn);
        const int hi = lo + 1 < B ? lo + 1 : B - 1;
        const float a = __uint_as_float(vk);
        const float b = (hi == lo || cnt >= (unsigned)(lo + 2)) ? a : __uint_as_float(mn);
        const float g = __fsub_rn(vi, (float)lo);
        const float d = __fsub_rn(b, a);
        // _lerp in float32: b - (b-a)*(1-g) for g >= 0.5, else a + (b-a)*g
        q_wall = g >= 0.5f ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g))) : __fadd_rn(a, __fmul_rn(d, g));
    }

    if (lane == 0) {
        const double ex = pose[0], ey = pose[1], ox = pose[2], oy = pose[3], oth = pose[4];
        const double e_s = p_s, e_t = p_t;
        const int seg0 = p_seg;
        // _Prog.update :129-167
        if (!r.has_s_prev[0]) { r.has_s_prev[0] = 1; r.s_prev[0] = e_s; }
        if (!r.has_s_prev[1]) { r.has_s_prev[1] = 1; r.s_prev[1] = o_s; }
        double de = signed_step(v, r, 0, ex, ey, e_s, r.s_prev[0], seg0);
        double dop = signed_step(v, r, 1, ox, oy, o_s, r.s_prev[1], seg1);
        r.s_prev[0] = e_s; r.s_prev[1] = o_s;
        if (r.buf_n < 20) {
            r.buf_sum += de; r.buf_n += 1;
            if (r.buf_n == 20 && r.buf_sum / 20 < 0.0) r.flip = -1.0;
        }
        de *= r.flip; dop *= r.flip;
        r.cum[0] += de; r.cum[1] += dop;
        r.ema_abs = 0.8 * r.ema_abs + (1.0 - 0.8) * fabs(de);
        r.t_last[0] = e_t; r.t_last[1] = o_t;
        double dego = de;
        if (steps < 10 && dego < 0.0) dego = 0.0;                        // :311-312
        const double r_prog = v.p.w_prog * v.p.forward_sign * dego;
        const double r_alive = v.p.alive_bonus;
        double r_lead = 0.0;
        if (v.p.w_rel_lead != 0.0) {
            double lead = r.cum[0] - r.cum[1];
            lead = lead < -v.p.lead_clip ? -v.p.lead_clip : (lead > v.p.lead_clip ? v.p.lead_clip : lead);
            r_lead = v.p.w_rel_lead * (lead / v.p.lead_clip);
        }
        const int idx = seg_index_at_s(v, e_s, seg0);                    // lateral :323-333
        double wR = v.p.default_half_width, wL = v.p.default_half_width;
        if (v.wR && v.wL) { wR = v.wR[idx]; wL = v.wL[idx]; }
        double w_eff = e_t >= 0.0 ? wL : wR;
        w_eff = w_eff < 0.2 ? 0.2 : w_eff;
        const double lat_norm = fabs(e_t) / w_eff;
        const double lat_sq = lat_norm * lat_norm;
        const double r_lat = -v.p.w_lat * (lat_sq < v.p.lat_cap ? lat_sq : v.p.lat_cap);
        double r_wall = 0.0;                                             // :335-343
        if (do_wall) {
            const double dmin = (double)q_wall;
            if (dmin < v.p.near_wall_dist) {
                const double x = (v.p.near_wall_dist - dmin) / (v.p.near_wall_dist > 1e-6 ? v.p.near_wall_dist : 1e-6);
                r_wall = -v.p.w_wall * (x * x);
            }
        }
        double r_opp = 0.0;                                              // :345-352
        if (steps >= v.p.grace_steps_opp) {
            const double rho = hypot(ex - ox, ey - oy);
            if (rho < v.p.opp_safe_dist) {
                const double y = (v.p.opp_safe_dist - rho) / (v.p.opp_safe_dist > 1e-6 ? v.p.opp_safe_dist : 1e-6);
                r_opp = -v.p.w_opp * (y * y);
            }
        }
        double r_flank = 0.0;                                            // :353-358
        {
            const double dx = ex - ox, dy = ey - oy;
            double sn, cs;
            sincos(-oth, &sn, &cs);
            const double x_rel = cs * dx - sn * dy, y_rel = sn * dx + cs * dy;
            if (0.2 <= x_rel && x_rel <= 1.8 && 0.25 <= fabs(y_rel) && fabs(y_rel) <= 0.8) {
                double yb = 0.8 - fabs(fabs(y_rel) - 0.525);
                yb = yb < 0.0 ? 0.0 : yb;
                r_flank = 0.1 * (x_rel / 1.8) * (yb / 0.8);
            }
        }
        const double total = r_prog + r_alive + r_lead + r_lat + r_wall + r_opp + r_flank;
        if (out64) out64[env] = total;
        if (out32) out32[env] = (float)total;
        v.st[env] = r;
    }
}

}  // namespace

extern "C" int f110_reward_create(const F110RewardConfig* cfg, const double* xy, const double* wR, const double* wL,
                                  F110Reward** out) {
    if (!cfg || !xy || !out || cfg->num_envs < 1 || cfg->num_points < 2 || cfg->num_beams < 1 || cfg->num_beams > 8192)
        return f110_set_error(F110_ERR_INVALID, "f110_reward_create: need num_envs >= 1, num_points >= 2, 1 <= num_beams <= 8192");
    if ((cfg->num_points - 1 + MID_BLOCK - 1) / MID_BLOCK > 256)
        return f110_set_error(F110_ERR_INVALID, "f110_reward_create: at most 16385 centerline points");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return f110_set_error(F110_ERR_NO_DEVICE, "no CUDA device visible: libf110_b200 has no CPU fallback");
    }
    int prev = 0;
    cudaGetDevice(&prev);
    if (cudaSetDevice(cfg->device) != cudaSuccess) return F110_ERR_CUDA;
    F110Reward* r = new F110Reward();
    r->cfg = *cfg; r->n = cfg->num_points; r->device = cfg->device;
    const int n = r->n;
    // CenterlineProgress.__init__, track_progress.py:33-49 (host, once)
    double* s = new double[n];
    double* tan = new double[2 * (n - 1)];
    double* nrm = new double[2 * (n - 1)];
    double* mid = new double[2 * (n - 1)];
    s[0] = 0.0;
    for (int i = 0; i < n - 1; ++i) {
        const double sx = xy[2 * i + 2] - xy[2 * i], sy = xy[2 * i + 3] - xy[2 * i + 1];
        const double len = sqrt(sx * sx + sy * sy);
        s[i + 1] = s[i] + len;
        const double den = len > 1e-12 ? len : 1e-12;
        tan[2 * i] = sx / den; tan[2 * i + 1] = sy / den;
        nrm[2 * i] = -tan[2 * i + 1]; nrm[2 * i + 1] = tan[2 * i];
        mid[2 * i] = (xy[2 * i] + xy[2 * i + 2]) * 0.5; mid[2 * i + 1] = (xy[2 * i + 1] + xy[2 * i + 3]) * 0.5;
    }
    r->L = s[n - 1];
    auto up = [](const double* h, size_t cnt, double** d) {
        if (cudaMalloc(d, cnt * sizeof(double)) != cudaSuccess) return false;
        return cudaMemcpy(*d, h, cnt * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess;
    };
    bool ok = up(xy, 2 * (size_t)n, &r->xy) && up(s, n, &r->s) && up(tan, 2 * (size_t)(n - 1), &r->tan) &&
              up(nrm, 2 * (size_t)(n - 1), &r->nrm) && up(mid, 2 * (size_t)(n - 1), &r->mid);
    r->wR = r->wL = nullptr;
    if (ok && wR && wL) ok = up(wR, n, &r->wR) && up(wL, n, &r->wL);
    {   // bounding circles of MID_BLOCK consecutive midpoints
        r->nblk = (n - 1 + MID_BLOCK - 1) / MID_BLOCK;
        std::vector<double> blk(3 * (size_t)r->nblk);
        for (int k = 0; k < r->nblk; ++k) {
            const int i0 = k * MID_BLOCK, i1 = (k + 1) * MID_BLOCK < n - 1 ? (k + 1) * MID_BLOCK : n - 1;
            double cx = 0, cy = 0;
            for (int i = i0; i < i1; ++i) { cx += mid[2 * i]; cy += mid[2 * i + 1]; }
            cx /= (i1 - i0); cy /= (i1 - i0);
            double R = 0;
            for (int i = i0; i < i1; ++i) { const double d = sqrt((mid[2 * i] - cx) * (mid[2 * i] - cx) + (mid[2 * i + 1] - cy) * (mid[2 * i + 1] - cy)); R = d > R ? d : R; }
            blk[3 * k] = cx; blk[3 * k + 1] = cy; blk[3 * k + 2] = R * (1.0 + 1e-12) + 1e-12;
        }
        r->blk = nullptr;
        if (ok) ok = r->nblk <= 256 && up(blk.data(), blk.size(), &r->blk);
    }
    delete[] s; delete[] tan; delete[] nrm; delete[] mid;
    if (ok) {
        std::vector<RewardState> init(cfg->num_envs);
        memset(init.data(), 0, sizeof(RewardState) * init.size());
        for (auto& st : init) st.flip = +1.0;
        ok = cudaMalloc(&r->state, sizeof(RewardState) * init.size()) == cudaSuccess &&
             cudaMemcpy(r->state, init.data(), sizeof(RewardState) * init.size(), cudaMemcpyHostToDevice) == cudaSuccess;
    }
    cudaSetDevice(prev);
    if (!ok) { f110_reward_destroy(r); cudaGetLastError(); return f110_set_error(F110_ERR_CUDA, "f110_reward_create: device allocation / upload failed"); }
    *out = r;
    return F110_OK;
}

extern "C" void f110_reward_destroy(F110Reward* r) {
    if (!r) return;
    cudaFree(r->xy); cudaFree(r->s); cudaFree(r->tan); cudaFree(r->nrm); cudaFree(r->mid); cudaFree(r->wR); cudaFree(r->wL);
    cudaFree(r->blk); cudaFree(r->state);
    delete r;
}

extern "C" int f110_reward_compute(F110Reward* r, const float* obs, const uint8_t* reset_mask, double* out_f64, float* out_f32,
                                   void* stream) {
    if (!r || !obs || (!out_f64 && !out_f32)) return f110_set_error(F110_ERR_INVALID, "f110_reward_compute: null handle, obs or outputs");
    RewardView v;
    v.p = r->cfg; v.n = r->n; v.L = r->L;
    v.blk = r->blk; v.nblk = r->nblk;
    v.xy = r->xy; v.s = r->s; v.tan = r->tan; v.nrm = r->nrm; v.mid = r->mid; v.wR = r->wR; v.wL = r->wL;
    v.st = static_cast<RewardState*>(r->state);
    // a warp per env where a warp's scratch (the scan as sortable words, a histogram, the block bounds) fits the 48 KB of
    // shared memory that need no opt-in; else (scans of more than ~11 000 beams) the CTA-per-env form
    const int B = r->cfg.num_beams;
    const size_t per_warp = ((sizeof(unsigned) * ((size_t)B + 256) + sizeof(double) * 256 + sizeof(int) * (256 + 2 * KNN + 2)) + 15) & ~size_t(15);
    const char* force_cta = getenv("F110_REWARD_CTA");      // test switch: the round-1 kernel
    if (per_warp <= 48 * 1024 && !(force_cta && force_cta[0] == '1')) {
        int warps = (int)((48 * 1024) / per_warp);
        warps = warps > RWW_MAX ? RWW_MAX : warps;
        shaped_reward_warp_kernel<<<(r->cfg.num_envs + warps - 1) / warps, warps * 32, per_warp * warps, (cudaStream_t)stream>>>(
            v, obs, reset_mask, out_f64, out_f32);
    } else {
        shaped_reward_kernel<<<r->cfg.num_envs, RW_THREADS, sizeof(unsigned) * r->cfg.num_beams, (cudaStream_t)stream>>>(
            v, obs, reset_mask, out_f64, out_f32);
    }
    return cudaPeekAtLastError() == cudaSuccess ? F110_OK : F110_ERR_CUDA;
}
