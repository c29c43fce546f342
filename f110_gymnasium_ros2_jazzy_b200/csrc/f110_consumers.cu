// f110_consumers.cu -- device-side forms of the consumers that sit directly around the env in the reference's
// training loop (SURVEY 8f), so a rollout never leaves the GPU.  Paths are relative to /root/reference/.
//
//   gap_follow_kernel : rl_training/utils/gap_follow.py:3-58, the rule-based opponent train_ddpg.py:168 drives
//                       from info["scans"][1].  One warp per scan; float32 arithmetic in numpy's order, so the
//                       chosen beam index -- and with it (steer, speed) -- is identical to the reference's.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
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
//   shaped_reward_warp_kernel : rl_training/utils/rewards.py:185-355 (CenterlineSafetyProgressReward, with _Prog :86-180
//                          and parse_flat_obs :11-39) over rl_training/utils/track_progress.py (CenterlineProgress.project_xy
//                          :58-95, delta_s :97-104) -- the reward train_ddpg.py:179 computes from the flat observation.
//                          One warp per env: exact 5-nearest segment midpoints for both cars (the reference's
//                          cKDTree.query(k=5)), radix select for numpy's float32 quantile of the lidar, then lane 0 runs
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
    int count;                                    // centerlines: 1, or a set of K (n, L, nblk and cfg.closed then unused)
    void* lines;                                  // device RewardLine[count] (sets only)
    int* prev_slot;                               // device [N]: each env's slot at its previous call, -1 at first (sets only)
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

// A set of K centerlines: the lines lie back to back in one allocation per array, line k's points from `off` on (xy, s,
// wR, wL; tan, nrm, mid likewise, one entry short), its bounding circles from block `boff` on.  The set kernel reads the
// env's slot, then the slot's record, and points a RewardView at that line; from there on it is the single-line kernel.
struct RewardLine {
    int off, n, nblk, boff;
    double L;
    int closed, has_widths;
};

struct RewardSetView {
    const RewardLine* lines;
    const int* slots;                             // [N] the caller's
    int* prev;                                    // [N] F110Reward::prev_slot
    int count;
};

constexpr int RW_MAX_BEAMS = 8192;   // the longest scan a reward object accepts
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

// v (a view of the whole set) <- the view of one of its lines
__device__ __forceinline__ void select_line(RewardView& v, const RewardLine& ln) {
    const size_t o = (size_t)ln.off;
    v.n = ln.n; v.L = ln.L; v.nblk = ln.nblk; v.p.closed = ln.closed;
    v.xy += 2 * o; v.s += o; v.tan += 2 * o; v.nrm += 2 * o; v.mid += 2 * o;
    v.wR = ln.has_widths ? v.wR + o : nullptr;
    v.wL = ln.has_widths ? v.wL + o : nullptr;
    v.blk += 3 * (size_t)ln.boff;
}

__device__ __forceinline__ void write_nan(double* out64, float* out32, int env) {
    if (out64) out64[env] = __longlong_as_double(0x7ff8000000000000LL);
    if (out32) out32[env] = __int_as_float(0x7fc00000);
}

// ONE WARP per env: the one-thread sections (observation parsing, projections, the progress state machine) are lane 0's
// (lanes 0 and 1 for the two projections), the 5-nearest search and the quantile's radix select take warp-wide steps, and
// nothing waits at a barrier -- with a CTA per env (round 1), a third of the stall samples were barriers around the
// one-thread sections.
constexpr int RWW_MAX = 4;      // envs per CTA

// a warp's share of shared memory: the scan as sortable words, a histogram, the block bounds and the candidates, rounded
// to 16 bytes so that the next warp's doubles stay aligned
__host__ __device__ constexpr size_t reward_warp_smem_bytes(int B) {
    return (sizeof(unsigned) * ((size_t)B + 256) + sizeof(double) * 256 + sizeof(int) * (256 + 2 * KNN + 2) + 15) & ~size_t(15);
}
// so every scan check_lines accepts runs with a warp per env in the 48 KB that need no opt-in
static_assert(reward_warp_smem_bytes(RW_MAX_BEAMS) <= 48 * 1024, "a warp's reward scratch must fit 48 KB at the longest scan");

__global__ void __launch_bounds__(RWW_MAX * 32) shaped_reward_warp_kernel(RewardView v, const float* __restrict__ obs,
                                                                          const uint8_t* __restrict__ reset_mask,
                                                                          double* __restrict__ out64, float* __restrict__ out32) {
#define F110_REWARD_SET 0
#include "f110_reward_warp_body.cuh"
#undef F110_REWARD_SET
}

// the warp-per-env kernel on a set of centerlines: each env on the line of its slot
__global__ void __launch_bounds__(RWW_MAX * 32) shaped_reward_set_warp_kernel(RewardView v, RewardSetView rs, const float* __restrict__ obs,
                                                                              const uint8_t* __restrict__ reset_mask,
                                                                              double* __restrict__ out64, float* __restrict__ out32) {
#define F110_REWARD_SET 1
#include "f110_reward_warp_body.cuh"
#undef F110_REWARD_SET
}

}  // namespace

namespace {

// Checks every line against the limits before anything is allocated; the message names the failing line and its limit.
int check_lines(const char* who, const F110RewardConfig* cfg, const F110Centerline* lines, int32_t count, F110Reward** out) {
    char msg[256];
    if (!cfg || !lines || !out || cfg->num_envs < 1 || cfg->num_beams < 1 || cfg->num_beams > RW_MAX_BEAMS) {
        snprintf(msg, sizeof(msg), "%s: need non-null arguments, num_envs >= 1, 1 <= num_beams <= %d", who, RW_MAX_BEAMS);
        return f110_set_error(F110_ERR_INVALID, msg);
    }
    if (count < 1 || count > F110_MAX_MAPS) {
        snprintf(msg, sizeof(msg), "%s: %d centerlines; 1 to %d allowed", who, (int)count, F110_MAX_MAPS);
        return f110_set_error(F110_ERR_INVALID, msg);
    }
    for (int k = 0; k < count; ++k) {
        const int n = lines[k].num_points;
        if (!lines[k].xy) {
            snprintf(msg, sizeof(msg), "%s: centerline %d has no points (xy is NULL)", who, k);
            return f110_set_error(F110_ERR_INVALID, msg);
        }
        if (n < 2 || (n - 1 + MID_BLOCK - 1) / MID_BLOCK > 256) {
            snprintf(msg, sizeof(msg), "%s: centerline %d has %d points; 2 to 16385 allowed (at most 256 blocks of %d midpoints)",
                     who, k, n, MID_BLOCK);
            return f110_set_error(F110_ERR_INVALID, msg);
        }
    }
    return F110_OK;
}

int reward_create(const char* who, const F110RewardConfig* cfg, const F110Centerline* lines, int32_t count, F110Reward** out) {
    const int rc = check_lines(who, cfg, lines, count, out);
    if (rc != F110_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return f110_set_error(F110_ERR_NO_DEVICE, "no CUDA device visible: libf110_b200 has no CPU fallback");
    }
    int prev = 0;
    cudaGetDevice(&prev);
    if (cudaSetDevice(cfg->device) != cudaSuccess) return F110_ERR_CUDA;
    F110Reward* r = new F110Reward();
    r->cfg = *cfg; r->device = cfg->device; r->count = count;
    if (count == 1) { r->cfg.num_points = lines[0].num_points; r->cfg.closed = lines[0].closed; }
    // the lines back to back: line k's points from off[k] on, its blocks from boff[k] on
    std::vector<RewardLine> table(count);
    size_t total = 0, total_blk = 0;
    bool widths = false;
    for (int k = 0; k < count; ++k) {
        RewardLine& t = table[k];
        t.off = (int)total; t.n = lines[k].num_points; t.boff = (int)total_blk;
        t.nblk = (t.n - 1 + MID_BLOCK - 1) / MID_BLOCK;
        t.closed = lines[k].closed; t.has_widths = lines[k].wR && lines[k].wL;
        widths = widths || t.has_widths;
        total += t.n; total_blk += t.nblk;
    }
    std::vector<double> xy(2 * total), s(total), tan(2 * total), nrm(2 * total), mid(2 * total), blk(3 * total_blk);
    std::vector<double> wR(widths ? total : 0), wL(widths ? total : 0);
    for (int k = 0; k < count; ++k) {
        RewardLine& t = table[k];
        const int n = t.n;
        const double* src = lines[k].xy;
        double *pxy = &xy[2 * (size_t)t.off], *ps = &s[t.off], *ptan = &tan[2 * (size_t)t.off], *pnrm = &nrm[2 * (size_t)t.off];
        double* pmid = &mid[2 * (size_t)t.off];
        memcpy(pxy, src, 2 * (size_t)n * sizeof(double));
        if (t.has_widths) {
            memcpy(&wR[t.off], lines[k].wR, (size_t)n * sizeof(double));
            memcpy(&wL[t.off], lines[k].wL, (size_t)n * sizeof(double));
        }
        // CenterlineProgress.__init__, track_progress.py:33-49 (host, once)
        ps[0] = 0.0;
        for (int i = 0; i < n - 1; ++i) {
            const double sx = src[2 * i + 2] - src[2 * i], sy = src[2 * i + 3] - src[2 * i + 1];
            const double len = sqrt(sx * sx + sy * sy);
            ps[i + 1] = ps[i] + len;
            const double den = len > 1e-12 ? len : 1e-12;
            ptan[2 * i] = sx / den; ptan[2 * i + 1] = sy / den;
            pnrm[2 * i] = -ptan[2 * i + 1]; pnrm[2 * i + 1] = ptan[2 * i];
            pmid[2 * i] = (src[2 * i] + src[2 * i + 2]) * 0.5; pmid[2 * i + 1] = (src[2 * i + 1] + src[2 * i + 3]) * 0.5;
        }
        t.L = ps[n - 1];
        for (int b = 0; b < t.nblk; ++b) {      // bounding circles of MID_BLOCK consecutive midpoints
            const int i0 = b * MID_BLOCK, i1 = (b + 1) * MID_BLOCK < n - 1 ? (b + 1) * MID_BLOCK : n - 1;
            double cx = 0, cy = 0;
            for (int i = i0; i < i1; ++i) { cx += pmid[2 * i]; cy += pmid[2 * i + 1]; }
            cx /= (i1 - i0); cy /= (i1 - i0);
            double R = 0;
            for (int i = i0; i < i1; ++i) { const double d = sqrt((pmid[2 * i] - cx) * (pmid[2 * i] - cx) + (pmid[2 * i + 1] - cy) * (pmid[2 * i + 1] - cy)); R = d > R ? d : R; }
            double* pb = &blk[3 * ((size_t)t.boff + b)];
            pb[0] = cx; pb[1] = cy; pb[2] = R * (1.0 + 1e-12) + 1e-12;
        }
    }
    r->n = table[0].n; r->L = table[0].L; r->nblk = table[0].nblk;
    auto up = [](const void* h, size_t bytes, void** d) {
        if (cudaMalloc(d, bytes) != cudaSuccess) return false;
        return cudaMemcpy(*d, h, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    };
    auto upd = [&](const std::vector<double>& h, double** d) { return up(h.data(), h.size() * sizeof(double), reinterpret_cast<void**>(d)); };
    bool ok = upd(xy, &r->xy) && upd(s, &r->s) && upd(tan, &r->tan) && upd(nrm, &r->nrm) && upd(mid, &r->mid) && upd(blk, &r->blk);
    if (ok && widths) ok = upd(wR, &r->wR) && upd(wL, &r->wL);
    if (ok && count > 1) {
        std::vector<int> minus1(cfg->num_envs, -1);
        ok = up(table.data(), table.size() * sizeof(RewardLine), &r->lines) &&
             up(minus1.data(), minus1.size() * sizeof(int), reinterpret_cast<void**>(&r->prev_slot));
    }
    if (ok) {
        std::vector<RewardState> init(cfg->num_envs);
        memset(init.data(), 0, sizeof(RewardState) * init.size());
        for (auto& st : init) st.flip = +1.0;
        ok = up(init.data(), sizeof(RewardState) * init.size(), &r->state);
    }
    cudaSetDevice(prev);
    if (!ok) {
        f110_reward_destroy(r);
        cudaGetLastError();
        char msg[128];
        snprintf(msg, sizeof(msg), "%s: device allocation / upload failed", who);
        return f110_set_error(F110_ERR_CUDA, msg);
    }
    *out = r;
    return F110_OK;
}

}  // namespace

extern "C" int f110_reward_create_set(const F110RewardConfig* cfg, const F110Centerline* lines, int32_t count, F110Reward** out) {
    return reward_create("f110_reward_create_set", cfg, lines, count, out);
}

extern "C" int f110_reward_create(const F110RewardConfig* cfg, const double* xy, const double* wR, const double* wL,
                                  F110Reward** out) {
    if (!cfg || !xy || !out) return f110_set_error(F110_ERR_INVALID, "f110_reward_create: null config, centerline or handle");
    F110Centerline line;
    line.xy = xy; line.wR = wR; line.wL = wL; line.num_points = cfg->num_points; line.closed = cfg->closed;
    return reward_create("f110_reward_create", cfg, &line, 1, out);
}

extern "C" int32_t f110_reward_count(const F110Reward* r) { return r ? r->count : 0; }

extern "C" void f110_reward_destroy(F110Reward* r) {
    if (!r) return;
    cudaFree(r->xy); cudaFree(r->s); cudaFree(r->tan); cudaFree(r->nrm); cudaFree(r->mid); cudaFree(r->wR); cudaFree(r->wL);
    cudaFree(r->blk); cudaFree(r->state); cudaFree(r->lines); cudaFree(r->prev_slot);
    delete r;
}

extern "C" int f110_reward_compute_slots(F110Reward* r, const float* obs, const uint8_t* reset_mask, const int32_t* slots,
                                         double* out_f64, float* out_f32, void* stream) {
    if (!r || !obs || (!out_f64 && !out_f32)) return f110_set_error(F110_ERR_INVALID, "f110_reward_compute: null handle, obs or outputs");
    if (r->count > 1 && !slots)
        return f110_set_error(F110_ERR_INVALID, "f110_reward_compute_slots: a set of centerlines needs the envs' slots");
    RewardView v;
    v.p = r->cfg; v.n = r->n; v.L = r->L;
    v.blk = r->blk; v.nblk = r->nblk;
    v.xy = r->xy; v.s = r->s; v.tan = r->tan; v.nrm = r->nrm; v.mid = r->mid; v.wR = r->wR; v.wL = r->wL;
    v.st = static_cast<RewardState*>(r->state);
    RewardSetView rs;
    rs.lines = static_cast<const RewardLine*>(r->lines); rs.slots = slots; rs.prev = r->prev_slot; rs.count = r->count;
    const bool set = r->count > 1;       // a set of one runs the single-line kernels and reads no slot
    // as many warps per CTA as the 48 KB of shared memory that need no opt-in hold, at least one (the static_assert above)
    const size_t per_warp = reward_warp_smem_bytes(r->cfg.num_beams);
    int warps = (int)((48 * 1024) / per_warp);
    warps = warps > RWW_MAX ? RWW_MAX : warps;
    const dim3 grid((r->cfg.num_envs + warps - 1) / warps), block(warps * 32);
    if (set) shaped_reward_set_warp_kernel<<<grid, block, per_warp * warps, (cudaStream_t)stream>>>(v, rs, obs, reset_mask, out_f64, out_f32);
    else shaped_reward_warp_kernel<<<grid, block, per_warp * warps, (cudaStream_t)stream>>>(v, obs, reset_mask, out_f64, out_f32);
    return cudaPeekAtLastError() == cudaSuccess ? F110_OK : F110_ERR_CUDA;
}

extern "C" int f110_reward_compute(F110Reward* r, const float* obs, const uint8_t* reset_mask, double* out_f64, float* out_f32,
                                   void* stream) {
    if (r && r->count > 1)
        return f110_set_error(F110_ERR_INVALID, "f110_reward_compute: this reward holds a set of centerlines; call "
                                                "f110_reward_compute_slots with the envs' slots");
    return f110_reward_compute_slots(r, obs, reset_mask, nullptr, out_f64, out_f32, stream);
}
