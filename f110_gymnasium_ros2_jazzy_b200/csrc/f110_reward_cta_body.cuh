// f110_reward_cta_body.cuh -- the body of the CTA-per-env shaped reward kernel, included by shaped_reward_kernel and
// shaped_reward_set_kernel in f110_consumers.cu, as f110_reward_warp_body.cuh is (see there why by textual inclusion).
// The set kernel names its parameter `base` and reads the view of the env's line from shared memory.
    const int env = blockIdx.x, tid = threadIdx.x;
#if F110_REWARD_SET
    // the view of the env's line lives in shared memory: in registers, its pointers did not survive the calls of the
    // one-thread sections without spilling
    __shared__ RewardView s_view;
    const int slot = rs.slots[env];
    if ((unsigned)slot >= (unsigned)rs.count) {     // NaN, the record and the stored slot untouched
        if (tid == 0) write_nan(out64, out32, env);
        return;
    }
    bool moved = false;                             // a changed slot restarts the record, as reset_mask does
    if (tid == 0) {
        RewardView w = base;
        select_line(w, rs.lines[slot]);
        s_view = w;
        moved = rs.prev[env] != slot;
        rs.prev[env] = slot;
    }
    __syncthreads();
    const RewardView& v = s_view;
#endif
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
#if F110_REWARD_SET
        if ((reset_mask && reset_mask[env]) || moved) {
#else
        if (reset_mask && reset_mask[env]) {        // reward_fn.reset() (rewards.py:262-264, _Prog.reset :98-106)
#endif
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
