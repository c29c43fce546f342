// f110_reward_warp_body.cuh -- the body of the warp-per-env shaped reward kernel, included by shaped_reward_warp_kernel
// and shaped_reward_set_warp_kernel in f110_consumers.cu.  The including kernel defines F110_REWARD_SET (0 or 1) and
// has the parameters v, obs, reset_mask, out64, out32 (and rs, the set's RewardSetView, when F110_REWARD_SET is 1).
// Textual inclusion, not an inlined function: the single-centerline kernel is then compiled as the same function it
// was before sets existed, instruction for instruction (DESIGN.md section 10).  The set kernel differs only inside
// the #if F110_REWARD_SET blocks: it reads the env's slot and that line's record, points v at the line, and counts a
// changed slot as a reset.
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int env = blockIdx.x * (blockDim.x >> 5) + wid;
    if (env >= v.p.num_envs) return;
#if F110_REWARD_SET
    const int slot = rs.slots[env];
    if ((unsigned)slot >= (unsigned)rs.count) {     // NaN, the record and the stored slot untouched
        if (lane == 0) write_nan(out64, out32, env);
        return;
    }
    select_line(v, rs.lines[slot]);
    bool moved = false;                             // a changed slot restarts the record, as reset_mask does
    if (lane == 0) { moved = rs.prev[env] != slot; rs.prev[env] = slot; }
#endif
    const int B = v.p.num_beams;
    extern __shared__ __align__(16) unsigned char s_raw[];
    unsigned char* mine = s_raw + (size_t)wid * reward_warp_smem_bytes(B);
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
#if F110_REWARD_SET
        if ((reset_mask && reset_mask[env]) || moved) {
#else
        if (reset_mask && reset_mask[env]) {        // reward_fn.reset() (rewards.py:262-264, _Prog.reset :98-106)
#endif
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

    // ---- 5 nearest midpoints of both cars (cKDTree.query(p, k=5)), exactly, without visiting all of them: the
    // midpoints are grouped in blocks of 64 consecutive ones with a bounding circle (centre, R).  A block of >= 5
    // midpoints holds 5 within |p - c| + R of p, so tau = min over blocks of that bound is an upper bound on the 5th-nearest
    // distance, and only blocks with |p - c| - R <= tau can contain one of the 5.  On a race track that is 1-3 blocks.
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
