// f110_lidar_body.cuh -- the body of the lidar kernel (K2), included by lidar_kernel and lidar_maps_kernel in f110_kernels.cu.
// Each kernel defines before the #include: constexpr bool MAPS (a map set is installed) and `ms` (the set's MapSet; unused
// when !MAPS), besides its parameters c, m, st, sc, io.  Textual inclusion, not an inlined function: the single-map kernel
// is then compiled as the same function it was before map sets existed, instruction for instruction.
// See the comment above lidar_kernel in f110_kernels.cu for what the body does.
    constexpr bool TUNED = FB != 0;
    constexpr bool DIRECT = MODE == 1 || MODE == 2, OBS_ONLY = MODE == 2, LEAN = MODE >= 2;
    cudaGridDependencySynchronize();   // PDL: everything below reads what the dynamics kernel (and the previous step) wrote
    const unsigned lane = threadIdx.x & 31u;
    const unsigned nwarps = gridDim.x * (LIDAR_THREADS / 32);
    const unsigned epoch = sc.ctrl[CTRL_EPOCH];
    const unsigned par = epoch & 1u;
    // A processed unit's class word is set to `done`; the array then serves as the next step's recording array (heavier
    // classes overwrite it by atomicMin) and comes back two steps later, when `done` is the other of the two values:
    // whatever is >= 3 and not this step's `done` is a light unit that has not been processed yet.
    const unsigned done = 4u + ((epoch >> 1) & 1u);
    // list ends (K1 may have pushed the third count past its capacity)
    const unsigned n0 = sc.ctrl[CTRL_CUR], n1 = n0 + sc.ctrl[CTRL_CUR + 1], n2 = n1 + min(sc.ctrl[CTRL_CUR + 2], sc.cap[2]);
    const unsigned cap0 = sc.cap[0], cap1 = sc.cap[1], cap2 = sc.cap[2];
    const unsigned* __restrict__ cur_list = sc.list[par];
    unsigned* cur_cls = sc.cls[par];
    unsigned* __restrict__ next_list = sc.list[par ^ 1u];
    unsigned* __restrict__ next_cls = sc.cls[par ^ 1u];
    unsigned cnt_look = 0, cnt_rays = 0, cnt_max = 0, cnt_redone = 0;

    // The segment the warp serves and the end of its positions: the heavy lists (one segment only), then its units.
    unsigned g = 0, npos = 0;
    auto seg_end = [&](unsigned seg) { return n2 + min(sc.seg_units, sc.num_units - seg * sc.seg_units); };

    // position -> unit: an entry of list b, valid if b is still the unit's class (a unit can have been entered on a lighter
    // list before a neighbour raised it to a heavier one), or, in the light region, the unit itself if its class is light
    auto resolve = [&](unsigned p, unsigned& unit, bool& skip) {
        unit = 0u; skip = true;
        if (p < n2) {
            const unsigned b = p < n0 ? 0u : (p < n1 ? 1u : 2u);
            const unsigned k = p < n0 ? p : (p < n1 ? cap0 + (p - n0) : cap0 + cap1 + (p - n1));
            unit = cur_list[k];
            skip = cur_cls[unit] != b;
        } else if (p < npos) {
            unit = g * sc.seg_units + (p - n2);
            skip = false;
            if (sc.ordered) { const unsigned v = cur_cls[unit]; skip = v < 3u || v == done; }
        }
    };

    unsigned f = 0, take = 1u;
    // guided self-scheduling: half of an even share of what is left, between LIDAR_MIN_TAKE and LIDAR_CHUNK positions; one at a
    // time in the heavy lists, where a unit is long and balance matters most.  Not one at a time at the end of the light
    // region: a fetch is an L2 atomic's round trip plus the class lookup behind it (1.9 us when every unit pays it: unit
    // timeline with LIDAR_CHUNK 1), a light unit is 3.3 us, and all 7 104 warps asking after every unit is more than the
    // one counter serves (about 1.4 fetches per ns) -- two at a time costs 1.6 us of balance and was 3 % faster at 4096 envs.
    // with one segment the first position of every warp is its own index: the counter starts at 0 and a fetch returns
    // old + nwarps; with several, a warp's first position is a fetch from its home
    const bool one = sc.homes == 1u;
    const unsigned share = one ? nwarps : max(nwarps / sc.homes, 1u);     // warps per segment
    auto fetch = [&](unsigned at) {
        take = (npos - at) / (2u * share);
        take = at < n1 ? 1u : at < n2 ? LIDAR_LIST2_TAKE : take < LIDAR_MIN_TAKE ? LIDAR_MIN_TAKE : (take > (sc.ordered ? LIDAR_CHUNK : 2u * LIDAR_CHUNK) ? (sc.ordered ? LIDAR_CHUNK : 2u * LIDAR_CHUNK) : take);
        if (lane == 0) f = atomicAdd(sc.ctrl + CTRL_SEG + g * SEG_STRIDE, take) + (one ? nwarps : 0u);
    };
    unsigned pos, end;
    // The warp's segment is drained: claim a chunk of the nearest segment that is not, in the order home, home + 1,
    // home - 1, home + 2, ...; false once every segment is drained (counters only grow, so that is final).
    auto steal = [&]() -> bool {
        const unsigned Q = sc.homes;
        if (Q == 1u) return false;                 // the one queue's fetch has just come back empty
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        const unsigned h = sc.home_of_sm[smid & (F110_SMID_TABLE - 1u)];
        for (;;) {
            bool found = false;
            for (unsigned v0 = 0; v0 < Q && !found; v0 += 32u) {
                const unsigned v = v0 + lane, off = (v + 1u) >> 1;
                unsigned seg = (v & 1u) ? h + off : h + Q - off, at = 0u;
                seg = seg >= Q ? seg - Q : seg;
                bool open = false;
                if (v < Q) { at = __ldcg(sc.ctrl + CTRL_SEG + seg * SEG_STRIDE); open = at < seg_end(seg); }
                const unsigned m = __ballot_sync(0xffffffffu, open);
                if (m) {
                    found = true;
                    g = __shfl_sync(0xffffffffu, seg, __ffs(m) - 1);
                    npos = seg_end(g);
                    fetch(__shfl_sync(0xffffffffu, at, __ffs(m) - 1));
                }
            }
            if (!found) return false;
            pos = __shfl_sync(0xffffffffu, f, 0);
            end = pos + take;
            if (pos < npos) return true;
        }
    };
    if (one) {
        npos = seg_end(0u);
        pos = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
        end = pos + 1u;
    } else {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        g = sc.home_of_sm[smid & (F110_SMID_TABLE - 1u)];
        npos = seg_end(g);
        fetch(0u);
        pos = __shfl_sync(0xffffffffu, f, 0);
        end = pos + take;
    }
    unsigned unit; bool skip;
    resolve(pos, unit, skip);
    for (;;) {
        if (pos >= npos) {
            if (!steal()) break;
            resolve(pos, unit, skip);
        }
        unsigned nlook = 0;
        bool live = false, redone_here = false;
        unsigned npos_next, nunit; bool nskip;
        if (!skip) {
            unsigned t_start = 0;
            if (COUNT) asm volatile("mov.u32 %0, %%globaltimer_lo;" : "=r"(t_start));
            // ---- the unit's scan and this lane's beam
            const unsigned s = fast_div(unit, c.div_ups);
            const unsigned i = (unit - s * c.ups) * 32u + lane;
            const unsigned env = DIRECT ? s : fast_div(s, c.div_A);
            live = i < (unsigned)c.B && (LEAN || !(io.active_mask && !io.active_mask[env]));
            const unsigned ic = i < (unsigned)c.B ? i : (unsigned)c.B - 1u;      // the dead lanes of a scan's last unit shadow its last beam
            const double4 head = reinterpret_cast<const double4*>(sc.head)[s];   // fixed-point start X, Y; theta index of beam 0; iTTC limit
            const unsigned stepc = st.step_count[env];
            const int slot = MAPS ? ms.env_map[env] : 0;
            // beam direction: closed form of the reference's running sum theta_index += increment with wrap
            // (laser_models.py:174-184).  The running sum differs from the closed form by < 1.3e-10 after
            // 1080 adds; only when the value sits within 1e-9 of an integer can int() disagree, and then the
            // sum is replayed exactly.
            const double td = (double)c.theta_dis;
            double t = head.z + (double)ic * c.theta_inc;
            if (t >= td) t -= td;
            if (fabs(t - rint(t)) < 1e-9 || t >= td) {
                t = head.z;
                for (unsigned k = 0; k < ic; ++k) {
                    t += c.theta_inc;
                    while (t >= td) t -= td;
                }
            }
            int ti = (int)t;
            // memory safety only: a NaN yaw (a car poisoned by a NaN command) converts to a NEGATIVE index on this hardware
            ti = (unsigned)ti < (unsigned)c.theta_dis ? ti : c.theta_dis - 1;
            const double2 dir = __ldg((MAPS ? ms.dir_fx + (size_t)slot * (unsigned)c.theta_dis : c.dir_fx) + ti);
            const double ttc_lim = head.w;      // iTTC prefilter of the scan, formed by the dynamics kernel
            // the ray's id: its element of the observation when the scan goes there, and the counter of its noise.  The one
            // thing about the ray's place that the common path still needs after the march (< 2^32: f110_create bounds
            // NA * B by 2^31 and B >= 32).
            const unsigned rid = s * (unsigned)(c.B + 8) + i;

            // ---- the march
            double X = head.x, Y = head.y, total_d = 0.0, d = 0.0;
            {
                const unsigned fb = TUNED ? (unsigned)FB : m.fx_bits;
                const unsigned gm = TUNED ? (((1u << FB) - 1u) & ~3u) : m.guard_mask;
                const int pitch = TUNED ? (1 << (32 - FB)) + 16 : m.pitch;
                const double eps = c.eps;
                const double max_range = TUNED ? 30.0 : c.max_range;   // an immediate: 30.0 has no low mantissa word
                const size_t stride = TUNED ? (size_t)(1u << (32 - FB)) * (size_t)((1u << (32 - FB)) + 16u) : ms.stride;
                const double* __restrict__ dt = MAPS ? m.dt + (size_t)slot * stride : m.dt;
                // The loop is software-pipelined by one lookup: the cell of the NEXT position is loaded before it is known
                // whether the ray goes on (any 32-bit fixed-point coordinate addresses a cell of the padded array, so the
                // load is always safe).  The dependent chain of a lookup is then load -> multiply-add -> convert -> index ->
                // load; the range / eps / guard tests run beside the load instead of in front of it.  Cost: one extra
                // lookup per ray.
                bool decided = true;
                if (live) {
                    unsigned ux = __double2uint_rz(X), uy = __double2uint_rz(Y);
                    unsigned tx, ty;
                    // fraction's upper bits all ones <=> within guard of a cell edge (MapView.fx_off).  (~u & gm) != 0 as one
                    // LOP3 with a predicate result each; written in C, NVVM turns it into (u & gm) != gm: two instructions
                    asm("lop3.b32 %0, %1, %2, 0, 0x0c;" : "=r"(tx) : "r"(ux), "r"(gm));
                    asm("lop3.b32 %0, %1, %2, 0, 0x0c;" : "=r"(ty) : "r"(uy), "r"(gm));
                    decided = tx != 0u && ty != 0u;
                    if (decided) {
                        // Two lookups per trip, the roles of the two cell registers swapped between them: written as one
                        // lookup per trip, ptxas rotates (d, d_next) through four register moves -- 4 of the loop's 23
                        // instructions.  One exit test per lookup (ray ended OR lookup undecided; told apart after the
                        // loop, where `still going` means undecided), one counter update per trip.
                        double da = __ldg(dt + ((int)(uy >> fb) * pitch + (int)(ux >> fb))), db = 0.0;
                        unsigned trips = 0;
                        bool second = false;
#define F110_MARCH_STEP(D_CUR, D_NEXT)                                                                         \
                            X += D_CUR * dir.x;                                                                \
                            Y += D_CUR * dir.y;                                                                \
                            ux = __double2uint_rz(X);                                                          \
                            uy = __double2uint_rz(Y);                                                          \
                            D_NEXT = __ldg(dt + ((int)(uy >> fb) * pitch + (int)(ux >> fb)));                  \
                            total_d += D_CUR;                                                                  \
                            asm("lop3.b32 %0, %1, %2, 0, 0x0c;" : "=r"(tx) : "r"(ux), "r"(gm));                \
                            asm("lop3.b32 %0, %1, %2, 0, 0x0c;" : "=r"(ty) : "r"(uy), "r"(gm));
                        for (;;) {
                            F110_MARCH_STEP(da, db)
                            if (!((TUNED ? da > 0.0 : da > eps) && total_d <= max_range && tx != 0u && ty != 0u)) break;
                            F110_MARCH_STEP(db, da)
                            if (!((TUNED ? db > 0.0 : db > eps) && total_d <= max_range && tx != 0u && ty != 0u)) { second = true; break; }
                            ++trips;
                        }
#undef F110_MARCH_STEP
                        d = second ? db : da;
                        nlook = 2u * trips + (second ? 2u : 1u);
                        // the ray ended on this lookup (d is its last cell: a sentinel means it left the map), or it goes on
                        // and the lookup after it could not be decided
                        decided = !((TUNED ? d > 0.0 : d > eps) && total_d <= max_range);
                    }
                }
                if (live && (!decided || d < 0.0)) {
                    const double2 ex = trace_ray_exact(MAPS ? ms.views[slot] : m, c, sc, s, ti);
                    total_d = ex.x;
                    nlook = (unsigned)ex.y;
                    if (COUNT) { ++cnt_redone; redone_here = true; }
                }
                if (total_d > c.max_range) total_d = c.max_range;
            }

            // ---- the next position: inside the chunk, what it holds is loaded now and arrives while the epilogue runs; at
            // the end of a chunk the fetch is issued now and resolved after the epilogue.  (Not earlier: a position reserved
            // at the start of a unit waits for that unit, and behind a 70 us unit sat positions handed out at 5 us.)
            npos_next = pos + 1u;
            const bool chunk_end = npos_next >= end;
            if (chunk_end) fetch(pos);
            else resolve(npos_next, nunit, nskip);

            if (live) {
                // scan += noise, laser_models.py:450-452
                const unsigned r = OBS_ONLY ? 0u : rid - 8u * s;      // s * B + i: the ray's element of the scan outputs
                double range = total_d;
                if (!LEAN && io.noise) {
                    range += io.noise[r];
                } else if (c.noise_std > 0.0) {
                    // counter = (ray id, steps since the env's reset): like the reference's generator, which is re-seeded by
                    // reset (base_classes.py:204), the stream restarts with every episode; unlike it, every ray has its own
                    const uint2 bits = philox2x32_10(make_uint2(rid, stepc), c.philox_key);
                    range += c.noise_std * (double)gaussian_from_bits(bits.x, bits.y);
                }
                // The scan goes straight to the caller's buffers.  With opponents (A >= 2) the post kernel lowers the few
                // beams that hit another car afterwards, in those same buffers.
                // Streaming stores (evict-first): nothing in this kernel reads the outputs back, and at 32 768 envs the
                // 142 MB of observations would otherwise push the map out of L2 (2.5 % of the kernel there).
                if (!LEAN && io.scans_f64) __stcs(io.scans_f64 + r, range);
                if (!OBS_ONLY && io.scans_f32) __stcs(io.scans_f32 + r, (float)range);
                if (DIRECT) {
                    if (OBS_ONLY || io.obs) __stcs(io.obs + rid, obs_lidar<TUNED>(range, c.lidar_max, c.obs_rcp));
                } else {
                    if (io.obs && s == env * (unsigned)c.A)
                        __stcs(io.obs + (env * (unsigned)(c.B + 8) + i), obs_lidar<TUNED>(range, c.lidar_max, c.obs_rcp));
                }
                // check_ttc_jit (any-reduction; the reference's early break is irrelevant)
                if (!(range > ttc_lim)) {
                    // (rare: re-derive the ray's place and re-read its table rather than keep them alive across the march)
                    const unsigned s2 = fast_div(unit, c.div_ups), i2 = (unit - s2 * c.ups) * 32u + lane;
                    const double2 bt2 = __ldg(c.beam_tt + i2);       // beam cosine, side distance
                    const double ttc = (range - bt2.y) / (st.x[3][s2] * bt2.x);
                    if ((ttc < c.ttc_thresh) && (ttc >= 0.0)) sc.ttc_hit[s2] = 1;
                }
            }
            // ---- history for the next step's launch order.  The class goes to the unit AND its two neighbours in the scan: a
            // long (wall-grazing) ray wanders across the beam index as the car yaws, and the unit it moves into has no
            // history of its own -- 22 units per step with >= 48 lookups were predicted light, the longest ~120 lookups;
            // with the neighbours 0.1 and ~27 (4096-env C3 workload, 60 steps recorded).  Lanes 0..2 do one target each.
            const unsigned wmax = __reduce_max_sync(0xffffffffu, nlook);
            if (lane == 3u && sc.ordered) cur_cls[unit] = done;
            if (wmax >= HEAVY_T2 && lane < 3u && sc.ordered) {
                const unsigned b = wmax >= HEAVY_T0 ? 0u : (wmax >= HEAVY_T1 ? 1u : 2u);
                const unsigned k = unit - fast_div(unit, c.div_ups) * c.ups;
                const bool in_scan = lane == 1u || (lane == 0u ? k > 0u : k + 1u < c.ups);
                if (in_scan) {
                    const unsigned u = unit + lane - 1u;
                    if (atomicMin(next_cls + u, b) > b) {      // this call made b the unit's class: enter it on list b
                        const unsigned slot = atomicAdd(sc.ctrl + CTRL_NEXT + b * CTRL_NEXT_STRIDE, 1u);
                        if (slot < (b == 0 ? cap0 : (b == 1 ? cap1 : cap2))) next_list[(b == 0 ? 0u : (b == 1 ? cap0 : cap0 + cap1)) + slot] = u;
                        else atomicMax(next_cls + u, 3u);      // list full: back to light (whatever others do next stays consistent)
                    }
                }
            }
            if (chunk_end) {
                npos_next = __shfl_sync(0xffffffffu, f, 0);
                end = npos_next + take;
                resolve(npos_next, nunit, nskip);
            }
            if (COUNT) {
                const unsigned redo_lanes = __popc(__ballot_sync(0xffffffffu, redone_here));   // timeline: bits 24.. of the lookup word
                if (sc.timeline && lane == 0) {
                    unsigned t_end, smid;
                    asm volatile("mov.u32 %0, %%globaltimer_lo;" : "=r"(t_end));
                    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                    sc.timeline[unit] = make_uint4(t_start, t_end, wmax | (redo_lanes << 24), (smid << 24) | (pos & 0xFFFFFFu));
                }
                cnt_look += nlook;
                cnt_rays += live ? 1u : 0u;
                cnt_max = max(cnt_max, nlook);
            }
        } else {
            npos_next = pos + 1u;
            if (npos_next >= end) { fetch(pos); npos_next = __shfl_sync(0xffffffffu, f, 0); end = npos_next + take; }
            resolve(npos_next, nunit, nskip);
        }
        pos = npos_next; unit = nunit; skip = nskip;
    }
    if (COUNT) {
        const unsigned wsum = __reduce_add_sync(0xffffffffu, cnt_look);
        const unsigned wrays = __reduce_add_sync(0xffffffffu, cnt_rays);
        const unsigned wmax = __reduce_max_sync(0xffffffffu, cnt_max);
        const unsigned wredone = __reduce_add_sync(0xffffffffu, cnt_redone);
        if (lane == 0 && wrays) {
            atomicAdd(sc.lookups, (unsigned long long)wsum);
            atomicAdd(sc.lookups + 1, (unsigned long long)wrays);
            atomicMax(sc.lookups + 2, (unsigned long long)wmax);   // longest ray seen so far
            if (wredone) atomicAdd(sc.lookups + 3, (unsigned long long)wredone);
        }
    }
