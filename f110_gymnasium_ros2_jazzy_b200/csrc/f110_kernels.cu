// f110_kernels.cu -- the three sm_100a kernels of one batched F110Env step.
//
//   K1 dynamics_kernel : one thread per vehicle.  Steering-delay FIFO, bang-bang/P controller,
//                        fp64 single-track RK4 (or Euler), post clamps, lidar pose.
//                        (RaceCar.update_pose, base_classes.py:256-422)
//   K2 lidar_kernel    : one thread per beam, flat over all N*A*B rays.  Ray-march over the
//                        distance transform, + noise, per-beam iTTC test.
//                        (get_scan/trace_ray laser_models.py:106-186, scan :429-454,
//                         check_ttc_jit :188-217)
//   K3 post_kernel     : one CTA per env.  iTTC state zeroing, GJK over all pairs, opponent
//                        ray-cast, finish-zone/lap bookkeeping, done, observation packing.
//                        (base_classes.py:229-254,206-227,549-563,592-602; f110_env.py:310-352,552-602)
//
// Reference paths are relative to f110_gymnasium/gym/f110_gym/envs/.
// Compile with -fmad=false: the operator order below is the reference's, without contraction.
#include "f110_kernels.cuh"

#include <math.h>
#include <string.h>

namespace {

enum { P_MU = F110_P_MU, P_CSF = F110_P_C_SF, P_CSR = F110_P_C_SR, P_LF = F110_P_LF, P_LR = F110_P_LR,
       P_H = F110_P_H, P_M = F110_P_M, P_I = F110_P_I, P_SMIN = F110_P_S_MIN, P_SMAX = F110_P_S_MAX,
       P_SVMIN = F110_P_SV_MIN, P_SVMAX = F110_P_SV_MAX, P_VSWITCH = F110_P_V_SWITCH, P_AMAX = F110_P_A_MAX,
       P_VMIN = F110_P_V_MIN, P_VMAX = F110_P_V_MAX, P_WIDTH = F110_P_WIDTH, P_LENGTH = F110_P_LENGTH };

// ---------------------------------------------------------------- numpy scalar semantics

// np.clip(x, lo, hi) = min(max(x, lo), hi), NaN propagating
__device__ __forceinline__ double clipd(double x, double lo, double hi) {
    x = (x < lo) ? lo : x;
    x = (x > hi) ? hi : x;
    return x;
}

// Python float `a % b` for b > 0 (floored modulo)
__device__ __forceinline__ double floored_mod(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) {
        if (m < 0.0) m += b;
    } else {
        m = 0.0;
    }
    return m;
}

__device__ __forceinline__ double wrap_angle(double a) {  // base_classes.py:408, f110_env.py:548-550
    return floored_mod(a + F110_PI, 2 * F110_PI) - F110_PI;
}

// ---------------------------------------------------------------- vehicle model

struct VehParams {
    double mu, C_Sf, C_Sr, lf, lr, h, m, I, s_min, s_max, sv_min, sv_max, v_switch, a_max, v_min, v_max;
};

__device__ __forceinline__ VehParams load_params(const double* __restrict__ p) {
    VehParams v;
    v.mu = __ldg(p + P_MU); v.C_Sf = __ldg(p + P_CSF); v.C_Sr = __ldg(p + P_CSR); v.lf = __ldg(p + P_LF);
    v.lr = __ldg(p + P_LR); v.h = __ldg(p + P_H); v.m = __ldg(p + P_M); v.I = __ldg(p + P_I);
    v.s_min = __ldg(p + P_SMIN); v.s_max = __ldg(p + P_SMAX); v.sv_min = __ldg(p + P_SVMIN);
    v.sv_max = __ldg(p + P_SVMAX); v.v_switch = __ldg(p + P_VSWITCH); v.a_max = __ldg(p + P_AMAX);
    v.v_min = __ldg(p + P_VMIN); v.v_max = __ldg(p + P_VMAX);
    return v;
}

// accl_constraints, dynamic_models.py:29-60
__device__ __forceinline__ double accl_constraints(double vel, double accl, const VehParams& p) {
    double pos_limit = (vel > p.v_switch) ? p.a_max * p.v_switch / vel : p.a_max;
    if ((vel <= p.v_min && accl <= 0) || (vel >= p.v_max && accl >= 0)) accl = 0.;
    else if (accl <= -p.a_max) accl = -p.a_max;
    else if (accl >= pos_limit) accl = pos_limit;
    return accl;
}

// steering_constraint, dynamic_models.py:62-87
__device__ __forceinline__ double steering_constraint(double sa, double sv, const VehParams& p) {
    if ((sa <= p.s_min && sv <= 0) || (sa >= p.s_max && sv >= 0)) sv = 0.;
    else if (sv <= p.sv_min) sv = p.sv_min;
    else if (sv >= p.sv_max) sv = p.sv_max;
    return sv;
}

// vehicle_dynamics_st (with the embedded vehicle_dynamics_ks branch), dynamic_models.py:90-176
__device__ __forceinline__ void vehicle_dynamics_st(const double (&x)[7], double u_sv, double u_accl,
                                                    const VehParams& p, double (&f)[7]) {
    const double g = 9.81;
    const double u0 = steering_constraint(x[2], u_sv, p);
    const double u1 = accl_constraints(x[3], u_accl, p);
    if (fabs(x[3]) < 0.5) {
        // kinematic branch :152-160; vehicle_dynamics_ks re-applies the (idempotent) constraints :112
        const double lwb = p.lf + p.lr;
        const double k0 = steering_constraint(x[2], u0, p);
        const double k1 = accl_constraints(x[3], u1, p);
        double s4, c4;
        sincos(x[4], &s4, &c4);
        const double t2 = tan(x[2]);
        const double c2 = cos(x[2]);
        f[0] = x[3] * c4;
        f[1] = x[3] * s4;
        f[2] = k0;
        f[3] = k1;
        f[4] = x[3] / lwb * t2;
        f[5] = u1 / lwb * t2 + x[3] / (lwb * (c2 * c2)) * u0;
        f[6] = 0.0;
    } else {
        double sb, cb;
        sincos(x[6] + x[4], &sb, &cb);
        const double lrlf = p.lr + p.lf;
        const double glr = g * p.lr - u1 * p.h;   // (g*lr - u[1]*h)
        const double glf = g * p.lf + u1 * p.h;   // (g*lf + u[1]*h)
        f[0] = x[3] * cb;
        f[1] = x[3] * sb;
        f[2] = u0;
        f[3] = u1;
        f[4] = x[5];
        f[5] = -p.mu * p.m / (x[3] * p.I * lrlf) * (p.lf * p.lf * p.C_Sf * glr + p.lr * p.lr * p.C_Sr * glf) * x[5]
             + p.mu * p.m / (p.I * lrlf) * (p.lr * p.C_Sr * glf - p.lf * p.C_Sf * glr) * x[6]
             + p.mu * p.m / (p.I * lrlf) * p.lf * p.C_Sf * glr * x[2];
        f[6] = (p.mu / (x[3] * x[3] * lrlf) * (p.C_Sr * glf * p.lr - p.C_Sf * glr * p.lf) - 1) * x[5]
             - p.mu / (x[3] * lrlf) * (p.C_Sr * glf + p.C_Sf * glr) * x[6]
             + p.mu / (x[3] * lrlf) * (p.C_Sf * glr) * x[2];
    }
}

// pid, dynamic_models.py:178-221
__device__ __forceinline__ void pid(double speed, double steer, double cur_speed, double cur_steer,
                                    const VehParams& p, double& accl, double& sv) {
    const double steer_diff = steer - cur_steer;
    if (fabs(steer_diff) > 1e-4) sv = (steer_diff / fabs(steer_diff)) * p.sv_max;
    else sv = 0.0;
    const double vel_diff = speed - cur_speed;
    double kp;
    if (cur_speed > 0.) {
        kp = (vel_diff > 0) ? 10.0 * p.a_max / p.v_max : 10.0 * p.a_max / (-p.v_min);
    } else {
        kp = (vel_diff > 0) ? 2.0 * p.a_max / p.v_max : 2.0 * p.a_max / (-p.v_min);
    }
    accl = kp * vel_diff;
}

// ---------------------------------------------------------------- K1: dynamics

// MAPS: the handle holds a map set; the scan head is formed in the frame of the env's own map (its slot's MapView) with the
// set's common fx_off.  Shared by dynamics_kernel (one map) and dynamics_maps_kernel.
template <bool MAPS>
__device__ __forceinline__ void dynamics_body(const SimConst& c, const MapView& m, const SimState& st, const StepScratch& sc,
                                              const F110StepIO& io, const MapSet& ms) {
    cudaGridDependencySynchronize();   // PDL: the previous step's post kernel (or whatever precedes in the stream) is done
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    // Every global load this thread needs is issued before the first store or branch that depends on one: the kernel is a
    // single dependent chain per thread, and with a cold L2 each load left in program order behind a branch costs a DRAM
    // round trip of its own (the masks, the state, the action and the parameters were four in a row).
    const bool veh = s < c.NA;
    const int env = veh ? s / c.A : 0;
    const int a = s - env * c.A;
    uint8_t active = 1, rst_flag = 0;
    double xl[7] = {0., 0., 0., 0., 0., 0., 0.}, b0 = 0., b1 = 0., px = 0., py = 0., pth = 0.;
    int cnt = 0;
    double raw_steer = 0., speed = 0.;
    int slot = 0;
    if (veh) {
        if (MAPS) slot = ms.env_map[env];
        if (io.active_mask) active = io.active_mask[env];
        if (io.reset_mask) {
            rst_flag = io.reset_mask[env];
            const double* ps = io.reset_poses + (size_t)s * 3;
            px = ps[0]; py = ps[1]; pth = ps[2];
        }
#pragma unroll
        for (int k = 0; k < 7; ++k) xl[k] = st.x[k][s];
        b0 = st.steer_buf0[s]; b1 = st.steer_buf1[s];
        cnt = st.steer_cnt[s];
        if (io.actions) {
            if (io.actions_f64) {
                const double2 v = reinterpret_cast<const double2*>(io.actions)[s];
                raw_steer = v.x; speed = v.y;
            } else {
                const float2 v = reinterpret_cast<const float2*>(io.actions)[s];
                raw_steer = (double)v.x; speed = (double)v.y;
            }
        }
    }
    const VehParams p = load_params(c.params + (veh ? a : 0) * F110_NUM_PARAMS);

    const bool run = veh && active;
    const bool rst = run && rst_flag != 0;
    if (run) {
    double x[7];
    if (rst) {
        // F110Env.reset bookkeeping (f110_env.py:440-451) + RaceCar.reset (base_classes.py:183-204)
        x[0] = px; x[1] = py; x[2] = 0.; x[3] = 0.; x[4] = pth; x[5] = 0.; x[6] = 0.;
        b0 = b1 = 0.;
        cnt = 0;
        st.start_x[s] = px; st.start_y[s] = py; st.start_th[s] = pth;
        st.near_start[s] = 1;
        st.toggles[s] = 0;
        st.collisions[s] = 0;
        if (a == c.ego) {
            const double th = -pth;
            st.rot_c[env] = cos(th);
            st.rot_s[env] = sin(th);
        }
        if (a == 0) { st.time[env] = 0.0; st.step_count[env] = 0u; }
        raw_steer = 0.; speed = 0.;   // the reset's own step uses a zero action (f110_env.py:457-458)
    } else {
#pragma unroll
        for (int k = 0; k < 7; ++k) x[k] = xl[k];
        if (a == 0) st.step_count[env] += 1u;
    }

    // steering delay FIFO, base_classes.py:270-278
    double steer;
    if (cnt < 2) { steer = 0.; cnt += 1; }
    else steer = b1;
    b1 = b0; b0 = raw_steer;

    double accl, sv;
    pid(speed, steer, x[3], x[2], p, accl, sv);
    sv = clipd(sv, p.sv_min, p.sv_max);         // :283
    accl = clipd(accl, -p.a_max, p.a_max);      // :284

    const double dt = c.timestep;
    if (c.integrator == F110_INTEGRATOR_RK4) {  // :285-374
        // One copy of the right-hand side, run four times, instead of four inlined copies: the kernel's instruction
        // stream is fetched cold by every SM, and the stages cannot overlap anyway.  Bit-identical to the reference's
        // unrolled form: k/2 == k*0.5 and 2*k are exact, k*1.0 == k, and k1 + 2*k2 + 2*k3 + k4 is summed left to right.
        double sum[7], xs[7], k[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) { xs[i] = x[i]; sum[i] = 0.; }
#pragma unroll 1
        for (int stage = 0; stage < 4; ++stage) {
            vehicle_dynamics_st(xs, sv, accl, p, k);
            const double wgt = (stage == 1 || stage == 2) ? 2.0 : 1.0;    // weight in the final sum
            const double half = stage < 2 ? 0.5 : 1.0;                    // k/2 for the two midpoint stages, k for the last
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                sum[i] = stage == 0 ? k[i] : sum[i] + wgt * k[i];
                xs[i] = x[i] + dt * (k[i] * half);
            }
        }
        const double w = dt * (1.0 / 6.0);
#pragma unroll
        for (int i = 0; i < 7; ++i) x[i] = x[i] + w * sum[i];
    } else {                                    // Euler :376-396
        double f[7];
        vehicle_dynamics_st(x, sv, accl, p, f);
#pragma unroll
        for (int i = 0; i < 7; ++i) x[i] = x[i] + dt * f[i];
    }

    // post clamps :400-417
    x[2] = clipd(x[2], p.s_min, p.s_max);
    x[3] = clipd(x[3], p.v_min, p.v_max);
    x[4] = wrap_angle(x[4]);
    const double YAW_RATE_CAP = 10.0;
    if (x[5] != x[5]) x[5] = 0.0;
    else if (isinf(x[5])) x[5] = x[5] > 0 ? YAW_RATE_CAP : -YAW_RATE_CAP;
    x[5] = clipd(x[5], -YAW_RATE_CAP, YAW_RATE_CAP);
    const double SLIP_CAP = 60 * (F110_PI / 180.0);
    if (x[6] != x[6]) x[6] = 0.0;
    x[6] = clipd(x[6], -SLIP_CAP, SLIP_CAP);

#pragma unroll
    for (int k = 0; k < 7; ++k) st.x[k][s] = x[k];
    st.steer_buf0[s] = b0; st.steer_buf1[s] = b1;
    st.steer_cnt[s] = cnt;

    // lidar pose :420-422 and the wrapped index of beam 0 (laser_models.py:167-172)
    double sx = x[0], sy = x[1];
    if (c.lidar_dist != 0.0) {
        double sn, cs;
        sincos(x[4], &sn, &cs);
        sx = x[0] + c.lidar_dist * cs;
        sy = x[1] + c.lidar_dist * sn;
    }
    sc.scan_x[s] = sx; sc.scan_y[s] = sy; sc.pre_yaw[s] = x[4];
    double ti = (double)c.theta_dis * (x[4] - c.fov / 2.) / (2. * F110_PI);
    ti = fmod(ti, (double)c.theta_dis);
    while (ti < 0) ti += (double)c.theta_dis;
    // what the lidar kernel needs of this scan, in one 32-byte record: the start of the march in fixed-point map
    // coordinates (xy_2_rc's translate / rotate, laser_models.py:66-77, then the scale 2^F / res), theta index of beam 0, speed
    const MapView& mv = MAPS ? ms.views[slot] : m;
    const double x_trans = sx - mv.ox, y_trans = sy - mv.oy;
    double4 head;
    head.x = (x_trans * mv.oc + y_trans * mv.os) * mv.inv_fx + m.fx_off;
    head.y = (-x_trans * mv.os + y_trans * mv.oc) * mv.inv_fx + m.fx_off;
    head.z = ti;
    // iTTC prefilter for the whole scan (check_ttc_jit, laser_models.py:205-213): ttc = (range - side) / (v cos) lies in
    // [0, thresh) only if range - side <= thresh |v cos|, so a range above max(side) + 2.5 thresh |v| max|cos| (the margin
    // swallows every rounding) cannot hit on ANY beam, and neither can a car at rest (the reference tests vel != 0 first).
    // NaN compares false in the lidar kernel's `range > limit` and falls through to the exact test.
    head.w = x[3] != 0.0 ? c.ttc_side_max + 2.5 * c.ttc_thresh * fabs(x[3]) * c.ttc_cos_max : -INFINITY;
    reinterpret_cast<double4*>(sc.head)[s] = head;
    sc.ttc_hit[s] = 0;
    }   // run

    // The launch order the lidar kernel is about to use classes a scan's units by their rays of the PREVIOUS step; for a
    // vehicle reset in this step those were taken from a pose that no longer exists.  A long unit met in the light region
    // would extend the lidar kernel's tail by its whole length, so every unit of a reset scan that is not on a list already
    // joins the third one (cost if it turns out short: none).  The warp does this together, lane k for units k, k + 32, ...
    // of each reset scan in turn, with one atomic per 32 units; a list that is full leaves the rest where it is.  When most
    // of the warp was reset (a global reset) the history is void anyway and nothing is done.
    const unsigned lane = threadIdx.x & 31u;
    unsigned rst_mask = __ballot_sync(0xffffffffu, rst);
    if (sc.ordered && rst_mask != 0u && __popc(rst_mask) <= 8) {
        const unsigned par = sc.ctrl[CTRL_EPOCH] & 1u;
        unsigned* cls = par ? sc.cls[1] : sc.cls[0];
        unsigned* list2 = (par ? sc.list[1] : sc.list[0]) + sc.cap[0] + sc.cap[1];
        while (rst_mask) {
            const int j = __ffs(rst_mask) - 1;
            rst_mask &= rst_mask - 1u;
            const unsigned sj = (unsigned)__shfl_sync(0xffffffffu, s, j);
            for (unsigned k0 = 0; k0 < c.ups; k0 += 32u) {
                const unsigned k = k0 + lane;
                const unsigned unit = sj * c.ups + k;
                const bool light = k < c.ups && cls[unit] >= 3u;
                const unsigned m_light = __ballot_sync(0xffffffffu, light);
                if (m_light == 0u) continue;
                unsigned base = 0;
                if (lane == 0) base = atomicAdd(sc.ctrl + CTRL_CUR + 2, (unsigned)__popc(m_light));
                base = __shfl_sync(0xffffffffu, base, 0);
                const unsigned slot = base + (unsigned)__popc(m_light & ((1u << lane) - 1u));
                if (light && slot < sc.cap[2]) { list2[slot] = unit; cls[unit] = 2u; }   // the lidar kernel clamps the count to cap[2]
            }
        }
    }
}

__global__ void __launch_bounds__(128) dynamics_kernel(SimConst c, MapView m, SimState st, StepScratch sc, F110StepIO io) {
    dynamics_body<false>(c, m, st, sc, io, MapSet());
}

__global__ void __launch_bounds__(128) dynamics_maps_kernel(SimConst c, MapView m, SimState st, StepScratch sc, F110StepIO io,
                                                            MapSet ms) {
    dynamics_body<true>(c, m, st, sc, io, ms);
}

// Simulator.reset alone (base_classes.py:627-643): poses only, no step, env bookkeeping untouched
__global__ void sim_reset_kernel(SimConst c, SimState st, const double* __restrict__ poses, const uint8_t* __restrict__ mask) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= c.NA) return;
    const int env = s / c.A;
    if (mask && !mask[env]) return;
    const double* ps = poses + (size_t)s * 3;
    st.x[0][s] = ps[0]; st.x[1][s] = ps[1]; st.x[2][s] = 0.; st.x[3][s] = 0.;
    st.x[4][s] = ps[2]; st.x[5][s] = 0.; st.x[6][s] = 0.;
    st.steer_buf0[s] = 0.; st.steer_buf1[s] = 0.; st.steer_cnt[s] = 0;
    if (s - env * c.A == 0) st.step_count[env] = 0u;
}

// ---------------------------------------------------------------- K2: lidar

// xy_2_rc, laser_models.py:55-86 -- the exact restatement (two IEEE divisions) on map-frame coordinates; returns the index
// into the padded device array.  Only trace_ray_exact calls it.
// (A float->int conversion of NaN does not give 0 on this hardware -- (int)NaN is negative -- hence the two-sided clamp.)
__device__ __forceinline__ int cell_index_exact(const MapView& m, double x_rot, double y_rot) {
    int flat;
    if (x_rot < 0 || x_rot >= m.wres || y_rot < 0 || y_rot >= m.hres) {
        flat = m.last;   // (r, c) = (-1, -1): numba wraps the negative indices to dt[H-1][W-1]
    } else {
        const int col = (int)(x_rot / m.res);
        const int row = (int)(y_rot / m.res);
        // numba indexes the flat buffer unchecked: col == W (x_rot one ulp under W*res) lands on the next row's first cell.
        // The clamp is memory safety for NaN poses.
        flat = row * m.W + col;
        flat = flat < 0 ? 0 : (flat > m.last ? m.last : flat);
    }
    const int row = flat / m.W;
    return (row + 1) * m.pitch + (flat - row * m.W) + 1;   // the map sits at [1 + r][1 + c] of the padded array
}

// trace_ray, laser_models.py:106-146, in the reference's own arithmetic from the ray's first lookup: world-frame march,
// translate and rotate per lookup.  Out of line: the lidar kernel calls it for the few rays per hundred thousand whose fast
// march met a lookup it could not decide (guard band, map border and beyond, non-finite coordinates).  Such a ray may be
// the longest of its launch, so this path must not be slow either: a lookup's cell is still taken from the fixed-point
// conversion of THIS lookup's exact map-frame position (one multiply-add away from the reference's quotient: < 1e-5
// units, no accumulated drift) whenever its fraction clears the guard band, and only the others -- and the lookups that
// land on a sentinel, i.e. off the map -- pay the reference's two IEEE divisions.
// -> (total distance before the clamp to max_range, number of lookups)
__device__ __noinline__ double2 trace_ray_exact(const MapView& m, const SimConst& c, const StepScratch& sc, unsigned s, int ti) {
    double x = sc.scan_x[s], y = sc.scan_y[s];
    const double sn = __ldg(c.sines + ti), cs = __ldg(c.cosines + ti);
    const double eps = c.eps, max_range = c.max_range;
    double total = 0.0;
    unsigned n = 0;
    for (;;) {
        const double x_trans = x - m.ox;
        const double y_trans = y - m.oy;
        const double x_rot = x_trans * m.oc + y_trans * m.os;
        const double y_rot = -x_trans * m.os + y_trans * m.oc;
        const unsigned ux = __double2uint_rz(x_rot * m.inv_fx + m.fx_off);
        const unsigned uy = __double2uint_rz(y_rot * m.inv_fx + m.fx_off);
        double d = -1.0;
        if ((~ux & m.guard_mask) != 0u && (~uy & m.guard_mask) != 0u)
            d = __ldg(m.dt + ((int)(uy >> m.fx_bits) * m.pitch + (int)(ux >> m.fx_bits)));
        if (d < 0.0) d = __ldg(m.dt + cell_index_exact(m, x_rot, y_rot));
        total += d;
        ++n;
        if (!(d > eps && total <= max_range)) break;
        x += d * cs;
        y += d * sn;
    }
    return make_double2(total, (double)n);
}

// Philox2x32-10 (Salmon et al. 2011), counter-based: no per-ray generator state in HBM.  One call yields the
// 64 bits one Box-Muller sample needs, at half the integer multiplies of Philox4x32.  The ten round keys
// (key + r * 0x9E3779B9) come precomputed from the host.
__device__ __forceinline__ uint2 philox2x32_10(uint2 ctr, const uint32_t (&key)[10]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi = __umulhi(0xD256D193u, ctr.x), lo = 0xD256D193u * ctr.x;
        ctr = make_uint2(hi ^ key[r] ^ ctr.y, lo);
    }
    return ctr;
}

// N(0, 1) from 48 random bits, Box-Muller on the SFU: u1, u2 in (0, 1) with 24 bits each, sqrt(-2 ln u1) cos(2 pi u2)
// through lg2.approx / sqrt.approx / cos.approx (relative errors ~1e-6: far below the 1 % noise the sample scales).
__device__ __forceinline__ float gaussian_from_bits(uint32_t a, uint32_t b) {
    const float u1 = fmaf((float)(a >> 8), 1.0f / 16777216.0f, 0.5f / 16777216.0f);
    const float u2 = fmaf((float)(b >> 8), 1.0f / 16777216.0f, 0.5f / 16777216.0f);
    float l2, rad;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(-1.3862943611198906f * l2));   // -2 ln 2 * log2(u1)
    return rad * __cosf(6.28318530717958647692f * u2);
}

// n / d for a run-time d through the multiply-shift pair the host precomputed (Granlund & Montgomery 1994)
__device__ __forceinline__ unsigned fast_div(unsigned n, FastDiv d) {
    const unsigned t = __umulhi(n, d.mul);
    return (t + ((n - t) >> d.sh1)) >> d.sh2;
}

// _pack_flat_obs lidar channel, f110_env.py:557-560: clip(nan_to_num(float32(range)), 0, lm) / lm
// FAST: lm == 30.0f.  rf / 30 through the reciprocal and two fused corrections equals the IEEE quotient for every
// float in [2^-120, 30] and for 0 (all 1 106 247 681 bit patterns of [0, 30] checked on the host, tools/checks/div30_check.c;
// the 279 620 mismatches all lie below 2^-125, where the quotient is subnormal) -- 3 instructions instead of ~15.
template <bool FAST>
__device__ __forceinline__ float obs_lidar(double range, float lm, float rcp) {
    float rf = (float)range;
    rf = rf != rf ? lm : rf;                 // nan -> lm; +inf -> lm and -inf -> 0 fall out of the clip
    rf = fminf(fmaxf(rf, 0.0f), lm);
    if (FAST && (rf == 0.0f || rf >= 7.5e-37f)) {
        const float q0 = rf * rcp;
        return fmaf(fmaf(-q0, lm, rf), rcp, q0);
    }
    return rf / lm;
}

// A unit's class for the next step's launch order, from the longest ray (in lookups) of its 32
#ifndef HEAVY_T0
#define HEAVY_T0 96u
#endif
#ifndef HEAVY_T1
#define HEAVY_T1 48u
#endif
#ifndef HEAVY_T2
#define HEAVY_T2 24u
#endif
#ifndef LIDAR_THREADS_OVERRIDE
#define LIDAR_THREADS_OVERRIDE 128
#endif
constexpr int LIDAR_THREADS = LIDAR_THREADS_OVERRIDE;
#ifndef LIDAR_MIN_BLOCKS
#define LIDAR_MIN_BLOCKS 12
#endif
#ifndef LIDAR_CHUNK_OVERRIDE
#define LIDAR_CHUNK_OVERRIDE 4
#endif
#ifndef LIDAR_LIST2_TAKE
#define LIDAR_LIST2_TAKE 2u    // positions per fetch in the third (lightest) heavy list (1 in the two heavier ones)
#endif
#ifndef LIDAR_MIN_TAKE
#define LIDAR_MIN_TAKE 2u     // positions per fetch in the last stretch of the light region (see `fetch`)
#endif
constexpr unsigned LIDAR_CHUNK = LIDAR_CHUNK_OVERRIDE;   // queue positions a warp takes per fetch in the bulk of the light region

// K2.  One thread per beam; a UNIT is 32 consecutive beams of one scan (the last unit of a scan is partly empty: 1080
// beams = 33.75 units), so everything that belongs to the scan -- its start in map coordinates, theta index, speed, noise
// counter, which K1 left in one 32-byte ScanHead -- is one broadcast load per warp.  A warp takes units from a device-wide
// queue until it is empty.
//
// * The march (trace_ray, laser_models.py:129-144) runs in FIXED-POINT MAP COORDINATES: X = x_rot * 2^F / res is advanced
//   by d * DX per step, DX = (direction rotated into the map frame) * 2^F / res read from a table set_map prepared,
//   instead of being recomputed from the world-frame position: no translate / rotate / scale per lookup (4 fp64
//   operations, 2 of them on the dependent chain), no in-map test (the map is padded with sentinels, see MapView).
//   X drifts from the reference's own rounded quotient by < 2e-6 fixed-point units per step (both are roundings of the
//   same real recurrence as long as they have visited the same cells, and every product and sum involved is below 2^32
//   with a 2^-53 relative rounding), so after any number of steps a ray can take (total <= 30 m in steps > 1e-4 m:
//   < 3e5) the two are less than one unit apart.  A lookup whose fixed-point fraction is at least m.guard (>= 2) units
//   away from both cell edges therefore addresses exactly the reference's cell; since every d read is then the
//   reference's, `total` is the reference's bit for bit.  The coordinates carry an offset of one cell minus the guard, so
//   that the guard test is one mask per axis (fraction's upper bits all set <=> within guard of either edge).  Any other
//   lookup is not decided here: negative and NaN coordinates convert to 0 (row / column 0 of the padded map: sentinels),
//   huge ones to 0xFFFFFFFF (inside the guard band), a coordinate beyond the map reads a sentinel, and in each case the
//   ray is redone from its first lookup by trace_ray_exact.
// * TUNED variants (FB = the map's fraction bits as a compile-time constant, for 19..22 bits = maps of 1 023 to 8 190 cells
//   a side; default eps test; lidar_max 30): ptxas re-loads every kernel parameter the loop uses from the constant bank
//   on EVERY iteration (7 of 30 instructions, and for a lone long ray their latency sits on the dependent chain: 590
//   cycles per lookup measured, against 270 for the L2 hit itself).  With the shifts, masks and pitch as immediates, the
//   eps test as d > 0 (valid when the smallest positive cell exceeds eps, which set_map checks) and max_range = 30 as an
//   immediate too, the loop has no constant load left (ptxas cannot be talked out of them: values made opaque with a
//   zero it cannot know are still re-derived inside the loop, whatever the register budget).  The generic variant (FB = 0) handles everything else,
//   and counts lookups for the roofline.
// * Persistent warps (the grid is one wave: SMs x resident CTAs).  With one CTA per 128 rays a CTA's slot is only
//   re-used when its slowest warp is through, and ray lengths are heavy-tailed (median 4 lookups, p99 42, max ~300 on
//   the Shanghai map): 60 % of the warp slots were occupied where the register file allows 75 %.
// * Longest-first order.  A ray's length changes little from one step to the next, so every unit is classed by its
//   longest ray (>= 96 / 48 / 24 lookups, else light) and the next step's queue serves the three heavy lists first, then
//   the light units in natural order (skipping the listed ones).  The kernel's tail is then made of light units.
//   Only the order depends on this history, never a result.  The lists are double-buffered by a parity word in device
//   memory which the post kernel flips, so a captured CUDA graph replays correctly.  The units of an env that K1 has just
//   reset have no usable history: K1 appends them to the third list (see dynamics_kernel).
// * The queue is one atomic counter (same-address atomics retire at about one per ns on this part: one fetch per unit
//   costs 45 % at 32 768 envs); a fetch takes up to LIDAR_CHUNK positions at a time in the bulk of the light region, one
//   near the ends, and is issued after the march of the chunk's last unit, so that its latency hides behind the epilogue.
// * Home segments, in launches without the longest-first order (more than 48 units per resident warp).  The units are cut
//   into sc.homes contiguous segments, one per SM, each with its own counter; a warp serves the segment of its SM (%smid
//   through sc.home_of_sm) and, once that is drained, the nearest one that is not (home + 1, home - 1, home + 2, ...: 32
//   looked at per round trip), and ends when every segment is drained.  Env order is track order (workloads.start_poses;
//   auto-reset returns a car to its own start), so the cars of a segment see the same walls and the map lines its warps
//   march stay in the SM's L1 (tools/locality_study.py).  Where the CTAs land only changes the order.  With one segment
//   the queue is the one above.  Smaller launches keep one: a warp's first position then costs no fetch, and at the end
//   no warp looks through other segments (DESIGN.md section 9).
// MODE 0: opponents follow (A >= 2); 1: single agent, the scan goes straight to the outputs; 2: single agent and the float32
// observation is the only scan output, noise from the device stream, no mask of active envs -- the bulk throughput case
// (BASELINE configs 3 / 4) -- without the unit's tests and address arithmetic for what is not there; 3: opponents, likewise
// lean (device noise, no fp64 scan output, no mask: BASELINE config 5).
// MAPS: the handle holds a map set (lidar_maps_kernel).  Per unit the env's slot is read in the same round as the scan head
// and the step count (all three are indexed from the unit alone); the slot's cell base is arithmetic from it (the blocks
// lie at a fixed stride), its direction table one level later, as the table of a single map is; the exact path reads the
// slot's MapView from global memory.  Everything else -- queue, lists, home segments -- is the single-map kernel's.
template <int FB, bool COUNT, int MODE>
__global__ void __launch_bounds__(LIDAR_THREADS, LIDAR_MIN_BLOCKS)
lidar_kernel(const __grid_constant__ SimConst c, const __grid_constant__ MapView m, const __grid_constant__ SimState st,
             const __grid_constant__ StepScratch sc, const __grid_constant__ F110StepIO io) {
    constexpr bool MAPS = false;
    const MapSet ms = {};
#include "f110_lidar_body.cuh"
}

// K2 for a map set: m is the set's common view (fraction bits, pitch, guard; dt = slot 0's block; min_positive over the set)
template <int FB, bool COUNT, int MODE>
__global__ void __launch_bounds__(LIDAR_THREADS, LIDAR_MIN_BLOCKS)
lidar_maps_kernel(const __grid_constant__ SimConst c, const __grid_constant__ MapView m, const __grid_constant__ SimState st,
                  const __grid_constant__ StepScratch sc, const __grid_constant__ F110StepIO io, const __grid_constant__ MapSet ms) {
    constexpr bool MAPS = true;
#include "f110_lidar_body.cuh"
}

// ---------------------------------------------------------------- K3: post

// End of a step's lidar bookkeeping, done by the post kernel: its threads rewind the segments' queues (one each), thread 0
// latches the recorded counts and flips the parity.  Everything it touches was written by the lidar kernel, which is
// complete before the post kernel's first instruction (cudaGridDependencySynchronize), and is next read by the following
// step's kernels, which wait for this grid in the same way -- no fence, no ticket.
__device__ __forceinline__ void latch_launch_order(const StepScratch& sc) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    for (unsigned g = t; g < sc.homes; g += gridDim.x * blockDim.x) sc.ctrl[CTRL_SEG + g * SEG_STRIDE] = 0u;
    if (t != 0) return;
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const unsigned n = sc.ctrl[CTRL_NEXT + b * CTRL_NEXT_STRIDE];
        sc.ctrl[CTRL_NEXT + b * CTRL_NEXT_STRIDE] = 0u;
        sc.ctrl[CTRL_CUR + b] = n < sc.cap[b] ? n : sc.cap[b];
    }
    sc.ctrl[CTRL_EPOCH] += 1u;
}

// get_trmtx + get_vertices, collision_models.py:218-260; order rl, rr, fr, fl
__device__ __forceinline__ void get_vertices(double px, double py, double yaw, double length, double width, double* v) {
    double sn, cs;
    sincos(yaw, &sn, &cs);
    const double hx[4] = { -length / 2, -length / 2, length / 2, length / 2 };
    const double hy[4] = { width / 2, -width / 2, -width / 2, width / 2 };
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[2 * k] = cs * hx[k] + (-sn) * hy[k] + px;
        v[2 * k + 1] = sn * hx[k] + cs * hy[k] + py;
    }
}

__device__ __forceinline__ int furthest_point(const double* v, double dx, double dy) {  // np.argmax: first maximum
    int best = 0;
    double bv = v[0] * dx + v[1] * dy;
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        const double d = v[2 * k] * dx + v[2 * k + 1] * dy;
        if (d > bv) { bv = d; best = k; }
    }
    return best;
}

__device__ __forceinline__ void gjk_support(const double* v1, const double* v2, double dx, double dy, double& ox, double& oy) {
    const int i = furthest_point(v1, dx, dy);
    const int j = furthest_point(v2, -dx, -dy);
    ox = v1[2 * i] - v2[2 * j];
    oy = v1[2 * i + 1] - v2[2 * j + 1];
}

// tripleProduct(a, b, c) = b*(a.c) - a*(b.c), collision_models.py:52-64
__device__ __forceinline__ void triple_product(double ax, double ay, double bx, double by, double cx, double cy,
                                               double& ox, double& oy) {
    const double ac = ax * cx + ay * cy;
    const double bc = bx * cx + by * cy;
    ox = bx * ac - ax * bc;
    oy = by * ac - ay * bc;
}

// collision (GJK), collision_models.py:113-182
__device__ bool gjk_collision(const double* v1, const double* v2) {
    double s0x, s0y, s1x = 0., s1y = 0.;   // simplex rows 0 and 1 (row 2 is always the newest point a)
    double dx = (v1[0] + v1[2] + v1[4] + v1[6]) / 4 - (v2[0] + v2[2] + v2[4] + v2[6]) / 4;
    double dy = (v1[1] + v1[3] + v1[5] + v1[7]) / 4 - (v2[1] + v2[3] + v2[5] + v2[7]) / 4;
    if (dx == 0 && dy == 0) dx = 1.0;
    double ax, ay;
    gjk_support(v1, v2, dx, dy, ax, ay);
    s0x = ax; s0y = ay;
    if (dx * ax + dy * ay <= 0) return false;
    dx = -ax; dy = -ay;
    int index = 0;
    for (int iter = 0; iter < 1000;) {
        gjk_support(v1, v2, dx, dy, ax, ay);
        index += 1;
        if (dx * ax + dy * ay <= 0) return false;
        const double aox = -ax, aoy = -ay;
        if (index < 2) {
            s1x = ax; s1y = ay;
            const double abx = s0x - ax, aby = s0y - ay;
            triple_product(abx, aby, aox, aoy, abx, aby, dx, dy);
            if (sqrt(dx * dx + dy * dy) < 1e-10) { dx = aby; dy = -1 * abx; }
            continue;   // the reference does not count this pass (:154-160)
        }
        const double abx = s1x - ax, aby = s1y - ay;
        const double acx = s0x - ax, acy = s0y - ay;
        double px, py;
        triple_product(abx, aby, acx, acy, acx, acy, px, py);      // acperp
        if (px * aox + py * aoy >= 0) {
            dx = px; dy = py;
        } else {
            triple_product(acx, acy, abx, aby, abx, aby, px, py);  // abperp
            if (px * aox + py * aoy < 0) return true;
            s0x = s1x; s0y = s1y;
            dx = px; dy = py;
        }
        s1x = ax; s1y = ay;   // simplex[1] = simplex[2]
        index -= 1;
        ++iter;
    }
    return false;
}

// index of the first minimum of |scan_angles[k] - a| over a strictly increasing table (np.argmin semantics).
// |ang[k] - a| is V-shaped over a monotone table, so a local minimum is the global one: start from the index a
// uniform table would give and walk; ties resolve to the lower index, as argmin does.
__device__ __forceinline__ int nearest_beam(const double* __restrict__ ang, int B, double a) {
    if (a != a) return 0;
    const double a0 = ang[0], a1 = ang[B - 1];
    double g = (a - a0) / (a1 - a0) * (double)(B - 1);
    g = g < 0. ? 0. : (g > (double)(B - 1) ? (double)(B - 1) : g);
    int k = (int)(g + 0.5);
    // the three candidates of a uniform table, loaded together
    const int km = k > 0 ? k - 1 : 0, kp = k + 1 < B ? k + 1 : B - 1;
    double dm = fabs(ang[km] - a), dk = fabs(ang[k] - a), dp = fabs(ang[kp] - a);
    if (dp < dk) { k = kp; dk = dp; } else if (dm <= dk && km != k) { k = km; dk = dm; }
    while (k + 1 < B) {
        const double dn = fabs(ang[k + 1] - a);
        if (dn < dk) { ++k; dk = dn; } else break;
    }
    while (k > 0) {
        const double dn = fabs(ang[k - 1] - a);
        if (dn <= dk) { --k; dk = dn; } else break;
    }
    return k;
}

// get_range (+ are_collinear), laser_models.py:230-280; v3 = (cos, sin)(beam_theta + pi/2) hoisted by the caller
__device__ __forceinline__ double get_range(double ox, double oy, double v3x, double v3y,
                                            double vax, double vay, double vbx, double vby) {
    const double v1x = ox - vax, v1y = oy - vay;
    const double v2x = vbx - vax, v2y = vby - vay;
    const double denom = v2x * v3x + v2y * v3y;
    double distance = INFINITY;
    if (fabs(denom) > 0.0) {
        // the reference forms d1 = cross/denom and d2 = dot/denom and accepts d1 >= 0 && 0 <= d2 <= 1.  Those tests do not
        // need the quotients: a rounded quotient is >= 0 (-0.0 included) iff the numerator is zero or has the divisor's
        // sign, and it is <= 1 iff |numerator| <= |divisor| (a larger numerator is at least one ulp larger, so the quotient
        // rounds above 1).  Most edges are missed by the beam, so the one division left is rarely executed.
        const double crs = v2x * v1y - v2y * v1x;
        const double dot = v1x * v3x + v1y * v3y;
        const bool neg = denom < 0.0;
        const bool d1_ok = crs == 0.0 || ((crs < 0.0) == neg);
        const bool d2_ok = (dot == 0.0 || ((dot < 0.0) == neg)) && fabs(dot) <= fabs(denom);
        if (d1_ok && d2_ok) distance = crs / denom;
    } else {
        const double bax = vax - ox, bay = vay - oy;
        const double cax = ox - vbx, cay = oy - vby;
        if (fabs(bax * cay - bay * cax) < 1e-8) {
            const double da = sqrt((vax - ox) * (vax - ox) + (vay - oy) * (vay - oy));
            const double db = sqrt((vbx - ox) * (vbx - ox) + (vby - oy) * (vby - oy));
            distance = da < db ? da : db;
        }
    }
    return distance;
}

constexpr int POST_THREADS = 128;
#ifndef POST_MIN_BLOCKS
#define POST_MIN_BLOCKS 8
#endif
#ifndef POST_EPC_CAP
#define POST_EPC_CAP 16      // tuning: upper bound on the envs per CTA
#endif

// Shared memory of one env inside a post_kernel CTA (doubles first, then ints; sized by A).
struct EnvSmem {
    double (*pose)[3];   // [A]    own pose AFTER iTTC zeroing (ray-cast origin, base_classes.py:225)
    double (*pre)[3];    // [A]    Simulator.agent_poses: BEFORE iTTC zeroing (:587)
    double (*verts)[8];  // [A*A]  opponent b as seen by a: a's own length/width (:223)
    int* ind;            // [4*A*A] nearest beam of each vertex
    int* cone;           // [4*A*A] beam-index intervals of the forward / backward cones, before the clip to the window
    int* coll;           // [A]    GJK flags, later GJK | iTTC
    int* hit;            // [A]    iTTC flags
    int* lapdone;        // [A]
};
__host__ __device__ constexpr int post_smem_doubles(int A) { return 6 * A + 8 * A * A + (8 * A * A + 3 * A + 1) / 2; }
__device__ __forceinline__ EnvSmem env_smem(double* base, int A) {
    EnvSmem e;
    e.pose = reinterpret_cast<double (*)[3]>(base);
    e.pre = reinterpret_cast<double (*)[3]>(base + 3 * A);
    e.verts = reinterpret_cast<double (*)[8]>(base + 6 * A);
    e.ind = reinterpret_cast<int*>(base + 6 * A + 8 * A * A);
    e.cone = e.ind + 4 * A * A;
    e.coll = e.cone + 4 * A * A;
    e.hit = e.coll + A;
    e.lapdone = e.hit + A;
    return e;
}
// Envs per CTA: as many as keep (a) the 5.5 A (A - 1) scalar work items per env of stage B within one pass of the CTA's lanes
// and (b) the 2 A ray-cast segments per env and round within one warp's scan (32).
__host__ __device__ constexpr int post_envs_per_cta(int A) {
    const int by_items = (2 * POST_THREADS) / (11 * A * (A - 1)), by_segs = 16 / A;
    const int e = by_items < by_segs ? by_items : by_segs;
    return e < 1 ? 1 : (e > POST_EPC_CAP ? POST_EPC_CAP : e);
}
// ints of CTA-wide shared memory behind the per-env blocks: per round and segment, where its items start and its first beam
__host__ __device__ constexpr int post_seg_ints(int A) { return (A - 1) * 2 * 33; }
// The beam-angle table is staged in shared memory (in front of the per-env blocks) when it is at most this long: the
// nearest-beam searches are chains of dependent table reads -- 16 of them in a row in a cone item -- and from L2 they were
// the longest thing a CTA did.
constexpr int POST_STAGED_BEAMS = 2048;   // 16 KB: with 16 agents the CTA still fits the 48 KB that need no opt-in
__host__ __device__ constexpr int post_angle_doubles(int B) { return B <= POST_STAGED_BEAMS ? B : 0; }

// The ordered pair (a, b != a) number p of A agents
__device__ __forceinline__ void pair_of(int p, int A, int& a, int& b) {
    a = p / (A - 1);
    b = p - a * (A - 1);
    b += b >= a ? 1 : 0;
}

__global__ void __launch_bounds__(POST_THREADS, POST_MIN_BLOCKS) post_kernel(SimConst c, SimState st, StepScratch sc, F110StepIO io) {
    cudaGridDependencySynchronize();
    const int A = c.A, B = c.B;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int epc = post_envs_per_cta(A);
    const int env0 = blockIdx.x * epc;
    extern __shared__ double s_all[];
    double* const s_dyn = s_all + post_angle_doubles(B);
    const int stride = post_smem_doubles(A);
    int* const s_seg = reinterpret_cast<int*>(s_dyn + epc * stride);   // [A - 1][2][33]
    __shared__ int s_active[16];
    const double* angles = c.scan_angles;
    if (post_angle_doubles(B)) {
        for (int k = tid; k < B; k += POST_THREADS) s_all[k] = __ldg(c.scan_angles + k);
        angles = s_all;
    }

    // ---- stage A: iTTC consequences, RaceCar.check_ttc base_classes.py:243-252.  One thread per (env, agent).
    for (int t = tid; t < epc * A; t += POST_THREADS) {
        const int le = t / A, a = t - le * A;
        const int env = env0 + le;
        const bool active = env < c.N && !(io.active_mask && !io.active_mask[env]);
        if (a == 0) s_active[le] = active;
        if (!active) continue;
        const EnvSmem e = env_smem(s_dyn + le * stride, A);
        const int s = env * A + a;
        const int hit = sc.ttc_hit[s];
        const double px = st.x[0][s], py = st.x[1][s];
        const double yaw_pre = sc.pre_yaw[s];
        if (hit) { st.x[3][s] = 0.; st.x[4][s] = 0.; st.x[5][s] = 0.; st.x[6][s] = 0.; }
        e.pose[a][0] = px; e.pose[a][1] = py; e.pose[a][2] = hit ? 0. : yaw_pre;
        e.pre[a][0] = px; e.pre[a][1] = py; e.pre[a][2] = yaw_pre;
        e.hit[a] = hit;
        e.coll[a] = 0;
    }
    __syncthreads();

    // ---- stage B: everything scalar about a pair of cars, ALL of it in one pass (each item is a chain of a few thousand
    // cycles of fp64 transcendentals; one item per lane): per ordered pair (a, b) the four vertices of b as a sees it with
    // their nearest beams (get_blocked_view_indices, laser_models.py:282-315) and the cones its bounding circle spans;
    // per unordered pair the GJK test (check_collision :549-563).
    // The three kinds of item sit in different warps where that still fits one pass (a warp that held all three would run
    // them one after the other).
    const int npair = A * (A - 1);
    const int nvert = 4 * npair, ncone = npair, ngjk = npair / 2;
    int oC = epc * nvert, oG = oC + epc * ncone;
    {
        const int pC = (oC + 31) & ~31, pG = (pC + epc * ncone + 31) & ~31;
        if (pG + epc * ngjk <= POST_THREADS) { oC = pC; oG = pG; }
    }
    for (int t = tid; t < oG + epc * ngjk; t += POST_THREADS) {
        int le, w;
        if (t < oC) { if (t >= epc * nvert) continue; le = t / nvert; w = t - le * nvert; }
        else if (t < oG) { if (t - oC >= epc * ncone) continue; le = (t - oC) / ncone; w = nvert + (t - oC) - le * ncone; }
        else { le = (t - oG) / ngjk; w = nvert + ncone + (t - oG) - le * ngjk; }
        if (!s_active[le]) continue;
        const EnvSmem e = env_smem(s_dyn + le * stride, A);
        if (w < nvert) {
            int a, b;
            pair_of(w >> 2, A, a, b);
            const int k = w & 3, u = a * A + b;
            // vertex k of opponent b, a's own length/width (ray_cast_agents :223); order rl, rr, fr, fl
            const double L = __ldg(c.params + a * F110_NUM_PARAMS + P_LENGTH), Wd = __ldg(c.params + a * F110_NUM_PARAMS + P_WIDTH);
            double sb, cb;
            sincos(e.pre[b][2], &sb, &cb);
            const double hx = (k < 2) ? -L / 2 : L / 2;
            const double hy = (k == 0 || k == 3) ? Wd / 2 : -Wd / 2;
            const double vxw = cb * hx + (-sb) * hy + e.pre[b][0];
            const double vyw = sb * hx + cb * hy + e.pre[b][1];
            e.verts[u][2 * k] = vxw;
            e.verts[u][2 * k + 1] = vyw;
            // arctan2(sin(yaw), cos(yaw)) == yaw for the wrapped yaw and arctan2(v/|v|) == arctan2(v), each to an ulp; the
            // angle only selects the nearest beam, so the shorter dependent chain cannot change a window except at an
            // exact tie between two beams
            const double vx = vxw - e.pose[a][0], vy = vyw - e.pose[a][1];
            double ang = e.pose[a][2] - atan2(vy, vx);
            if (vx == 0. && vy == 0.) ang = nan("");   // the reference divides by the zero norm -> NaN -> argmin 0
            if (ang > F110_PI) ang = ang - 2 * F110_PI;
            else if (ang < -F110_PI) ang = ang + 2 * F110_PI;
            e.ind[4 * u + k] = nearest_beam(angles, B, -ang);
        } else if (w < nvert + ncone) {
            int a, b;
            pair_of(w - nvert, A, a, b);
            const int u = a * A + b;
            // The reference walks every beam of the window (all 1080 when the opponent is behind the car) although only
            // beams whose LINE crosses the opponent can be lowered: a proper hit needs the ray to enter the car's bounding
            // circle, and the collinear fallback of get_range (:270-274) needs the beam's line to contain an edge, forwards
            // or backwards.  Beams further than alpha (+1e-6 rad) from both the bearing of the circle's centre and its
            // opposite are never visited -- for them get_range returns inf on all four edges.
            const double L = __ldg(c.params + a * F110_NUM_PARAMS + P_LENGTH), Wd = __ldg(c.params + a * F110_NUM_PARAMS + P_WIDTH);
            const double R = 0.5 * sqrt(L * L + Wd * Wd) * (1.0 + 1e-9) + 1e-9;
            const double dx = e.pre[b][0] - e.pose[a][0], dy = e.pre[b][1] - e.pose[a][1];
            const double dist = sqrt(dx * dx + dy * dy);
            // cone -> beam-index intervals (supersets by one beam each side); the clip to the reference window follows in
            // stage C, when the vertices' beams are known.  Default: no pruning, i.e. the whole window forwards.
            int f0 = 0, f1 = B - 1, b0 = B, b1 = -1;
            const double alpha = asin(R / dist) + 1e-6;
            // beam angles lie inside [-fov/2, fov/2]: a cone of half-width < pi - fov/2 around a bearing in [-pi, pi] can only
            // meet them un-wrapped (0.79 rad at the default 4.7 rad lidar; a lidar of 2 (pi - 0.05) rad or more is never pruned)
            const double cone_max = fmin(0.75, F110_PI - 0.5 * c.fov - 0.01);
            if (dist > R * (1.0 + 1e-6) && alpha < cone_max) {
                double phi = atan2(dy, dx) - e.pose[a][2];           // in [-2 pi, 2 pi] -> [-pi, pi]
                if (phi > F110_PI) phi -= 2 * F110_PI;
                else if (phi < -F110_PI) phi += 2 * F110_PI;
                const double back = phi > 0. ? phi - F110_PI : phi + F110_PI;
                const double amin = angles[0], amax = angles[B - 1];
                if (phi + alpha < amin || phi - alpha > amax) { f0 = B; f1 = -1; }
                else {
                    f0 = nearest_beam(angles, B, phi - alpha) - 1;
                    f1 = nearest_beam(angles, B, phi + alpha) + 1;
                }
                if (!(back + alpha < amin || back - alpha > amax)) {
                    b0 = nearest_beam(angles, B, back - alpha) - 1;
                    b1 = nearest_beam(angles, B, back + alpha) + 1;
                }
            }   // else: overlapping cars, NaN, or a cone too wide to reason about -> the whole reference window
            e.cone[4 * u] = f0; e.cone[4 * u + 1] = f1; e.cone[4 * u + 2] = b0; e.cone[4 * u + 3] = b1;
        } else {
            // unordered pair number p -> (a < b)
            int p = w - nvert - ncone, a = 0;
            while (p >= A - 1 - a) { p -= A - 1 - a; ++a; }
            const int b = a + 1 + p;
            double va[8], vb[8];
            const double L = __ldg(c.sim_params + P_LENGTH), Wd = __ldg(c.sim_params + P_WIDTH);
            get_vertices(e.pre[a][0], e.pre[a][1], e.pre[a][2], L, Wd, va);
            get_vertices(e.pre[b][0], e.pre[b][1], e.pre[b][2], L, Wd, vb);
            if (gjk_collision(va, vb)) { e.coll[a] = 1; e.coll[b] = 1; }
        }
    }
    __syncthreads();

    // ---- stage C, two jobs side by side.
    // (1) The ray-cast's work list.  Car a meets its opponents in A - 1 ROUNDS, b = (a + k) mod A in round k, so that within
    // a round every beam of every car is touched by at most one item (the minimum the reference forms opponent by
    // opponent does not depend on their order).  Per round one warp turns the 2 A segments per env (forward and backward
    // cone of the one opponent, clipped to the reference's window) into a prefix sum of their lengths.
    const int nseg = epc * A * 2;     // <= 32
    for (int k = 1 + wid; k < A; k += POST_THREADS / 32) {
        int i0 = B, len = 0;
        if (lane < nseg) {
            const int le = lane / (2 * A), r = lane - le * 2 * A, a = r >> 1, half = r & 1;
            if (s_active[le]) {
                const EnvSmem e = env_smem(s_dyn + le * stride, A);
                int b = a + k; b -= b >= A ? A : 0;
                const int u = a * A + b;
                const int* q = e.ind + 4 * u;
                const int lo = min(min(q[0], q[1]), min(q[2], q[3])), hi = max(max(q[0], q[1]), max(q[2], q[3]));
                int f0 = max(lo, e.cone[4 * u]), f1 = min(hi, e.cone[4 * u + 1]);
                int b0 = max(lo, e.cone[4 * u + 2]), b1 = min(hi, e.cone[4 * u + 3]);
                if (b0 <= f1 && f0 <= b1) { f0 = min(f0, b0); f1 = max(f1, b1); b0 = B; b1 = -1; }   // merge overlap
                i0 = half ? b0 : f0;
                len = max(0, (half ? b1 : f1) - i0 + 1);
            }
        }
        int run = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int other = __shfl_up_sync(0xffffffffu, run, o);
            if (lane >= o) run += other;
        }
        int* seg = s_seg + (k - 1) * 66;
        seg[lane + 1] = run;             // seg[j] = first item of segment j, seg[32] = number of items
        if (lane == 0) seg[0] = 0;
        seg[33 + lane] = i0;
    }
    // (2) finish zone / laps per agent, _check_done f110_env.py:320-348
    for (int t = tid; t < epc * A; t += POST_THREADS) {
        const int le = t / A, a = t - le * A;
        if (!s_active[le]) continue;
        const EnvSmem e = env_smem(s_dyn + le * stride, A);
        const int env = env0 + le;
        const int s = env * A + a;
        const double new_time = st.time[env] + c.timestep;   // :406 (written back in stage E, after the barrier)
        const int col = (e.coll[a] | e.hit[a]) ? 1 : 0;
        const double dxp = e.pose[a][0] - st.start_x[s];
        const double dyp = e.pose[a][1] - st.start_y[s];
        const double rc = st.rot_c[env], rs = st.rot_s[env];
        // start_rot = [[cos(-t), -sin(-t)], [sin(-t), cos(-t)]]
        const double lx = rc * dxp + (-rs) * dyp;
        double ty = rs * dxp + rc * dyp;
        if (ty > 2) ty -= 2;
        else if (ty < -2) ty = -2 - ty;
        else ty = 0;
        const double dist2 = lx * lx + ty * ty;
        const bool closes = dist2 <= 0.1;
        int near = st.near_start[s];
        int tog = st.toggles[s];
        if (closes && !near) { near = 1; tog += 1; }
        else if (!closes && near) { near = 0; tog += 1; }
        st.near_start[s] = (uint8_t)near;
        st.toggles[s] = tog;
        const double lapc = (double)(tog / 2);
        st.lap_counts[s] = lapc;
        double lapt = st.lap_times[s];
        if (tog < 4) { lapt = new_time; st.lap_times[s] = lapt; }
        st.collisions[s] = (uint8_t)col;
        e.lapdone[a] = tog >= 4;
        if (io.collisions) io.collisions[s] = (uint8_t)col;
        if (io.toggles) io.toggles[s] = tog;
        if (io.lap_times) io.lap_times[s] = lapt;
        if (io.lap_counts) io.lap_counts[s] = lapc;
        if (io.state) {
            double* o = io.state + (size_t)s * 7;
#pragma unroll
            for (int k = 0; k < 7; ++k) o[k] = st.x[k][s];   // this thread wrote the zeroed entries itself in stage A
        }
        if (io.agent_poses) { double* o = io.agent_poses + (size_t)s * 3; o[0] = e.pre[a][0]; o[1] = e.pre[a][1]; o[2] = e.pre[a][2]; }
    }
    __syncthreads();

    // ---- stage D: opponent ray-cast (ray_cast_agents :206-227).  The lidar kernel already wrote every scan; only the
    // beams inside some opponent's cone can get shorter, so only those are re-read, lowered and re-written -- one beam per
    // lane, the items of all envs and cars of the CTA packed back to back.
    const float lm = c.lidar_max;
    for (int k = 1; k < A; ++k) {
        const int* seg = s_seg + (k - 1) * 66;
        const int total = seg[32];
        for (int it = tid; it < total; it += POST_THREADS) {
            // the segment holding item `it`: the last j with seg[j] <= it (empty segments repeat a start and are skipped)
            int j = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) j += (j + step < 32 && seg[j + step] <= it) ? step : 0;
            const int le = j / (2 * A), a = (j - le * 2 * A) >> 1;
            int b = a + k; b -= b >= A ? A : 0;
            const EnvSmem e = env_smem(s_dyn + le * stride, A);
            const double* v = e.verts[a * A + b];
            const int i = seg[33 + j] + (it - seg[j]);
            const int env = env0 + le;
            const size_t g = (size_t)(env * A + a) * B + i;
            double v3x, v3y;
            sincos(e.pose[a][2] + angles[i] + F110_PI / 2., &v3y, &v3x);
            const double ox = e.pose[a][0], oy = e.pose[a][1];
            double best = INFINITY;      // where this beam meets the opponent, if it does
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int j2 = (jj + 1) & 3;
                const double rr = get_range(ox, oy, v3x, v3y, v[2 * jj], v[2 * jj + 1], v[2 * j2], v[2 * j2 + 1]);
                if (rr < best) best = rr;
            }
            // scan[i] = min(scan[i], best), in the caller's buffers (the lidar kernel wrote them).  With an fp64 scan
            // among the outputs that is the reference's statement; without one the float outputs are lowered each in its
            // own domain, which gives the same floats: float conversion and the observation's clip / scale are monotone,
            // so float(min(a, b)) == min(float(a), float(b)).  (One corner differs: a NaN scan -- only injected NaN noise
            // produces one on a finite pose -- stays NaN in the reference, whereas its observation value lm / lm can be
            // lowered here when no scan output was asked for.)
            if (best < INFINITY) {
                if (io.scans_f64) {
                    if (best < io.scans_f64[g]) {
                        io.scans_f64[g] = best;
                        if (io.scans_f32) io.scans_f32[g] = (float)best;
                        if (a == 0 && io.obs) io.obs[(size_t)env * (B + 8) + i] = obs_lidar<false>(best, lm, 0.0f);
                    }
                } else {
                    if (io.scans_f32) { const float nv = (float)best; if (nv < io.scans_f32[g]) io.scans_f32[g] = nv; }
                    if (a == 0 && io.obs) {
                        float* o = io.obs + (size_t)env * (B + 8) + i;
                        const float nv = obs_lidar<false>(best, lm, 0.0f);
                        if (nv < *o) *o = nv;
                    }
                }
            }
        }
        if (k + 1 < A) __syncthreads();   // the next round re-reads what this one lowered
    }
    __syncthreads();

    // ---- stage E: done, reward, time, pose part of the observation, episode statistics.  One thread per env.
    if (tid < epc && s_active[tid]) {
        const EnvSmem e = env_smem(s_dyn + tid * stride, A);
        const int env = env0 + tid;
        const double new_time = st.time[env] + c.timestep;
        bool all_laps = true;
        for (int a = 0; a < A; ++a) all_laps = all_laps && e.lapdone[a];
        const bool ego_col = (e.coll[c.ego] | e.hit[c.ego]) != 0;
        const bool done = ego_col || all_laps;   // f110_env.py:350
        st.time[env] = new_time;
        if (io.time) io.time[env] = new_time;
        if (io.reward) io.reward[env] = (float)c.timestep;
        if (io.terminated) io.terminated[env] = done ? 1 : 0;
        if (io.obs) {   // f110_env.py:563-579: slots for agents 0 and 1
            float* q = io.obs + (size_t)env * (B + 8) + B;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                q[4 * k] = (float)e.pose[k][0];
                q[4 * k + 1] = (float)e.pose[k][1];
                q[4 * k + 2] = (float)wrap_angle(e.pose[k][2]);
                q[4 * k + 3] = (e.coll[k] | e.hit[k]) ? 1.0f : 0.0f;
            }
        }
        if (done) {
            atomicAdd(sc.stats + F110_STAT_EPISODES, 1.0);
            atomicAdd(sc.stats + F110_STAT_EPISODE_STEPS, (double)st.step_count[env] + 1.0);
            atomicAdd(sc.stats + F110_STAT_EPISODE_TIME, new_time);
            if (ego_col) atomicAdd(sc.stats + F110_STAT_EGO_COLLISIONS, 1.0);
            if (all_laps) atomicAdd(sc.stats + F110_STAT_LAPS_DONE, 1.0);
        }
    }
    latch_launch_order(sc);
}

// K3 for A == 1: nothing to ray-cast and no pair to test, the lidar kernel already wrote the scans -> one thread
// per env applies the iTTC consequence and the finish-zone / done bookkeeping (same statements as post_kernel).
__global__ void __launch_bounds__(128) post_single_kernel(SimConst c, SimState st, StepScratch sc, F110StepIO io) {
    cudaGridDependencySynchronize();
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env < c.N && !(io.active_mask && !io.active_mask[env])) {
    const int s = env;
    const int hit = sc.ttc_hit[s];
    const double px = st.x[0][s], py = st.x[1][s];
    double yaw = sc.pre_yaw[s];
    if (hit) { st.x[3][s] = 0.; st.x[4][s] = 0.; st.x[5][s] = 0.; st.x[6][s] = 0.; yaw = 0.; }
    const double new_time = st.time[env] + c.timestep;
    const double dxp = px - st.start_x[s];
    const double dyp = py - st.start_y[s];
    const double rc = st.rot_c[env], rs = st.rot_s[env];
    const double lx = rc * dxp + (-rs) * dyp;
    double ty = rs * dxp + rc * dyp;
    if (ty > 2) ty -= 2;
    else if (ty < -2) ty = -2 - ty;
    else ty = 0;
    const bool closes = (lx * lx + ty * ty) <= 0.1;
    int near = st.near_start[s];
    int tog = st.toggles[s];
    if (closes && !near) { near = 1; tog += 1; }
    else if (!closes && near) { near = 0; tog += 1; }
    st.near_start[s] = (uint8_t)near;
    st.toggles[s] = tog;
    const double lapc = (double)(tog / 2);
    st.lap_counts[s] = lapc;
    double lapt = st.lap_times[s];
    if (tog < 4) { lapt = new_time; st.lap_times[s] = lapt; }
    st.collisions[s] = (uint8_t)hit;
    st.time[env] = new_time;
    const bool done = hit || tog >= 4;
    if (io.collisions) io.collisions[s] = (uint8_t)hit;
    if (io.toggles) io.toggles[s] = tog;
    if (io.lap_times) io.lap_times[s] = lapt;
    if (io.lap_counts) io.lap_counts[s] = lapc;
    if (io.state) {
        double* o = io.state + (size_t)s * 7;
#pragma unroll
        for (int k = 0; k < 7; ++k) o[k] = st.x[k][s];
    }
    if (io.agent_poses) { double* o = io.agent_poses + (size_t)s * 3; o[0] = px; o[1] = py; o[2] = sc.pre_yaw[s]; }
    if (io.time) io.time[env] = new_time;
    if (io.reward) io.reward[env] = (float)c.timestep;
    if (io.terminated) io.terminated[env] = done ? 1 : 0;
    if (io.obs) {
        float* q = io.obs + (size_t)env * (c.B + 8) + c.B;
        q[0] = (float)px; q[1] = (float)py; q[2] = (float)wrap_angle(yaw); q[3] = hit ? 1.0f : 0.0f;
        q[4] = q[5] = q[6] = q[7] = 0.0f;
    }
    if (done) {
        atomicAdd(sc.stats + F110_STAT_EPISODES, 1.0);
        atomicAdd(sc.stats + F110_STAT_EPISODE_STEPS, (double)st.step_count[env] + 1.0);
        atomicAdd(sc.stats + F110_STAT_EPISODE_TIME, new_time);
        if (hit) atomicAdd(sc.stats + F110_STAT_EGO_COLLISIONS, 1.0);
        if (tog >= 4) atomicAdd(sc.stats + F110_STAT_LAPS_DONE, 1.0);
    }
    }
    latch_launch_order(sc);
}

}  // namespace

// Launch with programmatic stream serialisation (PDL): the grid may be scheduled while the previous kernel of the stream
// drains; the kernel itself waits in cudaGridDependencySynchronize() before it touches anything that kernel wrote.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

cudaError_t launch_dynamics(const SimConst& c, const MapView& m, const SimState& st, const StepScratch& sc, const F110StepIO& io,
                            const MapSet* ms, cudaStream_t s) {
    const int threads = 128;
    const dim3 grid((c.NA + threads - 1) / threads);
    if (ms) return launch_pdl(dynamics_maps_kernel, grid, dim3(threads), 0, s, c, m, st, sc, io, *ms);
    return launch_pdl(dynamics_kernel, grid, dim3(threads), 0, s, c, m, st, sc, io);
}

typedef void (*LidarKernel)(SimConst, MapView, SimState, StepScratch, F110StepIO);
typedef void (*LidarMapsKernel)(SimConst, MapView, SimState, StepScratch, F110StepIO, MapSet);

template <int MODE>
static LidarKernel lidar_variant_t(int fb, bool count) {
    switch (fb) {
        case 19: return count ? lidar_kernel<19, true, MODE> : lidar_kernel<19, false, MODE>;
        case 20: return count ? lidar_kernel<20, true, MODE> : lidar_kernel<20, false, MODE>;
        case 21: return count ? lidar_kernel<21, true, MODE> : lidar_kernel<21, false, MODE>;
        case 22: return count ? lidar_kernel<22, true, MODE> : lidar_kernel<22, false, MODE>;
        default: return count ? lidar_kernel<0, true, MODE> : lidar_kernel<0, false, MODE>;
    }
}
// fb = the map's fraction bits when the TUNED variant applies, else 0; mode as in lidar_kernel
static LidarKernel lidar_variant(int fb, bool count, int mode) {
    return mode == 3 ? lidar_variant_t<3>(fb, count) : mode == 2 ? lidar_variant_t<2>(fb, count) :
           mode == 1 ? lidar_variant_t<1>(fb, count) : lidar_variant_t<0>(fb, count);
}

template <int MODE>
static LidarMapsKernel lidar_maps_variant_t(int fb, bool count) {
    switch (fb) {
        case 19: return count ? lidar_maps_kernel<19, true, MODE> : lidar_maps_kernel<19, false, MODE>;
        case 20: return count ? lidar_maps_kernel<20, true, MODE> : lidar_maps_kernel<20, false, MODE>;
        case 21: return count ? lidar_maps_kernel<21, true, MODE> : lidar_maps_kernel<21, false, MODE>;
        case 22: return count ? lidar_maps_kernel<22, true, MODE> : lidar_maps_kernel<22, false, MODE>;
        default: return count ? lidar_maps_kernel<0, true, MODE> : lidar_maps_kernel<0, false, MODE>;
    }
}
static LidarMapsKernel lidar_maps_variant(int fb, bool count, int mode) {
    return mode == 3 ? lidar_maps_variant_t<3>(fb, count) : mode == 2 ? lidar_maps_variant_t<2>(fb, count) :
           mode == 1 ? lidar_maps_variant_t<1>(fb, count) : lidar_maps_variant_t<0>(fb, count);
}

// CTAs of the lidar kernel that are resident at once on the current device (one wave of persistent warps)
int lidar_resident_blocks(bool single_agent) {
    int dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lidar_variant(21, false, single_agent ? 1 : 0), LIDAR_THREADS, 0) != cudaSuccess)
        return -1;
    return sms * per_sm;
}

namespace {
__global__ void smid_probe_kernel(unsigned char* seen) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (threadIdx.x == 0) seen[smid & (F110_SMID_TABLE - 1u)] = 1;
}
}  // namespace

cudaError_t probe_sm_ids(unsigned char* seen) {
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    unsigned char* d = nullptr;
    if (e == cudaSuccess) e = cudaMalloc(&d, F110_SMID_TABLE);
    if (e == cudaSuccess) e = cudaMemset(d, 0, F110_SMID_TABLE);
    if (e == cudaSuccess) { smid_probe_kernel<<<sms * 8, 128>>>(d); e = cudaPeekAtLastError(); }
    if (e == cudaSuccess) e = cudaMemcpy(seen, d, F110_SMID_TABLE, cudaMemcpyDeviceToHost);
    cudaFree(d);
    return e;
}

cudaError_t launch_lidar(const SimConst& c, const MapView& m, const SimState& st, const StepScratch& sc, const F110StepIO& io,
                         const MapSet* ms, bool count_lookups, int resident_blocks, int32_t* variant, cudaStream_t s) {
    // TUNED variant: compile-time fraction bits, d > 0 for d > eps, max_range 30, the observation's division by 30 through its
    // reciprocal.  For a map set m carries the set's common fraction bits and the smallest positive cell over all its maps.
    const bool tuned = m.guard == 2u && c.obs_fast_div && c.max_range == 30.0 && c.eps > 0.0 && m.min_positive > c.eps &&
                       m.fx_bits >= 19u && m.fx_bits <= 22u;
    const bool lean = !io.noise && !io.scans_f64 && !io.active_mask;
    const int mode = c.A != 1 ? (lean ? 3 : 0) : (lean && io.obs && !io.scans_f32) ? 2 : 1;
    variant[0] = (int32_t)m.fx_bits; variant[1] = tuned ? (int32_t)m.fx_bits : 0; variant[2] = mode; variant[3] = ms ? 1 : 0;
    // one wave of persistent warps, or fewer when there are not that many units
    const unsigned want = (sc.num_units + LIDAR_THREADS / 32 - 1) / (LIDAR_THREADS / 32);
    const unsigned blocks = want < (unsigned)resident_blocks ? want : (unsigned)resident_blocks;
    if (ms)
        return launch_pdl(lidar_maps_variant(tuned ? (int)m.fx_bits : 0, count_lookups, mode), dim3(blocks ? blocks : 1u),
                          dim3(LIDAR_THREADS), 0, s, c, m, st, sc, io, *ms);
    return launch_pdl(lidar_variant(tuned ? (int)m.fx_bits : 0, count_lookups, mode), dim3(blocks ? blocks : 1u), dim3(LIDAR_THREADS), 0,
                      s, c, m, st, sc, io);
}

namespace {
__global__ void set_env_maps_kernel(int32_t* __restrict__ env_map, const int32_t* __restrict__ slots,
                                    const uint8_t* __restrict__ mask, int N, int count) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N || (mask && !mask[e])) return;
    const int32_t k = slots[e];
    if (k >= 0 && k < count) env_map[e] = k;
}
}  // namespace

cudaError_t launch_set_env_maps(int32_t* env_map, const int32_t* slots, const uint8_t* mask, int N, int count, cudaStream_t s) {
    set_env_maps_kernel<<<(N + 127) / 128, 128, 0, s>>>(env_map, slots, mask, N, count);
    return cudaPeekAtLastError();
}

cudaError_t launch_post(const SimConst& c, const SimState& st, const StepScratch& sc, const F110StepIO& io, cudaStream_t s) {
    if (c.A == 1) return launch_pdl(post_single_kernel, dim3((c.N + 127) / 128), dim3(128), 0, s, c, st, sc, io);
    const int epc = post_envs_per_cta(c.A);
    return launch_pdl(post_kernel, dim3((c.N + epc - 1) / epc), dim3(POST_THREADS),
                      sizeof(double) * (post_angle_doubles(c.B) + post_smem_doubles(c.A) * epc) + sizeof(int) * post_seg_ints(c.A), s, c, st, sc, io);
}

cudaError_t launch_sim_reset(const SimConst& c, const SimState& st, const double* poses, const uint8_t* mask, cudaStream_t s) {
    const int threads = 128;
    sim_reset_kernel<<<(c.NA + threads - 1) / threads, threads, 0, s>>>(c, st, poses, mask);
    return cudaPeekAtLastError();
}

// ---------------------------------------------------------------- map padding (set_map time, off the step path)

namespace {
__global__ void pad_map_kernel(const double* __restrict__ dense, int H, int W, double* __restrict__ padded, int prows, int pitch) {
    const size_t n = (size_t)prows * pitch;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(k / pitch) - 1, col = (int)(k - (size_t)(row + 1) * pitch) - 1;
        padded[k] = (row >= 0 && row < H && col >= 0 && col < W) ? dense[(size_t)row * W + col] : -1.0;
    }
}

// doubles that are > 0 order like their bit patterns: atomicMin on the bits finds the smallest positive cell
__global__ void min_positive_kernel(const double* __restrict__ dense, size_t n, unsigned long long* out) {
    unsigned long long best = 0x7FF0000000000000ull;   // +inf
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) {
        const double v = dense[k];
        if (v > 0.0) { const unsigned long long b = (unsigned long long)__double_as_longlong(v); best = b < best ? b : best; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other < best ? other : best;
    }
    if ((threadIdx.x & 31) == 0) atomicMin(out, best);
}
}  // namespace

cudaError_t launch_pad_map(const double* dense, int H, int W, double* padded, int prows, int pitch, cudaStream_t s) {
    pad_map_kernel<<<148 * 8, 256, 0, s>>>(dense, H, W, padded, prows, pitch);
    return cudaPeekAtLastError();
}

cudaError_t map_min_positive(const double* dense, size_t cells, double* out, cudaStream_t s) {
    unsigned long long* d = nullptr;
    const unsigned long long inf = 0x7FF0000000000000ull;
    cudaError_t e = cudaMalloc(&d, sizeof(*d));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(d, &inf, sizeof(inf), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) { min_positive_kernel<<<148 * 4, 256, 0, s>>>(dense, cells, d); e = cudaPeekAtLastError(); }
    unsigned long long h = inf;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d);
    memcpy(out, &h, sizeof(h));
    return e;
}
