/*
 * f110_oracle.c -- CPU restatement of the F110Env step hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity checker for the CUDA library in
 * f110_gymnasium_ros2_jazzy_b200/csrc/.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load it.  The product never does.
 *
 * Parity status: PINNED.  tests/test_oracle_golden.py checks this restatement against
 *   (a) the reference's own known-answer vectors (dynamic_models.py:255-279 f_ks_gt/f_st_gt,
 *       collision_models.py:313-324), and
 *   (b) rollouts / scans recorded from the UNMODIFIED reference imported in the build
 *       container (tests/golden/make_golden.py -> tests/golden/<name>.npz).
 *
 * Every function cites the reference file:line it restates; paths are relative to
 * /root/reference/f110_gymnasium/gym/f110_gym/envs/.  Evaluation order follows Python
 * operator precedence exactly; build with -ffp-contract=off (numba emits no FMA).
 *
 * Plain C99 + libm (+ pthreads for the multi-core baseline runner).
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NPARAM 18
enum { P_MU, P_CSF, P_CSR, P_LF, P_LR, P_H, P_M, P_I, P_SMIN, P_SMAX, P_SVMIN, P_SVMAX,
       P_VSWITCH, P_AMAX, P_VMIN, P_VMAX, P_WIDTH, P_LENGTH };

#define PI 3.141592653589793 /* == numpy.pi */

/* ------------------------------------------------------------------ numpy scalar helpers */

/* np.clip on scalars == minimum(maximum(x, lo), hi); NaN propagates. */
static double np_clip(double x, double lo, double hi) {
    if (x < lo) x = lo;
    if (x > hi) x = hi;
    return x;
}

/* Python/numpy float `a % b` (floored modulo, npy_divmod). */
static double py_mod(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) {
        if ((b < 0) != (m < 0)) m += b;
    } else {
        m = copysign(0.0, b);
    }
    return m;
}

/* ------------------------------------------------------------------ dynamic_models.py */

/* accl_constraints, dynamic_models.py:29-60 */
static double accl_constraints(double vel, double accl, double v_switch, double a_max,
                               double v_min, double v_max) {
    double pos_limit;
    if (vel > v_switch) pos_limit = a_max * v_switch / vel;
    else pos_limit = a_max;
    if ((vel <= v_min && accl <= 0) || (vel >= v_max && accl >= 0)) accl = 0.;
    else if (accl <= -a_max) accl = -a_max;
    else if (accl >= pos_limit) accl = pos_limit;
    return accl;
}

/* steering_constraint, dynamic_models.py:62-87 */
static double steering_constraint(double sa, double sv, double s_min, double s_max,
                                  double sv_min, double sv_max) {
    if ((sa <= s_min && sv <= 0) || (sa >= s_max && sv >= 0)) sv = 0.;
    else if (sv <= sv_min) sv = sv_min;
    else if (sv >= sv_max) sv = sv_max;
    return sv;
}

/* vehicle_dynamics_ks, dynamic_models.py:90-121 (5 outputs) */
void f110o_vehicle_dynamics_ks(const double* x, const double* u_init, const double* p, double* f) {
    double lwb = p[P_LF] + p[P_LR];
    double u0 = steering_constraint(x[2], u_init[0], p[P_SMIN], p[P_SMAX], p[P_SVMIN], p[P_SVMAX]);
    double u1 = accl_constraints(x[3], u_init[1], p[P_VSWITCH], p[P_AMAX], p[P_VMIN], p[P_VMAX]);
    f[0] = x[3] * cos(x[4]);
    f[1] = x[3] * sin(x[4]);
    f[2] = u0;
    f[3] = u1;
    f[4] = x[3] / lwb * tan(x[2]);
}

/* vehicle_dynamics_st, dynamic_models.py:123-176 (7 outputs) */
void f110o_vehicle_dynamics_st(const double* x, const double* u_init, const double* p, double* f) {
    const double g = 9.81;
    double mu = p[P_MU], C_Sf = p[P_CSF], C_Sr = p[P_CSR], lf = p[P_LF], lr = p[P_LR];
    double h = p[P_H], m = p[P_M], I = p[P_I];
    double u[2];
    u[0] = steering_constraint(x[2], u_init[0], p[P_SMIN], p[P_SMAX], p[P_SVMIN], p[P_SVMAX]);
    u[1] = accl_constraints(x[3], u_init[1], p[P_VSWITCH], p[P_AMAX], p[P_VMIN], p[P_VMAX]);

    if (fabs(x[3]) < 0.5) {
        /* :152-160 kinematic branch; constraints are re-applied inside the ks model */
        double lwb = lf + lr;
        double fks[5];
        f110o_vehicle_dynamics_ks(x, u, p, fks);
        for (int i = 0; i < 5; ++i) f[i] = fks[i];
        double c2 = cos(x[2]);
        f[5] = u[1] / lwb * tan(x[2]) + x[3] / (lwb * (c2 * c2)) * u[0];
        f[6] = 0.0;
    } else {
        /* :164-174 */
        f[0] = x[3] * cos(x[6] + x[4]);
        f[1] = x[3] * sin(x[6] + x[4]);
        f[2] = u[0];
        f[3] = u[1];
        f[4] = x[5];
        f[5] = -mu * m / (x[3] * I * (lr + lf)) * (lf * lf * C_Sf * (g * lr - u[1] * h) + lr * lr * C_Sr * (g * lf + u[1] * h)) * x[5]
             + mu * m / (I * (lr + lf)) * (lr * C_Sr * (g * lf + u[1] * h) - lf * C_Sf * (g * lr - u[1] * h)) * x[6]
             + mu * m / (I * (lr + lf)) * lf * C_Sf * (g * lr - u[1] * h) * x[2];
        f[6] = (mu / (x[3] * x[3] * (lr + lf)) * (C_Sr * (g * lf + u[1] * h) * lr - C_Sf * (g * lr - u[1] * h) * lf) - 1) * x[5]
             - mu / (x[3] * (lr + lf)) * (C_Sr * (g * lf + u[1] * h) + C_Sf * (g * lr - u[1] * h)) * x[6]
             + mu / (x[3] * (lr + lf)) * (C_Sf * (g * lr - u[1] * h)) * x[2];
    }
}

/* pid, dynamic_models.py:178-221 */
void f110o_pid(double speed, double steer, double current_speed, double current_steer,
               double max_sv, double max_a, double max_v, double min_v, double* accl_out, double* sv_out) {
    double sv, accl, kp;
    double steer_diff = steer - current_steer;
    if (fabs(steer_diff) > 1e-4) sv = (steer_diff / fabs(steer_diff)) * max_sv;
    else sv = 0.0;
    double vel_diff = speed - current_speed;
    if (current_speed > 0.) {
        if (vel_diff > 0) { kp = 10.0 * max_a / max_v; accl = kp * vel_diff; }
        else              { kp = 10.0 * max_a / (-min_v); accl = kp * vel_diff; }
    } else {
        if (vel_diff > 0) { kp = 2.0 * max_a / max_v; accl = kp * vel_diff; }
        else              { kp = 2.0 * max_a / (-min_v); accl = kp * vel_diff; }
    }
    *accl_out = accl;
    *sv_out = sv;
}

/* ------------------------------------------------------------------ laser_models.py */

typedef struct {
    int height, width;
    double resolution, orig_x, orig_y, orig_c, orig_s;
    const double* dt;          /* [height][width] row-major, row 0 = bottom of the image */
    int theta_dis;
    const double* sines;       /* [theta_dis] */
    const double* cosines;     /* [theta_dis] */
    double fov, eps, max_range, theta_index_increment;
    int num_beams;
} ScanSim;

/* xy_2_rc + distance_transform, laser_models.py:55-104.
 * Out-of-map returns (r,c)=(-1,-1), which numba wraps to dt[H-1][W-1]. */
static double distance_transform(const ScanSim* s, double x, double y, long* lookups) {
    double x_trans = x - s->orig_x;
    double y_trans = y - s->orig_y;
    double x_rot = x_trans * s->orig_c + y_trans * s->orig_s;
    double y_rot = -x_trans * s->orig_s + y_trans * s->orig_c;
    int r, c;
    if (x_rot < 0 || x_rot >= s->width * s->resolution || y_rot < 0 || y_rot >= s->height * s->resolution) {
        c = s->width - 1;
        r = s->height - 1;
    } else {
        c = (int)(x_rot / s->resolution);
        r = (int)(y_rot / s->resolution);
    }
    if (lookups) ++*lookups;
    return s->dt[(size_t)r * s->width + c];
}

/* trace_ray, laser_models.py:106-146 */
static double trace_ray(const ScanSim* s, double x, double y, double theta_index, long* lookups) {
    int ti = (int)theta_index;
    if (ti >= s->theta_dis) ti = s->theta_dis - 1; /* memory safety only; unreachable short of a 1e-13 coincidence */
    double sn = s->sines[ti];
    double cs = s->cosines[ti];
    double d = distance_transform(s, x, y, lookups);
    double total = d;
    while (d > s->eps && total <= s->max_range) {
        x += d * cs;
        y += d * sn;
        d = distance_transform(s, x, y, lookups);
        total += d;
    }
    if (total > s->max_range) total = s->max_range;
    return total;
}

/* get_scan, laser_models.py:148-186 */
static void get_scan(const ScanSim* s, const double* pose, double* scan, long* lookups) {
    double theta_index = s->theta_dis * (pose[2] - s->fov / 2.) / (2. * PI);
    theta_index = fmod(theta_index, (double)s->theta_dis);
    while (theta_index < 0) theta_index += s->theta_dis;
    for (int i = 0; i < s->num_beams; ++i) {
        scan[i] = trace_ray(s, pose[0], pose[1], theta_index, lookups);
        theta_index += s->theta_index_increment;
        while (theta_index >= s->theta_dis) theta_index -= s->theta_dis;
    }
}

/* check_ttc_jit, laser_models.py:188-217 (error_model='numpy': x/0 -> inf/nan, no raise) */
static int check_ttc(const double* scan, double vel, const double* cosines, const double* side_distances,
                     double ttc_thresh, int num_beams) {
    if (vel != 0.0) {
        for (int i = 0; i < num_beams; ++i) {
            double proj_vel = vel * cosines[i];
            double ttc = (scan[i] - side_distances[i]) / proj_vel;
            if ((ttc < ttc_thresh) && (ttc >= 0.0)) return 1;
        }
    }
    return 0;
}

/* cross, laser_models.py:219-228 */
static double cross2(const double* v1, const double* v2) { return v1[0] * v2[1] - v1[1] * v2[0]; }

/* get_range (+ are_collinear), laser_models.py:230-280 */
static double get_range(const double* pose, double beam_theta, const double* va, const double* vb) {
    double o[2] = { pose[0], pose[1] };
    double v1[2] = { o[0] - va[0], o[1] - va[1] };
    double v2[2] = { vb[0] - va[0], vb[1] - va[1] };
    double v3[2] = { cos(beam_theta + PI / 2.), sin(beam_theta + PI / 2.) };
    double denom = v2[0] * v3[0] + v2[1] * v3[1];
    double distance = INFINITY;
    if (fabs(denom) > 0.0) {
        double d1 = cross2(v2, v1) / denom;
        double d2 = (v1[0] * v3[0] + v1[1] * v3[1]) / denom;
        if (d1 >= 0.0 && d2 >= 0.0 && d2 <= 1.0) distance = d1;
    } else {
        /* are_collinear(o, va, vb): ba = va - o ; ca = o - vb */
        double ba[2] = { va[0] - o[0], va[1] - o[1] };
        double ca[2] = { o[0] - vb[0], o[1] - vb[1] };
        if (fabs(cross2(ba, ca)) < 1e-8) {
            double da = sqrt((va[0] - o[0]) * (va[0] - o[0]) + (va[1] - o[1]) * (va[1] - o[1]));
            double db = sqrt((vb[0] - o[0]) * (vb[0] - o[0]) + (vb[1] - o[1]) * (vb[1] - o[1]));
            distance = da < db ? da : db;
        }
    }
    return distance;
}

static int argmin_abs_diff(const double* a, int n, double v) {
    int best = 0;
    double bv = fabs(a[0] - v);
    for (int i = 1; i < n; ++i) {
        double d = fabs(a[i] - v);
        if (d < bv) { bv = d; best = i; } /* first minimum; NaN never wins (np.argmin would pick the first NaN) */
    }
    if (bv != bv) best = 0;
    return best;
}

/* get_blocked_view_indices, laser_models.py:282-315 */
static void get_blocked_view_indices(const double* pose, const double* vertices /*[4][2]*/,
                                     const double* scan_angles, int num_beams, int* min_ind, int* max_ind) {
    double ex = cos(pose[2]), ey = sin(pose[2]);
    int lo = 0, hi = 0;
    for (int i = 0; i < 4; ++i) {
        double vx = vertices[2 * i] - pose[0];
        double vy = vertices[2 * i + 1] - pose[1];
        double norm = sqrt(vx * vx + vy * vy);
        double ux = vx / norm, uy = vy / norm;
        double angle = atan2(ey, ex) - atan2(uy, ux);
        if (angle > PI) angle = angle - 2 * PI;
        else if (angle < -PI) angle = angle + 2 * PI;
        double a = -angle;
        int ind;
        if (a != a) ind = 0; /* np.argmin over an all-NaN array returns 0 */
        else ind = argmin_abs_diff(scan_angles, num_beams, a);
        if (i == 0) { lo = hi = ind; }
        else { if (ind < lo) lo = ind; if (ind > hi) hi = ind; }
    }
    *min_ind = lo;
    *max_ind = hi;
}

/* ray_cast, laser_models.py:318-346 (scan modified in place) */
static void ray_cast(const double* pose, double* scan, const double* scan_angles, int num_beams,
                     const double* vertices /*[4][2]*/) {
    double looped[10];
    memcpy(looped, vertices, 8 * sizeof(double));
    looped[8] = vertices[0];
    looped[9] = vertices[1];
    int min_ind, max_ind;
    get_blocked_view_indices(pose, vertices, scan_angles, num_beams, &min_ind, &max_ind);
    for (int i = min_ind; i <= max_ind; ++i) {
        for (int j = 0; j < 4; ++j) {
            double r = get_range(pose, pose[2] + scan_angles[i], &looped[2 * j], &looped[2 * j + 2]);
            if (r < scan[i]) scan[i] = r;
        }
    }
}

/* ------------------------------------------------------------------ collision_models.py */

/* get_trmtx + get_vertices, collision_models.py:218-260.  The reference evaluates H.dot(col)
 * through BLAS; summation order below is the natural row-times-column order.  Vertices are
 * therefore equal to the reference to <= 1 ulp, not bit-for-bit (SURVEY a12). Order rl, rr, fr, fl. */
void f110o_get_vertices(const double* pose, double length, double width, double* v /*[4][2]*/) {
    double c = cos(pose[2]), s = sin(pose[2]);
    double hx[4] = { -length / 2, -length / 2, length / 2, length / 2 };
    double hy[4] = { width / 2, -width / 2, -width / 2, width / 2 };
    for (int i = 0; i < 4; ++i) {
        v[2 * i]     = c * hx[i] + -s * hy[i] + 0. * 0. + pose[0] * 1.;
        v[2 * i + 1] = s * hx[i] + c * hy[i] + 0. * 0. + pose[1] * 1.;
    }
}

static int furthest(const double* v /*[4][2]*/, double dx, double dy) {
    int best = 0;
    double bv = v[0] * dx + v[1] * dy;
    for (int i = 1; i < 4; ++i) {
        double d = v[2 * i] * dx + v[2 * i + 1] * dy;
        if (d > bv) { bv = d; best = i; } /* np.argmax: first maximum */
    }
    return best;
}

/* support, collision_models.py:97-111 */
static void support(const double* v1, const double* v2, const double* d, double* out) {
    int i = furthest(v1, d[0], d[1]);
    int j = furthest(v2, -d[0], -d[1]);
    out[0] = v1[2 * i] - v2[2 * j];
    out[1] = v1[2 * i + 1] - v2[2 * j + 1];
}

/* tripleProduct, collision_models.py:52-64: b*(a.c) - a*(b.c) */
static void triple(const double* a, const double* b, const double* c, double* out) {
    double ac = a[0] * c[0] + a[1] * c[1];
    double bc = b[0] * c[0] + b[1] * c[1];
    out[0] = b[0] * ac - a[0] * bc;
    out[1] = b[1] * ac - a[1] * bc;
}

/* collision (GJK), collision_models.py:113-182 */
int f110o_collision(const double* v1 /*[4][2]*/, const double* v2 /*[4][2]*/) {
    int index = 0;
    double simplex[3][2];
    double p1[2] = { (v1[0] + v1[2] + v1[4] + v1[6]) / 4, (v1[1] + v1[3] + v1[5] + v1[7]) / 4 };
    double p2[2] = { (v2[0] + v2[2] + v2[4] + v2[6]) / 4, (v2[1] + v2[3] + v2[5] + v2[7]) / 4 };
    double d[2] = { p1[0] - p2[0], p1[1] - p2[1] };
    double a[2];
    if (d[0] == 0 && d[1] == 0) d[0] = 1.0;
    support(v1, v2, d, a);
    simplex[index][0] = a[0]; simplex[index][1] = a[1];
    if (d[0] * a[0] + d[1] * a[1] <= 0) return 0;
    d[0] = -a[0]; d[1] = -a[1];
    int iter_count = 0;
    while (iter_count < 1000) {
        support(v1, v2, d, a);
        index += 1;
        simplex[index][0] = a[0]; simplex[index][1] = a[1];
        if (d[0] * a[0] + d[1] * a[1] <= 0) return 0;
        double ao[2] = { -a[0], -a[1] };
        if (index < 2) {
            double ab[2] = { simplex[0][0] - a[0], simplex[0][1] - a[1] };
            triple(ab, ao, ab, d);
            if (sqrt(d[0] * d[0] + d[1] * d[1]) < 1e-10) { d[0] = ab[1]; d[1] = -1 * ab[0]; } /* perpendicular :33-46 */
            continue;
        }
        double ab[2] = { simplex[1][0] - a[0], simplex[1][1] - a[1] };
        double ac[2] = { simplex[0][0] - a[0], simplex[0][1] - a[1] };
        double acperp[2], abperp[2];
        triple(ab, ac, ac, acperp);
        if (acperp[0] * ao[0] + acperp[1] * ao[1] >= 0) {
            d[0] = acperp[0]; d[1] = acperp[1];
        } else {
            triple(ac, ab, ab, abperp);
            if (abperp[0] * ao[0] + abperp[1] * ao[1] < 0) return 1;
            simplex[0][0] = simplex[1][0]; simplex[0][1] = simplex[1][1];
            d[0] = abperp[0]; d[1] = abperp[1];
        }
        simplex[1][0] = simplex[2][0]; simplex[1][1] = simplex[2][1];
        index -= 1;
        iter_count += 1;
    }
    return 0;
}

/* collision_multiple, collision_models.py:184-212 */
void f110o_collision_multiple(const double* vertices /*[n][4][2]*/, int n, double* collisions, double* collision_idx) {
    for (int i = 0; i < n; ++i) { collisions[i] = 0.; collision_idx[i] = -1.; }
    for (int i = 0; i < n - 1; ++i)
        for (int j = i + 1; j < n; ++j)
            if (f110o_collision(vertices + 8 * i, vertices + 8 * j)) {
                collisions[i] = 1.; collisions[j] = 1.;
                collision_idx[i] = j; collision_idx[j] = i;
            }
}

/* ------------------------------------------------------------------ base_classes.py / f110_env.py */

typedef struct {
    double state[7];        /* [x, y, steer_angle, vel, yaw, yaw_rate, slip] base_classes.py:97-98 */
    double steer_buf[2];    /* newest first (np.append(raw, buf)) :270-278 */
    int steer_cnt;
    int in_collision;
    double params[NPARAM];
} Car;

typedef struct {
    Car* cars;              /* [A] */
    double time;
    int* near_starts;       /* [A] */
    double* toggle_list;    /* [A] */
    double* lap_times;      /* [A] */
    double* lap_counts;     /* [A] */
    double* start_xs; double* start_ys; double* start_thetas;
    double start_rot[4];
    double* collisions;     /* [A] last step */
    uint64_t rng[4];        /* baseline-only noise generator state */
} Env;

typedef struct F110Oracle {
    int N, A, B;
    int integrator, ego_idx;
    double timestep, lidar_dist, ttc_thresh, lidar_max, noise_std;
    ScanSim sim;
    double* dt_own; double* sines_own; double* cosines_own;
    double* scan_angles; double* beam_cosines; double* side_distances; /* [B] */
    Env* envs;
    double sim_params[NPARAM]; /* Simulator.params (construction time) */
    int num_threads;
    long lookups; /* dt lookups of the last step (sum over all rays) */
} F110Oracle;

/* RaceCar.__init__ statics, base_classes.py:118-158 */
static void build_beam_tables(F110Oracle* o, const double* params) {
    int B = o->B;
    double fov = o->sim.fov;
    double incr = fov / (B - 1); /* ScanSimulator2D.angle_increment laser_models.py:367 */
    double dist_sides = params[P_WIDTH] / 2.;
    double dist_fr = (params[P_LF] + params[P_LR]) / 2.;
    for (int i = 0; i < B; ++i) {
        double angle = -fov / 2. + i * incr;
        double to_side, to_fr;
        o->scan_angles[i] = angle;
        o->beam_cosines[i] = cos(angle);
        if (angle > 0) {
            if (angle < PI / 2) { to_side = dist_sides / sin(angle); to_fr = dist_fr / cos(angle); }
            else { to_side = dist_sides / cos(angle - PI / 2.); to_fr = dist_fr / sin(angle - PI / 2.); }
        } else {
            if (angle > -PI / 2) { to_side = dist_sides / sin(-angle); to_fr = dist_fr / cos(-angle); }
            else { to_side = dist_sides / cos(-angle - PI / 2); to_fr = dist_fr / sin(-angle - PI / 2); }
        }
        o->side_distances[i] = to_side < to_fr ? to_side : to_fr;
    }
}

F110Oracle* f110o_create(int N, int A, int B, double fov, int theta_dis, double eps, double max_range,
                         double timestep, int integrator, int ego_idx, double lidar_dist, double ttc_thresh,
                         double lidar_max, double noise_std, uint64_t seed, const double* params /*[18]*/) {
    F110Oracle* o = (F110Oracle*)calloc(1, sizeof(F110Oracle));
    o->N = N; o->A = A; o->B = B;
    o->integrator = integrator; o->ego_idx = ego_idx;
    o->timestep = timestep; o->lidar_dist = lidar_dist; o->ttc_thresh = ttc_thresh;
    o->lidar_max = lidar_max; o->noise_std = noise_std;
    o->num_threads = 1;
    memcpy(o->sim_params, params, sizeof(double) * NPARAM);
    ScanSim* s = &o->sim;
    s->num_beams = B; s->fov = fov; s->eps = eps; s->theta_dis = theta_dis; s->max_range = max_range;
    /* laser_models.py:367-368 */
    double angle_increment = fov / (B - 1);
    s->theta_index_increment = theta_dis * angle_increment / (2. * PI);
    /* laser_models.py:379-381: linspace(0, 2pi, theta_dis) INCLUDES the endpoint */
    o->sines_own = (double*)malloc(sizeof(double) * theta_dis);
    o->cosines_own = (double*)malloc(sizeof(double) * theta_dis);
    double step = (2 * PI - 0.0) / (theta_dis - 1);
    for (int i = 0; i < theta_dis; ++i) {
        double th = (i == theta_dis - 1) ? 2 * PI : 0.0 + i * step; /* numpy.linspace: arange*step+start, endpoint fixed */
        o->sines_own[i] = sin(th);
        o->cosines_own[i] = cos(th);
    }
    s->sines = o->sines_own; s->cosines = o->cosines_own;
    o->scan_angles = (double*)malloc(sizeof(double) * B);
    o->beam_cosines = (double*)malloc(sizeof(double) * B);
    o->side_distances = (double*)malloc(sizeof(double) * B);
    build_beam_tables(o, params);
    o->envs = (Env*)calloc(N, sizeof(Env));
    for (int e = 0; e < N; ++e) {
        Env* v = &o->envs[e];
        v->cars = (Car*)calloc(A, sizeof(Car));
        for (int a = 0; a < A; ++a) memcpy(v->cars[a].params, params, sizeof(double) * NPARAM);
        v->near_starts = (int*)calloc(A, sizeof(int));
        v->toggle_list = (double*)calloc(A, sizeof(double));
        v->lap_times = (double*)calloc(A, sizeof(double));
        v->lap_counts = (double*)calloc(A, sizeof(double));
        v->start_xs = (double*)calloc(A, sizeof(double));
        v->start_ys = (double*)calloc(A, sizeof(double));
        v->start_thetas = (double*)calloc(A, sizeof(double));
        v->collisions = (double*)calloc(A, sizeof(double));
        for (int a = 0; a < A; ++a) v->near_starts[a] = 1;
        v->start_rot[0] = 1; v->start_rot[3] = 1;
        /* splitmix64 seeding of the baseline noise generator */
        uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(e + 1);
        for (int k = 0; k < 4; ++k) {
            z += 0x9E3779B97F4A7C15ull;
            uint64_t t = z;
            t = (t ^ (t >> 30)) * 0xBF58476D1CE4E5B9ull;
            t = (t ^ (t >> 27)) * 0x94D049BB133111EBull;
            v->rng[k] = t ^ (t >> 31);
        }
    }
    return o;
}

void f110o_destroy(F110Oracle* o) {
    if (!o) return;
    for (int e = 0; e < o->N; ++e) {
        Env* v = &o->envs[e];
        free(v->cars); free(v->near_starts); free(v->toggle_list); free(v->lap_times); free(v->lap_counts);
        free(v->start_xs); free(v->start_ys); free(v->start_thetas); free(v->collisions);
    }
    free(o->envs); free(o->dt_own); free(o->sines_own); free(o->cosines_own);
    free(o->scan_angles); free(o->beam_cosines); free(o->side_distances);
    free(o);
}

void f110o_set_threads(F110Oracle* o, int n) { o->num_threads = n < 1 ? 1 : n; }

/* ScanSimulator2D.set_map, laser_models.py:383-427: the caller supplies dt = resolution*edt(img)
 * (host scipy, as in the reference), flipped so that row 0 is the bottom image row. */
void f110o_set_map(F110Oracle* o, const double* dt, int H, int W, double resolution,
                   double orig_x, double orig_y, double orig_theta) {
    free(o->dt_own);
    o->dt_own = (double*)malloc(sizeof(double) * (size_t)H * W);
    memcpy(o->dt_own, dt, sizeof(double) * (size_t)H * W);
    o->sim.dt = o->dt_own;
    o->sim.height = H; o->sim.width = W; o->sim.resolution = resolution;
    o->sim.orig_x = orig_x; o->sim.orig_y = orig_y;
    o->sim.orig_s = sin(orig_theta);
    o->sim.orig_c = cos(orig_theta);
}

/* the reference builds its 2000-entry tables with numpy (laser_models.py:379-381); a caller that
 * wants bit-identical tables passes numpy's. */
void f110o_set_tables(F110Oracle* o, const double* sines, const double* cosines) {
    memcpy(o->sines_own, sines, sizeof(double) * o->sim.theta_dis);
    memcpy(o->cosines_own, cosines, sizeof(double) * o->sim.theta_dis);
}

void f110o_set_beam_tables(F110Oracle* o, const double* scan_angles, const double* beam_cosines, const double* side_distances) {
    memcpy(o->scan_angles, scan_angles, sizeof(double) * o->B);
    memcpy(o->beam_cosines, beam_cosines, sizeof(double) * o->B);
    memcpy(o->side_distances, side_distances, sizeof(double) * o->B);
}

void f110o_get_beam_tables(F110Oracle* o, double* scan_angles, double* beam_cosines, double* side_distances) {
    memcpy(scan_angles, o->scan_angles, sizeof(double) * o->B);
    memcpy(beam_cosines, o->beam_cosines, sizeof(double) * o->B);
    memcpy(side_distances, o->side_distances, sizeof(double) * o->B);
}

/* Simulator.update_params, base_classes.py:527-547 (returns -1 for the IndexError case) */
int f110o_update_params(F110Oracle* o, const double* params, int agent_idx) {
    if (agent_idx >= o->A) return -1;
    for (int e = 0; e < o->N; ++e)
        for (int a = 0; a < o->A; ++a)
            if (agent_idx < 0 || a == agent_idx) memcpy(o->envs[e].cars[a].params, params, sizeof(double) * NPARAM);
    return 0;
}

/* noise-free ScanSimulator2D.scan(pose, None), laser_models.py:429-454 */
void f110o_scan(F110Oracle* o, const double* pose, double* scan, long* lookups) {
    long n = 0;
    get_scan(&o->sim, pose, scan, &n);
    if (lookups) *lookups = n;
}

int f110o_check_ttc(F110Oracle* o, const double* scan, double vel) {
    return check_ttc(scan, vel, o->beam_cosines, o->side_distances, o->ttc_thresh, o->B);
}

void f110o_ray_cast(F110Oracle* o, const double* pose, double* scan, const double* vertices) {
    ray_cast(pose, scan, o->scan_angles, o->B, vertices);
}

/* RaceCar.update_pose without the scan, base_classes.py:256-417 */
static void update_pose(F110Oracle* o, Car* car, double raw_steer, double vel) {
    const double* p = car->params;
    double steer = 0.;
    if (car->steer_cnt < 2) {
        steer = 0.;
        /* np.append(raw_steer, buf): newest first */
        car->steer_buf[1] = car->steer_buf[0];
        car->steer_buf[0] = raw_steer;
        car->steer_cnt += 1;
    } else {
        steer = car->steer_buf[1];
        car->steer_buf[1] = car->steer_buf[0];
        car->steer_buf[0] = raw_steer;
    }
    double accl, sv;
    f110o_pid(vel, steer, car->state[3], car->state[2], p[P_SVMAX], p[P_AMAX], p[P_VMAX], p[P_VMIN], &accl, &sv);
    sv = np_clip(sv, p[P_SVMIN], p[P_SVMAX]);
    accl = np_clip(accl, -p[P_AMAX], p[P_AMAX]);
    double u[2] = { sv, accl };
    double* x = car->state;
    double dt = o->timestep;
    if (o->integrator == 1) {
        double k1[7], k2[7], k3[7], k4[7], xs[7];
        f110o_vehicle_dynamics_st(x, u, p, k1);
        for (int i = 0; i < 7; ++i) xs[i] = x[i] + dt * (k1[i] / 2);
        f110o_vehicle_dynamics_st(xs, u, p, k2);
        for (int i = 0; i < 7; ++i) xs[i] = x[i] + dt * (k2[i] / 2);
        f110o_vehicle_dynamics_st(xs, u, p, k3);
        for (int i = 0; i < 7; ++i) xs[i] = x[i] + dt * k3[i];
        f110o_vehicle_dynamics_st(xs, u, p, k4);
        double w = dt * (1.0 / 6.0); /* time_step*(1/6) is formed first :374 */
        for (int i = 0; i < 7; ++i) x[i] = x[i] + w * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
    } else {
        double f[7];
        f110o_vehicle_dynamics_st(x, u, p, f);
        for (int i = 0; i < 7; ++i) x[i] = x[i] + dt * f[i];
    }
    x[2] = np_clip(x[2], p[P_SMIN], p[P_SMAX]);
    x[3] = np_clip(x[3], p[P_VMIN], p[P_VMAX]);
    x[4] = py_mod(x[4] + PI, 2 * PI) - PI;
    const double YAW_RATE_CAP = 10.0;
    if (x[5] != x[5]) x[5] = 0.0;
    else if (isinf(x[5])) x[5] = x[5] > 0 ? YAW_RATE_CAP : -YAW_RATE_CAP;
    x[5] = np_clip(x[5], -YAW_RATE_CAP, YAW_RATE_CAP);
    const double SLIP_CAP = 60 * (PI / 180.0); /* np.deg2rad(60) = 60 * (pi/180) */
    if (x[6] != x[6]) x[6] = 0.0; /* nan_to_num default: +/-inf -> +/-DBL_MAX, then clipped */
    x[6] = np_clip(x[6], -SLIP_CAP, SLIP_CAP);
}

/* RaceCar.update_pose for n cars sharing one parameter set, one step each (test entry point): state [n][7],
 * steer_buf [n][2] (newest first) and steer_cnt [n] are updated in place; raw_steer / speed [n] are the action. */
void f110o_update_pose(const double* params, double timestep, int integrator, int n, double* state, double* steer_buf,
                       int* steer_cnt, const double* raw_steer, const double* speed) {
    F110Oracle o;
    memset(&o, 0, sizeof(o));
    o.timestep = timestep;
    o.integrator = integrator;
    for (int i = 0; i < n; ++i) {
        Car car;
        memset(&car, 0, sizeof(car));
        memcpy(car.params, params, sizeof(double) * NPARAM);
        memcpy(car.state, state + 7 * i, sizeof(double) * 7);
        car.steer_buf[0] = steer_buf[2 * i]; car.steer_buf[1] = steer_buf[2 * i + 1];
        car.steer_cnt = steer_cnt[i];
        update_pose(&o, &car, raw_steer[i], speed[i]);
        memcpy(state + 7 * i, car.state, sizeof(double) * 7);
        steer_buf[2 * i] = car.steer_buf[0]; steer_buf[2 * i + 1] = car.steer_buf[1];
        steer_cnt[i] = car.steer_cnt;
    }
}

/* baseline-only Gaussian generator (xoshiro256++ + Marsaglia polar). NOT numpy's stream: parity
 * runs inject the numpy noise through the `noise` argument instead. */
static inline uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
static uint64_t xoshiro(uint64_t* s) {
    uint64_t r = rotl(s[0] + s[3], 23) + s[0], t = s[1] << 17;
    s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45);
    return r;
}
static void fill_normal(uint64_t* s, double std, double* out, int n) {
    int i = 0;
    while (i < n) {
        double u = (double)(xoshiro(s) >> 11) * (2.0 / 9007199254740992.0) - 1.0;
        double v = (double)(xoshiro(s) >> 11) * (2.0 / 9007199254740992.0) - 1.0;
        double q = u * u + v * v;
        if (q >= 1.0 || q == 0.0) continue;
        double f = sqrt(-2.0 * log(q) / q);
        out[i++] = std * u * f;
        if (i < n) out[i++] = std * v * f;
    }
}

typedef struct {
    const void* actions; int actions_f64;
    const double* noise;
    const uint8_t* reset_mask; const double* reset_poses; const uint8_t* active_mask;
    float* obs; float* reward; uint8_t* terminated;
    double* scans; double* state; uint8_t* collisions;
    int32_t* toggles; double* lap_times; double* lap_counts; double* time;
} StepArgs;

/* RaceCar.reset base_classes.py:183-204 for every car (Simulator.reset :627-643) */
static void cars_reset(F110Oracle* o, Env* v, const double* poses /*[A][3]*/) {
    for (int a = 0; a < o->A; ++a) {
        Car* c = &v->cars[a];
        memset(c->state, 0, sizeof(c->state));
        c->state[0] = poses[3 * a]; c->state[1] = poses[3 * a + 1]; c->state[4] = poses[3 * a + 2];
        c->steer_cnt = 0; c->steer_buf[0] = c->steer_buf[1] = 0.;
        c->in_collision = 0;
    }
}

/* RaceCar.reset base_classes.py:183-204 + F110Env.reset bookkeeping f110_env.py:438-455 */
static void env_reset(F110Oracle* o, Env* v, const double* poses /*[A][3]*/) {
    int A = o->A;
    v->time = 0.0;
    for (int a = 0; a < A; ++a) {
        v->collisions[a] = 0.;
        v->near_starts[a] = 1;
        v->toggle_list[a] = 0.;
        v->start_xs[a] = poses[3 * a];
        v->start_ys[a] = poses[3 * a + 1];
        v->start_thetas[a] = poses[3 * a + 2];
    }
    cars_reset(o, v, poses);
    double th = -v->start_thetas[o->ego_idx];
    v->start_rot[0] = cos(th); v->start_rot[1] = -sin(th);
    v->start_rot[2] = sin(th); v->start_rot[3] = cos(th);
}

/* Simulator.step base_classes.py:566-625 followed by F110Env.step f110_env.py:371-421 */
static long env_step(F110Oracle* o, int e, const StepArgs* io, double* scratch /*[A*B + A*3 + A*8]*/) {
    int A = o->A, B = o->B;
    Env* v = &o->envs[e];
    long lookups = 0;
    double* scans = scratch;
    double* agent_poses = scratch + (size_t)A * B;
    double* verts = agent_poses + 3 * A;
    int is_reset = io->reset_mask && io->reset_mask[e];
    if (is_reset) env_reset(o, v, io->reset_poses + (size_t)e * A * 3);

    /* :581-587 */
    for (int a = 0; a < A; ++a) {
        Car* c = &v->cars[a];
        double steer = 0., speed = 0.;
        if (!is_reset) { /* F110Env.reset steps with a zero action f110_env.py:457-458 */
            size_t k = ((size_t)e * A + a) * 2;
            if (io->actions_f64) { steer = ((const double*)io->actions)[k]; speed = ((const double*)io->actions)[k + 1]; }
            else { steer = ((const float*)io->actions)[k]; speed = ((const float*)io->actions)[k + 1]; }
        }
        update_pose(o, c, steer, speed);
        /* :420-423 */
        double pose[3];
        pose[0] = c->state[0] + o->lidar_dist * cos(c->state[4]);
        pose[1] = c->state[1] + o->lidar_dist * sin(c->state[4]);
        pose[2] = c->state[4];
        double* scan = scans + (size_t)a * B;
        get_scan(&o->sim, pose, scan, &lookups);
        if (io->noise) {
            const double* nz = io->noise + ((size_t)e * A + a) * B;
            for (int i = 0; i < B; ++i) scan[i] += nz[i];
        } else if (o->noise_std > 0) {
            double nz[4320 + 8];
            int done = 0;
            while (done < B) {
                int n = B - done < 4320 ? B - done : 4320;
                fill_normal(v->rng, o->noise_std, nz, n);
                for (int i = 0; i < n; ++i) scan[done + i] += nz[i];
                done += n;
            }
        }
        agent_poses[3 * a] = c->state[0]; agent_poses[3 * a + 1] = c->state[1]; agent_poses[3 * a + 2] = c->state[4];
    }
    /* check_collision :549-563 */
    for (int a = 0; a < A; ++a)
        f110o_get_vertices(agent_poses + 3 * a, o->sim_params[P_LENGTH], o->sim_params[P_WIDTH], verts + 8 * a);
    /* NOTE: Simulator.check_collision uses Simulator.params, the construction-time dict (:562,
     * never touched by update_params), while RaceCar.ray_cast_agents uses the scanning car's own
     * params (:223). */
    double coll[64], cidx[64];
    f110o_collision_multiple(verts, A, coll, cidx);
    /* :592-602 */
    for (int a = 0; a < A; ++a) {
        Car* c = &v->cars[a];
        double* scan = scans + (size_t)a * B;
        int hit = check_ttc(scan, c->state[3], o->beam_cosines, o->side_distances, o->ttc_thresh, B);
        if (hit) { c->state[3] = 0.; c->state[4] = 0.; c->state[5] = 0.; c->state[6] = 0.; }
        c->in_collision = hit;
        double own[3] = { c->state[0], c->state[1], c->state[4] };
        for (int b = 0; b < A; ++b) {
            if (b == a) continue;
            double ov[8];
            f110o_get_vertices(agent_poses + 3 * b, c->params[P_LENGTH], c->params[P_WIDTH], ov);
            ray_cast(own, scan, o->scan_angles, B, ov);
        }
        if (hit) coll[a] = 1.;
    }
    for (int a = 0; a < A; ++a) v->collisions[a] = coll[a];

    /* F110Env.step :404-412 */
    v->time = v->time + o->timestep;
    /* _check_done :310-352 */
    int all_done = 1;
    for (int a = 0; a < A; ++a) {
        double px = v->cars[a].state[0] - v->start_xs[a];
        double py = v->cars[a].state[1] - v->start_ys[a];
        double dx = v->start_rot[0] * px + v->start_rot[1] * py;
        double ty = v->start_rot[2] * px + v->start_rot[3] * py;
        if (ty > 2) ty -= 2;
        else if (ty < -2) ty = -2 - ty;
        else ty = 0;
        double dist2 = dx * dx + ty * ty;
        int closes = dist2 <= 0.1;
        if (closes && !v->near_starts[a]) { v->near_starts[a] = 1; v->toggle_list[a] += 1; }
        else if (!closes && v->near_starts[a]) { v->near_starts[a] = 0; v->toggle_list[a] += 1; }
        v->lap_counts[a] = floor(v->toggle_list[a] / 2);
        if (v->toggle_list[a] < 4) v->lap_times[a] = v->time;
        if (!(v->toggle_list[a] >= 4)) all_done = 0;
    }
    int done = (v->collisions[o->ego_idx] != 0.) || all_done;

    /* outputs */
    size_t ea = (size_t)e * A;
    if (io->scans) memcpy(io->scans + ea * B, scans, sizeof(double) * A * B);
    for (int a = 0; a < A; ++a) {
        if (io->state) memcpy(io->state + (ea + a) * 7, v->cars[a].state, sizeof(double) * 7);
        if (io->collisions) io->collisions[ea + a] = v->collisions[a] != 0.;
        if (io->toggles) io->toggles[ea + a] = (int32_t)v->toggle_list[a];
        if (io->lap_times) io->lap_times[ea + a] = v->lap_times[a];
        if (io->lap_counts) io->lap_counts[ea + a] = v->lap_counts[a];
    }
    if (io->time) io->time[e] = v->time;
    if (io->reward) io->reward[e] = (float)o->timestep;
    if (io->terminated) io->terminated[e] = (uint8_t)done;
    if (io->obs) {
        /* _pack_flat_obs :552-584 (e,o = 0,1 hard-coded; single-agent extension: opponent slots = 0) */
        float* ob = io->obs + (size_t)e * (B + 8);
        float lm = (float)o->lidar_max;
        for (int i = 0; i < B; ++i) {
            float r = (float)scans[i];
            if (r != r) r = lm; else if (isinf(r)) r = r > 0 ? lm : 0.0f;
            if (r < 0.0f) r = 0.0f;
            if (r > lm) r = lm;
            ob[i] = r / lm;
        }
        for (int k = 0; k < 2; ++k) {
            float* q = ob + B + 4 * k;
            if (k < A) {
                const double* st = v->cars[k].state;
                q[0] = (float)st[0]; q[1] = (float)st[1];
                q[2] = (float)(py_mod(st[4] + PI, 2 * PI) - PI);
                q[3] = v->collisions[k] != 0. ? 1.0f : 0.0f;
            } else { q[0] = q[1] = q[2] = q[3] = 0.0f; }
        }
    }
    return lookups;
}

typedef struct { F110Oracle* o; const StepArgs* io; int e0, e1; long lookups; } Job;

static void* worker(void* arg) {
    Job* j = (Job*)arg;
    F110Oracle* o = j->o;
    double* scratch = (double*)malloc(sizeof(double) * ((size_t)o->A * o->B + 11 * o->A));
    long n = 0;
    for (int e = j->e0; e < j->e1; ++e) {
        if (j->io->active_mask && !j->io->active_mask[e]) continue;
        n += env_step(o, e, j->io, scratch);
    }
    j->lookups = n;
    free(scratch);
    return NULL;
}

int f110o_step(F110Oracle* o, const void* actions, int actions_f64, const double* noise,
               const uint8_t* reset_mask, const double* reset_poses, const uint8_t* active_mask,
               float* obs, float* reward, uint8_t* terminated, double* scans, double* state,
               uint8_t* collisions, int32_t* toggles, double* lap_times, double* lap_counts, double* time) {
    if (!o->sim.dt) return -2; /* ValueError('Map is not set for scan simulator.') laser_models.py:445-446 */
    if (o->A > 64) return -3;
    StepArgs io = { actions, actions_f64, noise, reset_mask, reset_poses, active_mask, obs, reward, terminated,
                    scans, state, collisions, toggles, lap_times, lap_counts, time };
    int T = o->num_threads;
    if (T > o->N) T = o->N;
    Job jobs[256];
    pthread_t th[256];
    if (T > 256) T = 256;
    for (int t = 0; t < T; ++t) {
        jobs[t].o = o; jobs[t].io = &io;
        jobs[t].e0 = (int)((long)o->N * t / T); jobs[t].e1 = (int)((long)o->N * (t + 1) / T);
        jobs[t].lookups = 0;
    }
    if (T == 1) worker(&jobs[0]);
    else {
        for (int t = 1; t < T; ++t) pthread_create(&th[t], NULL, worker, &jobs[t]);
        worker(&jobs[0]);
        for (int t = 1; t < T; ++t) pthread_join(th[t], NULL);
    }
    o->lookups = 0;
    for (int t = 0; t < T; ++t) o->lookups += jobs[t].lookups;
    return 0;
}

/* Simulator.reset only (base_classes.py:627-643): the cars move, no zero-action step, and F110Env's bookkeeping (start
 * poses, toggles, time) stays as it was; -1 = the ValueError case */
int f110o_sim_reset(F110Oracle* o, const double* poses /*[N][A][3]*/, int num_poses_per_env) {
    if (num_poses_per_env != o->A) return -1;
    for (int e = 0; e < o->N; ++e) cars_reset(o, &o->envs[e], poses + (size_t)e * o->A * 3);
    return 0;
}

long f110o_last_lookups(F110Oracle* o) { return o->lookups; }

/* ------------------------------------------------------------------ rl_training/utils/gap_follow.py
 * (SURVEY 8f row 1: the rule-based opponent of train_ddpg.py:168).  Paths relative to /root/reference/.
 * preprocess_lidar :3-12, create_bubble :14-19, find_max_gap :21-38, find_best_point :40-41,
 * gap_follow_action :43-58.  scan is float32 (info["scans"][1]); numpy's mean of a float32 slice sums it in
 * float32 in numpy's pairwise order (np_sum_f32) and divides by the count in float32. */

/* np.add.reduce of a contiguous float32 slice of n <= 128 elements: fewer than 8 in sequence from 0; otherwise eight
 * partial sums over stride-8 columns, joined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the remainder in sequence */
static float np_sum_f32(const float* a, int n) {
    if (n < 8) {
        float res = 0.f;
        for (int i = 0; i < n; ++i) res += a[i];
        return res;
    }
    float r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += a[i + j];
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i];
    return res;
}

void f110o_gap_follow(const float* scan, int n, double angle_min, double angle_increment,
                      float max_distance, int window_size, int bubble_radius, float threshold,
                      double* steer_out, double* speed_out, int* best_out, float* proc_out /* [n] or NULL */) {
    float* clipped = (float*)malloc(sizeof(float) * n);
    float* proc = (float*)malloc(sizeof(float) * n);
    for (int i = 0; i < n; ++i) {                 /* np.clip: NaN stays NaN */
        float v = scan[i];
        if (v < 0.f) v = 0.f;
        if (v > max_distance) v = max_distance;
        clipped[i] = v;
    }
    int half = window_size / 2;
    for (int i = 0; i < n; ++i) {
        int s = i - half < 0 ? 0 : i - half;
        int e = i + half > n - 1 ? n - 1 : i + half;
        proc[i] = np_sum_f32(clipped + s, e - s + 1) / (float)(e - s + 1);
    }
    if (proc_out) memcpy(proc_out, proc, sizeof(float) * n);
    /* np.argmin: the first NaN if there is one, otherwise the first minimum */
    int closest = 0;
    for (int i = 1; i < n && proc[closest] == proc[closest]; ++i)
        if (proc[i] != proc[i] || proc[i] < proc[closest]) closest = i;
    if (bubble_radius > n) bubble_radius = n;     /* python slices cannot overflow: the same bubble */
    {
        int s = closest - bubble_radius < 0 ? 0 : closest - bubble_radius;
        int e = closest + bubble_radius > n - 1 ? n - 1 : closest + bubble_radius;
        for (int i = s; i <= e; ++i) proc[i] = 0.f;
    }
    int best_s = 0, best_e = n - 1, best_len = -1, start = -1;
    for (int i = 0; i < n; ++i) {
        int val = proc[i] > threshold;
        if (val && start < 0) start = i;
        else if (!val && start >= 0) {
            if (i - 1 - start > best_len) { best_len = i - 1 - start; best_s = start; best_e = i - 1; }
            start = -1;
        }
    }
    if (start >= 0 && n - 1 - start > best_len) { best_len = n - 1 - start; best_s = start; best_e = n - 1; }
    int best = (best_s + best_e) / 2;
    double steering = angle_min + best * angle_increment;
    double speed;
    const double d10 = 10 * (PI / 180.0), d20 = 20 * (PI / 180.0);   /* np.radians */
    if (fabs(steering) < d10) speed = 2.5;
    else if (fabs(steering) < d20) speed = 2;
    else speed = 1.5;
    *steer_out = steering; *speed_out = speed; *best_out = best;
    free(proc); free(clipped);
}

/* ------------------------------------------------------------------ shaped reward (SURVEY 8f row 2)
 * rl_training/utils/rewards.py: parse_flat_obs :11-39, _Prog :86-180, CenterlineSafetyProgressReward :185-355;
 * rl_training/utils/track_progress.py: CenterlineProgress.__init__ :17-55, project_xy :58-95, delta_s :97-104.
 * Paths relative to /root/reference/.  One independent reward object per env (the reference has one env). */
typedef struct {
    int has_s_prev[2], has_p_prev[2];
    double s_prev[2], p_prev[2][2], cum[2], ema_abs, t_last[2], flip, buf_sum;
    int buf_n, steps;
} RewardState;

typedef struct F110RewardOracle {
    int N, n, closed, has_widths, B;
    double *xy, *s, *tan, *nrm, *mid, *wR, *wL;   /* [n][2], [n], [n-1][2] x3, [n], [n] */
    double L;
    double dt, w_prog, forward_sign, alive_bonus, w_rel_lead, lead_clip, w_lat, lat_cap, default_half_width, lidar_max,
           near_wall_dist, w_wall, wall_q, opp_safe_dist, w_opp, ego_crash_penalty, opp_crash_bonus;
    int grace_wall, grace_opp;
    RewardState* st;
} F110RewardOracle;

static void reward_state_reset(RewardState* r) {   /* _Prog.reset :98-106 + reward reset :262-264 */
    memset(r, 0, sizeof(*r));
    r->flip = +1.0;
}

F110RewardOracle* f110o_reward_create(int N, int B, const double* xy, const double* wR, const double* wL, int n, int closed,
                                      const double* p /*[17]*/, int grace_wall, int grace_opp) {
    F110RewardOracle* o = (F110RewardOracle*)calloc(1, sizeof(*o));
    o->N = N; o->n = n; o->closed = closed; o->B = B; o->has_widths = wR && wL;
    o->xy = (double*)malloc(sizeof(double) * 2 * n); memcpy(o->xy, xy, sizeof(double) * 2 * n);
    o->s = (double*)calloc(n, sizeof(double));
    o->tan = (double*)malloc(sizeof(double) * 2 * (n - 1));
    o->nrm = (double*)malloc(sizeof(double) * 2 * (n - 1));
    o->mid = (double*)malloc(sizeof(double) * 2 * (n - 1));
    for (int i = 0; i < n - 1; ++i) {             /* track_progress.py:33-49 */
        double sx = xy[2 * i + 2] - xy[2 * i], sy = xy[2 * i + 3] - xy[2 * i + 1];
        double len = sqrt(sx * sx + sy * sy);
        o->s[i + 1] = o->s[i] + len;              /* np.cumsum: sequential */
        double den = len > 1e-12 ? len : 1e-12;
        o->tan[2 * i] = sx / den; o->tan[2 * i + 1] = sy / den;
        o->nrm[2 * i] = -o->tan[2 * i + 1]; o->nrm[2 * i + 1] = o->tan[2 * i];
        o->mid[2 * i] = (xy[2 * i] + xy[2 * i + 2]) * 0.5; o->mid[2 * i + 1] = (xy[2 * i + 1] + xy[2 * i + 3]) * 0.5;
    }
    o->L = o->s[n - 1];
    if (o->has_widths) {
        o->wR = (double*)malloc(sizeof(double) * n); memcpy(o->wR, wR, sizeof(double) * n);
        o->wL = (double*)malloc(sizeof(double) * n); memcpy(o->wL, wL, sizeof(double) * n);
    }
    o->dt = p[0]; o->w_prog = p[1]; o->forward_sign = p[2]; o->alive_bonus = p[3]; o->w_rel_lead = p[4]; o->lead_clip = p[5];
    o->w_lat = p[6]; o->lat_cap = p[7]; o->default_half_width = p[8]; o->lidar_max = p[9]; o->near_wall_dist = p[10];
    o->w_wall = p[11]; o->wall_q = p[12]; o->opp_safe_dist = p[13]; o->w_opp = p[14]; o->ego_crash_penalty = p[15];
    o->opp_crash_bonus = p[16];
    o->grace_wall = grace_wall; o->grace_opp = grace_opp;
    o->st = (RewardState*)malloc(sizeof(RewardState) * N);
    for (int e = 0; e < N; ++e) reward_state_reset(&o->st[e]);
    return o;
}

void f110o_reward_destroy(F110RewardOracle* o) {
    if (!o) return;
    free(o->xy); free(o->s); free(o->tan); free(o->nrm); free(o->mid); free(o->wR); free(o->wL); free(o->st); free(o);
}

/* project_xy, track_progress.py:58-95: the 5 nearest segment midpoints (cKDTree.query, ascending distance), best
 * orthogonal projection among them (first strictly smaller distance wins) */
static void project_xy(const F110RewardOracle* o, double x, double y, double* s_out, double* t_out,
                       double* knn_out /*[5] or NULL*/, double* fallback_out /* or NULL */) {
    int K = o->n - 1 < 5 ? o->n - 1 : 5;
    int idx[5]; double dd[5];
    for (int k = 0; k < K; ++k) { idx[k] = -1; dd[k] = INFINITY; }
    for (int i = 0; i < o->n - 1; ++i) {
        double dx = o->mid[2 * i] - x, dy = o->mid[2 * i + 1] - y;
        double d2 = dx * dx + dy * dy;
        if (d2 < dd[K - 1]) {
            int k = K - 1;
            while (k > 0 && dd[k - 1] > d2) { dd[k] = dd[k - 1]; idx[k] = idx[k - 1]; --k; }
            dd[k] = d2; idx[k] = i;
        }
    }
    if (knn_out) for (int k = 0; k < 5; ++k) knn_out[k] = k < K ? (double)idx[k] : -1.0;
    int have = 0; double best_d = 0, best_s = 0, best_t = 0;
    for (int k = 0; k < K; ++k) {
        int i = idx[k];
        if (i < 0) continue;
        double ax = o->xy[2 * i], ay = o->xy[2 * i + 1];
        double abx = o->xy[2 * i + 2] - ax, aby = o->xy[2 * i + 3] - ay;
        double L2 = abx * abx + aby * aby;
        if (L2 <= 1e-12) continue;
        double apx = x - ax, apy = y - ay;
        double tp = (apx * abx + apy * aby) / L2;
        tp = tp < 0.0 ? 0.0 : (tp > 1.0 ? 1.0 : tp);
        double px = ax + tp * abx, py = ay + tp * aby;
        double s_proj = o->s[i] + tp * sqrt(abx * abx + aby * aby);
        double t_signed = (x - px) * o->nrm[2 * i] + (y - py) * o->nrm[2 * i + 1];
        double dist = sqrt((x - px) * (x - px) + (y - py) * (y - py));
        if (!have || dist < best_d) { have = 1; best_d = dist; best_s = s_proj; best_t = t_signed; }
    }
    if (!have) {   /* degenerate fallback :90-93 */
        int j = 0; double bd = INFINITY;
        for (int i = 0; i < o->n; ++i) {
            double dx = o->xy[2 * i] - x, dy = o->xy[2 * i + 1] - y;
            double d = sqrt(dx * dx + dy * dy);
            if (d < bd) { bd = d; j = i; }
        }
        *s_out = o->s[j]; *t_out = 0.0;
        if (fallback_out) *fallback_out = 1.0;
        return;
    }
    if (fallback_out) *fallback_out = 0.0;
    *s_out = best_s; *t_out = best_t;
}

/* np.searchsorted(P.s, s, side="right") - 1, clamped to [0, n-2] (rewards.py:108-110, :272-274) */
static int seg_index_at_s(const F110RewardOracle* o, double s) {
    int lo = 0, hi = o->n;
    while (lo < hi) { int m = (lo + hi) / 2; if (o->s[m] <= s) lo = m + 1; else hi = m; }
    int idx = lo - 1;
    if (idx < 0) idx = 0;
    if (idx > o->n - 2) idx = o->n - 2;
    return idx;
}

static double delta_s(const F110RewardOracle* o, double sc, double sp) {   /* track_progress.py:97-104 */
    double ds = sc - sp;
    if (o->closed) { if (ds > 0.5 * o->L) ds -= o->L; if (ds < -0.5 * o->L) ds += o->L; }
    return ds;
}

static double signed_step(const F110RewardOracle* o, RewardState* r, int who, double x, double y, double s_curr, double s_prev) {
    double ds_geom = delta_s(o, s_curr, s_prev);   /* rewards.py:113-127 */
    if (!r->has_p_prev[who]) { r->has_p_prev[who] = 1; r->p_prev[who][0] = x; r->p_prev[who][1] = y; return 0.0; }
    double dx = x - r->p_prev[who][0], dy = y - r->p_prev[who][1];
    r->p_prev[who][0] = x; r->p_prev[who][1] = y;
    int idx = seg_index_at_s(o, s_curr);
    double ds_sign = dx * o->tan[2 * idx] + dy * o->tan[2 * idx + 1];
    return copysign(fabs(ds_geom), fabs(ds_sign) > 1e-6 ? ds_sign : ds_geom);
}

static int cmp_f32(const void* a, const void* b) { float x = *(const float*)a, y = *(const float*)b; return (x > y) - (x < y); }

/* np.quantile(float32 array, q), method 'linear': q and the virtual index are float32 (numpy converts q to the array
 * dtype), gamma = vi - floor(vi) in float32, and _lerp evaluates b - (b-a)*(1-gamma) for gamma >= 0.5 else a + (b-a)*gamma,
 * all in float32 */
static float quantile_f32(float* v, int n, double q) {
    qsort(v, n, sizeof(float), cmp_f32);
    float vi = (float)(n - 1) * (float)q;
    int lo = (int)floorf(vi);
    int hi = lo + 1 < n ? lo + 1 : n - 1;
    float g = vi - (float)lo;
    float a = v[lo], b = v[hi], d = b - a;
    return g >= 0.5f ? b - d * (1.0f - g) : a + d * g;
}

static double wrap_pi(double a) { return py_mod(a + PI, 2 * PI) - PI; }

/* Per-env breakdown of one reward call, F110O_REWARD_TERMS doubles (f110_oracle.py REWARD_TERM_NAMES):
 *  0-4 the ego's 5 nearest midpoints (distance, then index; -1 where the centerline has fewer), 5-9 the opponent's,
 *  10, 11 1 where the ego's / opponent's projection fell back to the nearest node, 12-15 e_s, e_t, o_s, o_t,
 *  16 the lateral segment index, 17-19 de, dop (after the flip) and flip, 20 the wall quantile dmin (NaN when not taken),
 *  21-27 r_prog, r_alive, r_lead, r_lat, r_wall, r_opp, r_flank, 28 the early return (0 none, 1 ego crash, 2 opponent
 *  crash bonus), 29 steps, 30 oth (wrapped to [-pi, pi)), 31 w_eff.  Fields a call does not reach are NaN. */
#define F110O_REWARD_TERMS 32

static double reward_one(const F110RewardOracle* o, RewardState* r, const float* obs, double* t) {
    double tt[F110O_REWARD_TERMS];
    if (!t) t = tt;
    for (int k = 0; k < F110O_REWARD_TERMS; ++k) t[k] = NAN;
    int B = o->B;
    double ex = (double)obs[B + 0], ey = (double)obs[B + 1];
    int ego_col = obs[B + 3] != 0.0f;
    double ox = (double)obs[B + 4], oy = (double)obs[B + 5], oth = wrap_pi((double)obs[B + 6]);
    int opp_col = obs[B + 7] != 0.0f;
    r->steps += 1;                                                              /* :299 */
    t[29] = r->steps; t[30] = oth; t[28] = 0.0;
    if (ego_col) { t[28] = 1.0; return -o->ego_crash_penalty; }                 /* :302-303 */
    if (opp_col && o->opp_crash_bonus > 0.0) { t[28] = 2.0; return +o->opp_crash_bonus; }   /* :304-305 */
    /* _Prog.update :129-167 */
    double e_s, e_t, o_s, o_t;
    project_xy(o, ex, ey, &e_s, &e_t, t + 0, t + 10);
    project_xy(o, ox, oy, &o_s, &o_t, t + 5, t + 11);
    t[12] = e_s; t[13] = e_t; t[14] = o_s; t[15] = o_t;
    if (!r->has_s_prev[0]) { r->has_s_prev[0] = 1; r->s_prev[0] = e_s; }
    if (!r->has_s_prev[1]) { r->has_s_prev[1] = 1; r->s_prev[1] = o_s; }
    double de = signed_step(o, r, 0, ex, ey, e_s, r->s_prev[0]);
    double dop = signed_step(o, r, 1, ox, oy, o_s, r->s_prev[1]);
    r->s_prev[0] = e_s; r->s_prev[1] = o_s;
    if (r->buf_n < 20) {
        r->buf_sum += de; r->buf_n += 1;                                       /* sum(list) is sequential */
        if (r->buf_n == 20 && r->buf_sum / 20 < 0.0) r->flip = -1.0;
    }
    de *= r->flip; dop *= r->flip;
    t[17] = de; t[18] = dop; t[19] = r->flip;
    r->cum[0] += de; r->cum[1] += dop;
    r->ema_abs = 0.8 * r->ema_abs + (1.0 - 0.8) * fabs(de);
    r->t_last[0] = e_t; r->t_last[1] = o_t;
    double dego = de;
    if (r->steps < 10 && dego < 0.0) dego = 0.0;                                /* :311-312 */
    double r_prog = o->w_prog * o->forward_sign * dego;
    double r_alive = o->alive_bonus;
    double r_lead = 0.0;
    if (o->w_rel_lead != 0.0) {
        double lead = r->cum[0] - r->cum[1];
        lead = lead < -o->lead_clip ? -o->lead_clip : (lead > o->lead_clip ? o->lead_clip : lead);
        r_lead = o->w_rel_lead * (lead / o->lead_clip);
    }
    /* lateral :323-333 */
    int idx = seg_index_at_s(o, e_s);
    t[16] = idx;
    double wR = o->default_half_width, wL = o->default_half_width;
    if (o->has_widths) { wR = o->wR[idx]; wL = o->wL[idx]; }
    double w_eff = e_t >= 0.0 ? wL : wR;
    if (w_eff < 0.2) w_eff = 0.2;
    t[31] = w_eff;
    double lat_norm = fabs(e_t) / w_eff;
    double lat_term = lat_norm * lat_norm < o->lat_cap ? lat_norm * lat_norm : o->lat_cap;
    double r_lat = -o->w_lat * lat_term;
    /* wall :335-343 */
    double r_wall = 0.0;
    if (r->steps >= o->grace_wall) {
        float tmp[8192];
        float lm = (float)o->lidar_max;
        for (int i = 0; i < B; ++i) {
            float v = obs[i];
            if (v <= 0.0f || !isfinite(v)) v = lm;
            v = v < 0.0f ? 0.0f : (v > lm ? lm : v);
            tmp[i] = v;
        }
        double dmin = (double)quantile_f32(tmp, B, o->wall_q);
        t[20] = dmin;
        if (dmin < o->near_wall_dist) {
            double x = (o->near_wall_dist - dmin) / (o->near_wall_dist > 1e-6 ? o->near_wall_dist : 1e-6);
            r_wall = -o->w_wall * (x * x);
        }
    }
    /* opponent bubble :345-352 */
    double r_opp = 0.0;
    if (r->steps >= o->grace_opp) {
        double rho = hypot(ex - ox, ey - oy);
        if (rho < o->opp_safe_dist) {
            double y = (o->opp_safe_dist - rho) / (o->opp_safe_dist > 1e-6 ? o->opp_safe_dist : 1e-6);
            r_opp = -o->w_opp * (y * y);
        }
    }
    /* flank bonus :353-358 (_rot_into_opp_frame :62-67) */
    double r_flank = 0.0;
    {
        double dx = ex - ox, dy = ey - oy;
        double c = cos(-oth), s = sin(-oth);
        double x_rel = c * dx - s * dy, y_rel = s * dx + c * dy;
        if (0.2 <= x_rel && x_rel <= 1.8 && 0.25 <= fabs(y_rel) && fabs(y_rel) <= 0.8) {
            double yb = 0.8 - fabs(fabs(y_rel) - 0.525);
            if (yb < 0.0) yb = 0.0;
            r_flank = 0.1 * (x_rel / 1.8) * (yb / 0.8);
        }
    }
    t[21] = r_prog; t[22] = r_alive; t[23] = r_lead; t[24] = r_lat; t[25] = r_wall; t[26] = r_opp; t[27] = r_flank;
    return r_prog + r_alive + r_lead + r_lat + r_wall + r_opp + r_flank;
}

void f110o_reward_compute_terms(F110RewardOracle* o, const float* obs /*[N][B+8]*/, const uint8_t* reset_mask, double* out,
                                double* terms /*[N][F110O_REWARD_TERMS] or NULL*/) {
    for (int e = 0; e < o->N; ++e) {
        if (reset_mask && reset_mask[e]) reward_state_reset(&o->st[e]);
        out[e] = reward_one(o, &o->st[e], obs + (size_t)e * (o->B + 8), terms ? terms + (size_t)e * F110O_REWARD_TERMS : NULL);
    }
}

void f110o_reward_compute(F110RewardOracle* o, const float* obs /*[N][B+8]*/, const uint8_t* reset_mask, double* out) {
    f110o_reward_compute_terms(o, obs, reset_mask, out, NULL);
}

/* the oracle's own float32 quantile and lateral segment lookup, for the tests that pin them to numpy */
float f110o_quantile_f32(const float* v, int n, double q) {
    float* tmp = (float*)malloc(sizeof(float) * (n > 0 ? n : 1));
    memcpy(tmp, v, sizeof(float) * n);
    float r = quantile_f32(tmp, n, q);
    free(tmp);
    return r;
}

int f110o_reward_seg_index(const F110RewardOracle* o, double s) { return seg_index_at_s(o, s); }

void f110o_reward_knn(const F110RewardOracle* o, double x, double y, double* knn /*[5]*/, double* st /*[2]*/) {
    double fb;
    project_xy(o, x, y, st, st + 1, knn, &fb);
}
