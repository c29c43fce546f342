// f110_capi.cu -- the C ABI declared in include/f110_b200.h.
//
// Owns the device arena (persistent simulation state + per-step scratch + lookup tables + map)
// and sequences the three step kernels on the caller's stream.  No torch types, no hidden
// allocation or synchronisation on the step path, no CPU fallback.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "f110_kernels.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                            \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) return fail(F110_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

struct Arena {
    // bump allocator over one cudaMalloc'd block, 256-byte aligned sub-allocations
    char* base = nullptr;
    size_t used = 0, cap = 0;
    template <typename T>
    T* take(size_t n) {
        used = (used + 255) & ~size_t(255);
        T* p = base ? reinterpret_cast<T*>(base + used) : nullptr;
        used += n * sizeof(T);
        return p;
    }
};

}  // namespace

// records the message f110_last_error() returns (used by the other translation units of the library)
int f110_set_error(int code, const char* msg) { g_err = msg ? msg : ""; return code; }

struct F110Sim {
    F110Config cfg;
    SimConst c;
    SimState st;
    StepScratch sc;
    MapView map;                  // the maps' common view: slot 0's, with min_positive over all of them
    int64_t map_generation = 0;   // bumped by every set_map / set_maps: a CUDA graph captured before holds the old map by value
    int32_t map_count = 0;        // maps installed, 0 before any; the *_maps kernels run for K >= 2, the single-map ones for 1
    MapSet ms;                    // the maps' device descriptors (passed to the kernels for K >= 2)
    std::vector<MapView> h_views; // [K] host copies of ms.views: the direction tables are rebuilt from them
    bool count_lookups = false;
    bool narrow_fraction = false;
    bool debug_sync = false;
    // device memory
    char* state_blob = nullptr;   size_t state_bytes = 0;    // checkpointable
    char* scratch_blob = nullptr; size_t scratch_bytes = 0;
    double* d_tables = nullptr;   // params[A][18], sim_params[18], sines, cosines, scan_angles, beam_cos, side_dist
    double* d_map = nullptr;      // the K padded maps back to back
    double2* d_beam_tt = nullptr; // [B] beam_tt
    MapView* d_views = nullptr;   // [K] per-slot views
    double2* d_map_dir = nullptr; // [K][theta_dis] direction tables; slot 0's is c.dir_fx
    int32_t* d_env_map = nullptr; // [N] slot of each env (all 0 for one map)
    std::vector<double> h_sines, h_cosines;   // host copies: the direction tables are rebuilt from them whenever a map changes
    // host-buffer path (f110_step_host)
    cudaStream_t host_stream = nullptr;
    char* io_blob = nullptr; size_t io_bytes = 0;
    int64_t launches = 0;
    bool timing = false;
    unsigned long long max_lookups = 0;   // longest ray (lookups) seen, refreshed by f110_get_lookup_count
    unsigned long long redone_rays = 0;   // rays the lidar kernel redid in exact arithmetic, refreshed likewise
    int lidar_blocks = 0;         // CTAs of one resident wave of the lidar kernel (persistent warps)
    int32_t lidar_variant[4] = {0, 0, 0, 0};   // what the last launch_lidar selected (f110_get_lidar_variant)
    bool lidar_ran = false;
    std::vector<cudaEvent_t> tev;   // 4 events per timed step
    uint64_t ckpt_header_words[8] = {0};   // host staging of the checkpoint header (see f110_get_state)
    EdtScratch edt;               // f110_set_map_image's device scratch, kept between calls
};

namespace {

// lays out SimState inside `a`; with a.base == nullptr only measures
void layout_state(Arena& a, SimState& st, int N, int NA) {
    for (int k = 0; k < 7; ++k) st.x[k] = a.take<double>(NA);
    st.steer_buf0 = a.take<double>(NA); st.steer_buf1 = a.take<double>(NA);
    st.start_x = a.take<double>(NA); st.start_y = a.take<double>(NA); st.start_th = a.take<double>(NA);
    st.lap_times = a.take<double>(NA); st.lap_counts = a.take<double>(NA);
    st.time = a.take<double>(N); st.rot_c = a.take<double>(N); st.rot_s = a.take<double>(N);
    st.steer_cnt = a.take<int32_t>(NA); st.toggles = a.take<int32_t>(NA);
    st.step_count = a.take<uint32_t>(N);
    st.near_start = a.take<uint8_t>(NA); st.collisions = a.take<uint8_t>(NA);
}

void layout_scratch(Arena& a, StepScratch& sc, int NA, int B, bool timeline, unsigned homes) {
    sc.scan_x = a.take<double>(NA); sc.scan_y = a.take<double>(NA); sc.pre_yaw = a.take<double>(NA);
    sc.head = a.take<double>((size_t)NA * 4);
    sc.ttc_hit = a.take<int32_t>(NA);
    sc.lookups = a.take<unsigned long long>(4);
    sc.stats = a.take<double>(F110_NUM_STATS);
    sc.num_units = (unsigned)((size_t)NA * ((B + 31) / 32));
    // capacities of the three heavy-unit lists (classes >= 96 / 48 / 24 lookups); a list that overflows sends the rest of
    // its class to the light region, which costs order, never correctness
    sc.cap[0] = sc.num_units / 16 + 8; sc.cap[1] = sc.num_units / 8 + 8; sc.cap[2] = sc.num_units / 4 + 8;
    // home segments of equal size (the last may be short), none empty
    homes = homes < 1u ? 1u : (homes > sc.num_units ? sc.num_units : homes);
    sc.seg_units = (sc.num_units + homes - 1u) / homes;
    sc.homes = (sc.num_units + sc.seg_units - 1u) / sc.seg_units;
    sc.ctrl = a.take<unsigned>(ctrl_words(sc.homes));
    const size_t ncap = (size_t)sc.cap[0] + sc.cap[1] + sc.cap[2];
    sc.list[0] = a.take<unsigned>(ncap); sc.list[1] = a.take<unsigned>(ncap);
    sc.cls[0] = a.take<unsigned>(sc.num_units); sc.cls[1] = a.take<unsigned>(sc.num_units);
    sc.timeline = (timeline && sc.num_units <= (1u << 22)) ? a.take<uint4>(sc.num_units) : nullptr;
    sc.home_of_sm = a.take<unsigned>(F110_SMID_TABLE);
}

FastDiv make_fast_div(uint32_t d) {
    // Granlund & Montgomery: l = ceil(log2 d), mul = floor(2^32 (2^l - d) / d) + 1, sh1 = min(l, 1), sh2 = max(l - 1, 0)
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;
    FastDiv f;
    f.mul = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
    f.sh1 = l < 1 ? l : 1;
    f.sh2 = l > 0 ? l - 1 : 0;
    return f;
}

struct Guard {   // selects the handle's device for the duration of a call
    int prev = -1;
    bool ok = true;
    explicit Guard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

int check_step_io(const F110Sim* sim, const F110StepIO* io) {
    if (!sim || !io) return fail(F110_ERR_INVALID, "null handle or io");
    if (sim->map_count == 0) return fail(F110_ERR_MAP_NOT_SET, "Map is not set for scan simulator.");
    if (io->reset_mask && !io->reset_poses) return fail(F110_ERR_INVALID, "reset_mask given without reset_poses");
    return F110_OK;
}

int run_step(F110Sim* sim, const F110StepIO& io, cudaStream_t s) {
    cudaEvent_t e[4] = { nullptr, nullptr, nullptr, nullptr };
    if (sim->timing) {
        for (int i = 0; i < 4; ++i) { CUDA_TRY(cudaEventCreate(&e[i])); sim->tev.push_back(e[i]); }
        CUDA_TRY(cudaEventRecord(e[0], s));
    }
    // F110_DEBUG_SYNC=1 in the environment: wait for each kernel and name the one that faulted (not while the stream is
    // being captured into a CUDA graph, where a synchronisation is illegal)
    bool dbg = sim->debug_sync;
    if (dbg) {
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) dbg = false;
    }
#define DEBUG_SYNC(name)                                                                                           \
    if (dbg) {                                                                                                     \
        const cudaError_t de = cudaStreamSynchronize(s);                                                           \
        if (de != cudaSuccess) return fail(F110_ERR_CUDA, "%s: %s", name, cudaGetErrorString(de));                 \
    }
    const MapSet* ms = sim->map_count >= 2 ? &sim->ms : nullptr;
    CUDA_TRY(launch_dynamics(sim->c, sim->map, sim->st, sim->sc, io, ms, s));
    DEBUG_SYNC("dynamics_kernel")
    if (sim->timing) CUDA_TRY(cudaEventRecord(e[1], s));
    CUDA_TRY(launch_lidar(sim->c, sim->map, sim->st, sim->sc, io, ms, sim->count_lookups, sim->lidar_blocks, sim->lidar_variant, s));
    sim->lidar_ran = true;
    DEBUG_SYNC("lidar_kernel")
    if (sim->timing) CUDA_TRY(cudaEventRecord(e[2], s));
    CUDA_TRY(launch_post(sim->c, sim->st, sim->sc, io, s));
    DEBUG_SYNC("post_kernel")
#undef DEBUG_SYNC
    if (sim->timing) CUDA_TRY(cudaEventRecord(e[3], s));
    sim->launches += 3;
    CUDA_TRY(cudaPeekAtLastError());
    return F110_OK;
}

}  // namespace

extern "C" {

const char* f110_last_error(void) { return g_err.c_str(); }
int f110_abi_version(void) { return F110_ABI_VERSION; }

int f110_create(const F110Config* cfg, const double* params, F110Sim** out) {
    if (!cfg || !params || !out) return fail(F110_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != F110_ABI_VERSION) return fail(F110_ERR_INVALID, "ABI version %d != %d", cfg->abi_version, F110_ABI_VERSION);
    if (cfg->num_envs < 1 || cfg->num_agents < 1 || cfg->num_agents > F110_MAX_AGENTS || cfg->num_beams < 32 || cfg->num_beams > 32768 || cfg->theta_dis < 2)
        return fail(F110_ERR_INVALID, "need num_envs >= 1, 1 <= num_agents <= %d, 32 <= num_beams <= 32768, theta_dis >= 2", F110_MAX_AGENTS);
    if (cfg->ego_idx < 0 || cfg->ego_idx >= cfg->num_agents) return fail(F110_ERR_INDEX, "ego_idx out of range");
    // beams further than 2 pi apart would wrap the direction table more than once and are the same directions again
    if (!(cfg->fov > 0.0) || cfg->fov > 2.0 * F110_PI) return fail(F110_ERR_INVALID, "fov must lie in (0, 2 pi]");
    if (!(cfg->eps >= 0.0) || !(cfg->max_range > 0.0) || !(cfg->timestep > 0.0)) return fail(F110_ERR_INVALID, "need eps >= 0, max_range > 0, timestep > 0");
    if (cfg->integrator != F110_INTEGRATOR_RK4 && cfg->integrator != F110_INTEGRATOR_EULER)
        return fail(F110_ERR_INTEGRATOR, "Invalid Integrator Specified. Please choose RK4 or Euler");
    if ((double)cfg->num_envs * cfg->num_agents * cfg->num_beams >= 2147483648.0)
        return fail(F110_ERR_INVALID, "num_envs*num_agents*num_beams must be < 2^31 per handle; shard across handles/GPUs");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(F110_ERR_NO_DEVICE, "no CUDA device visible: libf110_b200 has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(F110_ERR_INVALID, "device %d out of range (%d visible)", cfg->device, ndev);
    Guard g(cfg->device);
    if (!g.ok) return fail(F110_ERR_CUDA, "cudaSetDevice(%d) failed", cfg->device);

    F110Sim* sim = new F110Sim();
    sim->cfg = *cfg;
    const int N = cfg->num_envs, A = cfg->num_agents, B = cfg->num_beams, NA = N * A;
    sim->count_lookups = (cfg->flags & F110_FLAG_COUNT_LOOKUPS) != 0;
    sim->narrow_fraction = (cfg->flags & F110_FLAG_NARROW_FRACTION) != 0;
    sim->debug_sync = getenv("F110_DEBUG_SYNC") != nullptr;
    sim->lidar_blocks = lidar_resident_blocks(A == 1);
    sim->sc.ordered = 0;   // set below, once the unit count is known
    if (sim->lidar_blocks < 1) {
        cudaGetLastError();
        delete sim;
        return fail(F110_ERR_CUDA, "cannot query the lidar kernel's occupancy (is this an sm_100a device?)");
    }

    Arena measure;
    layout_state(measure, sim->st, N, NA);
    sim->state_bytes = (measure.used + 255) & ~size_t(255);
    // Longest-first order for launches of up to 48 units per resident warp; larger ones get home segments, one per SM
    // (F110_LIDAR_HOMES=n forces n segments, and natural order with them).  SM ids are not contiguous, so a wave of probe
    // CTAs finds the ones in use and home k goes to the SMs of rank k * homes / SMs.
    unsigned char seen[F110_SMID_TABLE];
    if (probe_sm_ids(seen) != cudaSuccess) {
        cudaGetLastError();
        delete sim;
        return fail(F110_ERR_CUDA, "cannot probe the device's SM ids");
    }
    unsigned nsm = 0;
    for (int k = 0; k < F110_SMID_TABLE; ++k) nsm += seen[k];
    if (nsm == 0) { delete sim; return fail(F110_ERR_CUDA, "the SM id probe saw no SM"); }
    const size_t units = (size_t)NA * ((B + 31) / 32);
    bool ordered = units <= (size_t)48 * 4 * (size_t)sim->lidar_blocks;
    unsigned homes = ordered ? 1u : nsm;
    { const char* h = getenv("F110_LIDAR_HOMES"); if (h && atoi(h) > 0) { homes = (unsigned)atoi(h); ordered = ordered && homes == 1u; } }
    Arena measure2;
    layout_scratch(measure2, sim->sc, NA, B, sim->count_lookups, homes);
    sim->scratch_bytes = (measure2.used + 255) & ~size_t(255);
    const size_t ntab = (size_t)A * F110_NUM_PARAMS + F110_NUM_PARAMS + 2 * (size_t)cfg->theta_dis + 3 * (size_t)B;

    cudaError_t e = cudaMalloc(&sim->state_blob, sim->state_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&sim->scratch_blob, sim->scratch_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&sim->d_tables, ntab * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(sim->state_blob, 0, sim->state_bytes);
    if (e == cudaSuccess) e = cudaMemset(sim->scratch_blob, 0, sim->scratch_bytes);
    if (e == cudaSuccess) e = cudaMemset(sim->d_tables, 0, ntab * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&sim->d_beam_tt, (size_t)B * sizeof(double2));
    if (e == cudaSuccess) e = cudaMemset(sim->d_beam_tt, 0, (size_t)B * sizeof(double2));
    if (e == cudaSuccess) e = cudaMalloc(&sim->d_env_map, (size_t)N * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemset(sim->d_env_map, 0, (size_t)N * sizeof(int32_t));
    if (e == cudaSuccess) {
        // host_stream_rank r > 0: the r-th highest stream priority the device offers, so that a caller pipelining several
        // handles (f110_step_host_multi) gets handle 1's kernels finished -- and its download started -- first
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        int prio = least;
        if (cfg->host_stream_rank > 0) { prio = greatest + (int)cfg->host_stream_rank - 1; if (prio > least) prio = least; }
        e = cudaStreamCreateWithPriority(&sim->host_stream, cudaStreamNonBlocking, prio);
    }
    if (e != cudaSuccess) {
        fail(F110_ERR_CUDA, "device allocation failed: %s", cudaGetErrorString(e));
        f110_destroy(sim);
        return F110_ERR_CUDA;
    }
    Arena a; a.base = sim->state_blob; layout_state(a, sim->st, N, NA);
    Arena b; b.base = sim->scratch_blob; layout_scratch(b, sim->sc, NA, B, sim->count_lookups, homes);
    sim->sc.ordered = ordered ? 1u : 0u;
    // before the first step no unit is on a list: every unit is class 3 (light, natural order)
    {
        const std::vector<unsigned> light(sim->sc.num_units, 3u);
        e = cudaMemcpy(sim->sc.cls[0], light.data(), light.size() * sizeof(unsigned), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(sim->sc.cls[1], light.data(), light.size() * sizeof(unsigned), cudaMemcpyHostToDevice);
        std::vector<unsigned> table(F110_SMID_TABLE);
        for (unsigned k = 0, rank = 0; k < F110_SMID_TABLE; ++k) {
            table[k] = seen[k] ? (unsigned)((size_t)rank * sim->sc.homes / nsm) : k % sim->sc.homes;
            rank += seen[k];
        }
        if (e == cudaSuccess) e = cudaMemcpy((void*)sim->sc.home_of_sm, table.data(), table.size() * sizeof(unsigned), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        fail(F110_ERR_CUDA, "scratch initialisation failed: %s", cudaGetErrorString(e));
        f110_destroy(sim);
        return F110_ERR_CUDA;
    }

    double* t = sim->d_tables;
    SimConst& c = sim->c;
    c.N = N; c.A = A; c.B = B; c.NA = NA;
    c.theta_dis = cfg->theta_dis; c.integrator = cfg->integrator; c.ego = cfg->ego_idx;
    c.fov = cfg->fov; c.eps = cfg->eps; c.max_range = cfg->max_range; c.timestep = cfg->timestep;
    c.lidar_dist = cfg->lidar_dist; c.ttc_thresh = cfg->ttc_thresh; c.noise_std = cfg->noise_std;
    c.lidar_max = (float)cfg->lidar_max; c.seed = cfg->seed;
    c.noise_key = (uint32_t)cfg->seed ^ ((uint32_t)(cfg->seed >> 32) * 0x85EBCA6Bu) ^ 0x46313130u;
    c.div_B = make_fast_div((uint32_t)B); c.div_A = make_fast_div((uint32_t)A);
    c.ups = (unsigned)((B + 31) / 32); c.div_ups = make_fast_div(c.ups);
    for (int r = 0; r < 10; ++r) c.philox_key[r] = c.noise_key + (uint32_t)r * 0x9E3779B9u;
    c.obs_rcp = 1.0f / c.lidar_max;
    c.obs_fast_div = c.lidar_max == 30.0f ? 1 : 0;
    // ScanSimulator2D.__init__ laser_models.py:367-368
    const double angle_increment = cfg->fov / (B - 1);
    c.theta_inc = cfg->theta_dis * angle_increment / (2. * F110_PI);
    c.params = t; t += (size_t)A * F110_NUM_PARAMS;
    c.sim_params = t; t += F110_NUM_PARAMS;
    c.sines = t; t += cfg->theta_dis;
    c.cosines = t; t += cfg->theta_dis;
    c.scan_angles = t; t += B;
    c.beam_cos = t; t += B;
    c.side_dist = t; t += B;
    c.beam_tt = sim->d_beam_tt;
    c.ttc_side_max = INFINITY; c.ttc_cos_max = INFINITY;
    sim->h_sines.assign(cfg->theta_dis, 0.0); sim->h_cosines.assign(cfg->theta_dis, 1.0);

    std::vector<double> hp((size_t)(A + 1) * F110_NUM_PARAMS);
    for (int i = 0; i <= A; ++i) memcpy(&hp[(size_t)i * F110_NUM_PARAMS], params, sizeof(double) * F110_NUM_PARAMS);
    e = cudaMemcpy(sim->d_tables, hp.data(), hp.size() * sizeof(double), cudaMemcpyHostToDevice);
    // near_start is True at construction (f110_env.py:213)
    if (e == cudaSuccess) e = cudaMemset(sim->st.near_start, 1, NA);
    if (e != cudaSuccess) {
        fail(F110_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e));
        f110_destroy(sim);
        return F110_ERR_CUDA;
    }
    memset(&sim->map, 0, sizeof(sim->map));
    *out = sim;
    return F110_OK;
}

void f110_destroy(F110Sim* sim) {
    if (!sim) return;
    Guard g(sim->cfg.device);
    if (sim->host_stream) { cudaStreamSynchronize(sim->host_stream); cudaStreamDestroy(sim->host_stream); }
    cudaFree(sim->state_blob); cudaFree(sim->scratch_blob); cudaFree(sim->d_tables); cudaFree(sim->d_map); cudaFree(sim->d_beam_tt);
    cudaFree(sim->d_views); cudaFree(sim->d_map_dir); cudaFree(sim->d_env_map);
    cudaFree(sim->io_blob);
    edt_scratch_free(&sim->edt);
    for (cudaEvent_t e : sim->tev) cudaEventDestroy(e);
    delete sim;
}

// The lidar kernel's direction tables [K][theta_dis] of the maps `views`: table direction k rotated into each map's frame and
// scaled to fixed-point cells per metre.  Depend on the sin / cos tables and on each map (origin yaw, resolution, fraction bits).
static std::vector<double2> direction_tables(const F110Sim* sim, const std::vector<MapView>& views) {
    const size_t n = sim->h_sines.size();
    std::vector<double2> dir(n * views.size());
    for (size_t v = 0; v < views.size(); ++v) {
        const MapView& m = views[v];
        for (size_t k = 0; k < n; ++k) {
            const double cs = sim->h_cosines[k], sn = sim->h_sines[k];
            dir[v * n + k].x = (cs * m.oc + sn * m.os) * m.inv_fx;
            dir[v * n + k].y = (-cs * m.os + sn * m.oc) * m.inv_fx;
        }
    }
    return dir;
}

// Fixed-point format of the lidar kernel's fast march for a map whose larger side is `side_cells`: as many fraction bits as
// a 32-bit coordinate leaves beside the cell index (+ 1: the map is stored one cell in from the padded array's corner).
// Fills fx_bits, guard, guard_mask, prows, pitch and fx_off.
static void fixed_point_format(const F110Sim* sim, unsigned side_cells, MapView& m) {
    auto bit_length = [](unsigned v) { unsigned b = 0; while ((v >> b) != 0u) ++b; return b; };
    const unsigned side = side_cells + 1u;
    m.fx_bits = 32u - bit_length(side) > 24u ? 24u : 32u - bit_length(side);
    m.guard = sim->narrow_fraction ? (1u << (m.fx_bits - 5u)) : 2u;     // F110_FLAG_NARROW_FRACTION: 1/16 of every cell undecided
    m.guard_mask = ((1u << m.fx_bits) - 1u) & ~(2u * m.guard - 1u);
    m.prows = 1 << (32u - m.fx_bits);
    m.pitch = m.prows + 16;
    m.fx_off = (double)(1u << m.fx_bits) - (double)m.guard;
}

// The per-map fields of a view in format `m` (dt, size, resolution, origin)
static void place_map(MapView& m, double* padded, int height, int width, double resolution,
                      double orig_x, double orig_y, double orig_cos, double orig_sin) {
    m.dt = padded; m.H = height; m.W = width;
    m.last = (height - 1) * width + (width - 1);
    m.res = resolution;
    m.inv_fx = (1.0 / resolution) * (double)(1u << m.fx_bits);
    m.ox = orig_x; m.oy = orig_y; m.oc = orig_cos; m.os = orig_sin;
    m.wres = width * resolution; m.hres = height * resolution;   // laser_models.py:79
}

// The dense fp64 map of a mask through the device EDT: DEVICE [H][W] in *out (caller frees), or an error code
static int dense_from_mask(F110Sim* sim, const uint8_t* free_mask, int32_t height, int32_t width, double resolution, double** out) {
    const size_t cells = (size_t)height * width;
    uint8_t* d_mask = nullptr;
    double* d = nullptr;
    *out = nullptr;
    CUDA_TRY(cudaMalloc(&d_mask, cells));
    cudaError_t e = cudaMalloc(&d, cells * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(d_mask, free_mask, cells, cudaMemcpyHostToDevice);
    int rc = -1;
    if (e == cudaSuccess) rc = edt_device(d_mask, height, width, resolution, d, &sim->edt, sim->host_stream);
    cudaFree(d_mask);
    if (e != cudaSuccess || rc != 0) { cudaFree(d); cudaGetLastError(); return fail(F110_ERR_CUDA, "device EDT failed"); }
    *out = d;
    return F110_OK;
}

int f110_set_map(F110Sim* sim, const double* dt, int32_t height, int32_t width, double resolution,
                 double orig_x, double orig_y, double orig_cos, double orig_sin) {
    const F110MapDesc d = { dt, nullptr, height, width, resolution, orig_x, orig_y, orig_cos, orig_sin };
    return f110_set_maps(sim, &d, 1);
}

int f110_set_map_image(F110Sim* sim, const uint8_t* free_mask, int32_t height, int32_t width, double resolution,
                       double orig_x, double orig_y, double orig_cos, double orig_sin) {
    const F110MapDesc d = { nullptr, free_mask, height, width, resolution, orig_x, orig_y, orig_cos, orig_sin };
    return f110_set_maps(sim, &d, 1);
}

float f110_edt_kernel_ms(const F110Sim* sim) { return sim ? sim->edt.kernel_ms : -1.f; }

// The one map installer: a single map is the set of one.  Everything is built aside and committed at the end, so a failure
// leaves the handle's maps as they were.
int f110_set_maps(F110Sim* sim, const F110MapDesc* maps, int32_t count) {
    if (!sim || !maps) return fail(F110_ERR_INVALID, "null argument");
    if (count < 1 || count > F110_MAX_MAPS) return fail(F110_ERR_INVALID, "a map set holds 1 to %d maps, not %d", F110_MAX_MAPS, count);
    unsigned side = 0;
    for (int k = 0; k < count; ++k) {
        const F110MapDesc& d = maps[k];
        if ((!d.dt && !d.free_mask) || d.height < 1 || d.width < 1 || !(d.resolution > 0))
            return fail(F110_ERR_INVALID, "bad arguments for map %d", k);
        if ((double)d.height * d.width >= 2147483648.0 || d.height >= 65536 || d.width >= 65536)
            return fail(F110_ERR_INVALID, "map %d too large (need H*W < 2^31 and H, W < 65536)", k);
        const unsigned s = (unsigned)(d.width > d.height ? d.width : d.height);
        side = s > side ? s : side;
    }
    // one fixed-point format for all maps, that of the largest side; every map padded to it, at a fixed stride
    MapView common;
    memset(&common, 0, sizeof(common));
    fixed_point_format(sim, side, common);
    const size_t stride = (size_t)common.prows * (size_t)common.pitch;
    if ((double)stride * count >= 2147483648.0)
        return fail(F110_ERR_INVALID, "maps too large: %d padded to %d x %d cells each (the largest side is %u) reach 2^31 cells",
                    count, common.prows, common.pitch, side);
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    double* padded = nullptr;
    MapView* d_views = nullptr;
    double2* d_dir = nullptr;
    const size_t nt = sim->h_sines.size();
    cudaError_t e = cudaMalloc(&padded, stride * count * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&d_views, (size_t)count * sizeof(MapView));
    if (e == cudaSuccess) e = cudaMalloc(&d_dir, (size_t)count * nt * sizeof(double2));
    auto undo = [&]() { cudaFree(padded); cudaFree(d_views); cudaFree(d_dir); cudaGetLastError(); };
    if (e != cudaSuccess) { undo(); return fail(F110_ERR_CUDA, "map allocation (%d x %zu cells): %s", count, stride, cudaGetErrorString(e)); }
    std::vector<MapView> views(count, common);
    double min_positive = INFINITY;
    for (int k = 0; k < count; ++k) {
        const F110MapDesc& d = maps[k];
        const size_t cells = (size_t)d.height * d.width;
        double* dense = nullptr;
        if (d.dt) {
            e = cudaMalloc(&dense, cells * sizeof(double));
            if (e == cudaSuccess) e = cudaMemcpy(dense, d.dt, cells * sizeof(double), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { cudaFree(dense); undo(); return fail(F110_ERR_CUDA, "upload of map %d: %s", k, cudaGetErrorString(e)); }
        } else {
            const int rc = dense_from_mask(sim, d.free_mask, d.height, d.width, d.resolution, &dense);
            if (rc != F110_OK) { undo(); return rc; }
        }
        MapView& v = views[k];
        double* block = padded + (size_t)k * stride;
        e = map_min_positive(dense, cells, &v.min_positive, sim->host_stream);
        if (e == cudaSuccess) e = launch_pad_map(dense, d.height, d.width, block, common.prows, common.pitch, sim->host_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(sim->host_stream);
        cudaFree(dense);
        if (e != cudaSuccess) { undo(); return fail(F110_ERR_CUDA, "padding of map %d: %s", k, cudaGetErrorString(e)); }
        place_map(v, block, d.height, d.width, d.resolution, d.orig_x, d.orig_y, d.orig_cos, d.orig_sin);
        min_positive = v.min_positive < min_positive ? v.min_positive : min_positive;
    }
    const std::vector<double2> dir = direction_tables(sim, views);
    e = cudaMemcpy(d_views, views.data(), views.size() * sizeof(MapView), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_dir, dir.data(), dir.size() * sizeof(double2), cudaMemcpyHostToDevice);
    // every env to its contiguous block: env e drives on slot floor(e K / N)
    std::vector<int32_t> slots(sim->c.N);
    for (int n = 0; n < sim->c.N; ++n) slots[n] = (int32_t)((int64_t)n * count / sim->c.N);
    if (e == cudaSuccess) e = cudaMemcpy(sim->d_env_map, slots.data(), slots.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { undo(); return fail(F110_ERR_CUDA, "map upload: %s", cudaGetErrorString(e)); }
    // commit
    cudaFree(sim->d_map); cudaFree(sim->d_views); cudaFree(sim->d_map_dir);
    sim->d_map = padded; sim->d_views = d_views; sim->d_map_dir = d_dir;
    sim->h_views = views;
    sim->map = views[0];
    sim->map.min_positive = min_positive;
    sim->c.dir_fx = d_dir;   // slot 0's table, which the single-map kernels read
    sim->ms.env_map = sim->d_env_map;
    sim->ms.views = d_views;
    sim->ms.dir_fx = d_dir;
    sim->ms.stride = stride;
    sim->map_count = count;
    sim->map_generation += 1;
    return F110_OK;
}

int32_t f110_map_count(const F110Sim* sim) { return sim ? sim->map_count : 0; }

int f110_get_map_slot(F110Sim* sim, int32_t slot, double* dt_host, int64_t capacity_cells) {
    if (!sim || !dt_host) return fail(F110_ERR_INVALID, "null argument");
    if (sim->map_count == 0) return fail(F110_ERR_MAP_NOT_SET, "Map is not set for scan simulator.");
    if (slot < 0 || slot >= sim->map_count) return fail(F110_ERR_INDEX, "map slot %d out of range (%d maps)", slot, sim->map_count);
    const MapView& m = sim->h_views[slot];
    const size_t cells = (size_t)m.H * m.W;
    if ((size_t)capacity_cells < cells) return fail(F110_ERR_INVALID, "buffer too small for %d x %d cells", m.H, m.W);
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy2D(dt_host, (size_t)m.W * sizeof(double), m.dt + m.pitch + 1, (size_t)m.pitch * sizeof(double),
                          (size_t)m.W * sizeof(double), (size_t)m.H, cudaMemcpyDeviceToHost));
    return F110_OK;
}

int f110_get_map(F110Sim* sim, double* dt_host, int64_t capacity_cells) { return f110_get_map_slot(sim, 0, dt_host, capacity_cells); }

int f110_set_env_maps(F110Sim* sim, const int32_t* slots, const uint8_t* env_mask, void* stream) {
    if (!sim || !slots) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    CUDA_TRY(launch_set_env_maps(sim->d_env_map, slots, env_mask, sim->c.N, sim->map_count, (cudaStream_t)stream));
    sim->launches += 1;
    return F110_OK;
}

int f110_set_env_maps_host(F110Sim* sim, const int32_t* slots, const uint8_t* env_mask) {
    if (!sim || !slots) return fail(F110_ERR_INVALID, "null argument");
    const int N = sim->c.N;
    for (int n = 0; n < N; ++n)
        if ((!env_mask || env_mask[n]) && (slots[n] < 0 || slots[n] >= sim->map_count))
            return fail(F110_ERR_INDEX, "env %d: map slot %d out of range (%d maps)", n, slots[n], sim->map_count);
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    int32_t* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, (size_t)N * sizeof(int32_t) + N));
    uint8_t* d_mask = env_mask ? reinterpret_cast<uint8_t*>(d + N) : nullptr;
    cudaStream_t s = sim->host_stream;
    cudaError_t e = cudaMemcpyAsync(d, slots, (size_t)N * sizeof(int32_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && env_mask) e = cudaMemcpyAsync(d_mask, env_mask, N, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = launch_set_env_maps(sim->d_env_map, d, d_mask, N, sim->map_count, s);
    if (e == cudaSuccess) { sim->launches += 1; e = cudaStreamSynchronize(s); }
    cudaFree(d);
    if (e != cudaSuccess) return fail(F110_ERR_CUDA, "f110_set_env_maps_host: %s", cudaGetErrorString(e));
    return F110_OK;
}

int f110_get_env_maps(F110Sim* sim, int32_t* slots_out, void* stream) {
    if (!sim || !slots_out) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaMemcpyAsync(slots_out, sim->d_env_map, (size_t)sim->c.N * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return F110_OK;
}

int f110_set_tables(F110Sim* sim, const double* sines, const double* cosines) {
    if (!sim || !sines || !cosines) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t n = sizeof(double) * sim->cfg.theta_dis;
    CUDA_TRY(cudaMemcpy(const_cast<double*>(sim->c.sines), sines, n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(const_cast<double*>(sim->c.cosines), cosines, n, cudaMemcpyHostToDevice));
    sim->h_sines.assign(sines, sines + sim->cfg.theta_dis);
    sim->h_cosines.assign(cosines, cosines + sim->cfg.theta_dis);
    const std::vector<double2> dir = direction_tables(sim, sim->h_views);   // empty before any map
    if (!dir.empty()) CUDA_TRY(cudaMemcpy(sim->d_map_dir, dir.data(), dir.size() * sizeof(double2), cudaMemcpyHostToDevice));
    return F110_OK;
}

int f110_set_beam_tables(F110Sim* sim, const double* scan_angles, const double* beam_cosines, const double* side_distances) {
    if (!sim || !scan_angles || !beam_cosines || !side_distances) return fail(F110_ERR_INVALID, "null argument");
    for (int i = 1; i < sim->cfg.num_beams; ++i)
        if (!(scan_angles[i] > scan_angles[i - 1])) return fail(F110_ERR_INVALID, "scan_angles must be strictly increasing");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t n = sizeof(double) * sim->cfg.num_beams;
    CUDA_TRY(cudaMemcpy(const_cast<double*>(sim->c.scan_angles), scan_angles, n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(const_cast<double*>(sim->c.beam_cos), beam_cosines, n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(const_cast<double*>(sim->c.side_dist), side_distances, n, cudaMemcpyHostToDevice));
    std::vector<double2> bt(sim->cfg.num_beams);
    for (int i = 0; i < sim->cfg.num_beams; ++i) { bt[i].x = beam_cosines[i]; bt[i].y = side_distances[i]; }
    CUDA_TRY(cudaMemcpy(const_cast<double2*>(sim->c.beam_tt), bt.data(), bt.size() * sizeof(double2), cudaMemcpyHostToDevice));
    // the scan-wide iTTC prefilter of the dynamics kernel: bounds over the tables (non-finite entries switch it off)
    double side_max = 0.0, cos_max = 0.0;
    for (int i = 0; i < sim->cfg.num_beams; ++i) {
        const double sd = side_distances[i], bc = fabs(beam_cosines[i]);
        side_max = sd > side_max || !(sd == sd) ? (sd == sd ? sd : INFINITY) : side_max;
        cos_max = bc > cos_max || !(bc == bc) ? (bc == bc ? bc : INFINITY) : cos_max;
    }
    sim->c.ttc_side_max = side_max;
    sim->c.ttc_cos_max = cos_max;
    return F110_OK;
}

int f110_set_params(F110Sim* sim, const double* params, int32_t agent_idx) {
    if (!sim || !params) return fail(F110_ERR_INVALID, "null argument");
    if (agent_idx >= sim->cfg.num_agents) return fail(F110_ERR_INDEX, "Index given is out of bounds for list of agents.");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    double* base = const_cast<double*>(sim->c.params);
    for (int a = 0; a < sim->cfg.num_agents; ++a)
        if (agent_idx < 0 || a == agent_idx)
            CUDA_TRY(cudaMemcpy(base + (size_t)a * F110_NUM_PARAMS, params, sizeof(double) * F110_NUM_PARAMS, cudaMemcpyHostToDevice));
    return F110_OK;
}

int f110_sim_reset(F110Sim* sim, const double* poses, int32_t num_poses, const uint8_t* env_mask, void* stream) {
    if (!sim || !poses) return fail(F110_ERR_INVALID, "null argument");
    if (num_poses != sim->cfg.num_agents) return fail(F110_ERR_POSE_COUNT, "Number of poses for reset does not match number of agents.");
    Guard g(sim->cfg.device);
    CUDA_TRY(launch_sim_reset(sim->c, sim->st, poses, env_mask, (cudaStream_t)stream));
    sim->launches += 1;
    return F110_OK;
}

int f110_sim_reset_host(F110Sim* sim, const double* poses, int32_t num_poses, const uint8_t* env_mask) {
    if (!sim || !poses) return fail(F110_ERR_INVALID, "null argument");
    if (num_poses != sim->cfg.num_agents) return fail(F110_ERR_POSE_COUNT, "Number of poses for reset does not match number of agents.");
    Guard g(sim->cfg.device);
    const size_t N = sim->c.N, NA = sim->c.NA;
    double* d_poses = nullptr;
    CUDA_TRY(cudaMalloc(&d_poses, NA * 3 * sizeof(double) + N));
    uint8_t* d_mask = env_mask ? reinterpret_cast<uint8_t*>(d_poses + NA * 3) : nullptr;
    cudaStream_t s = sim->host_stream;
    cudaError_t e = cudaMemcpyAsync(d_poses, poses, NA * 3 * sizeof(double), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && env_mask) e = cudaMemcpyAsync(d_mask, env_mask, N, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        e = launch_sim_reset(sim->c, sim->st, d_poses, d_mask, s);
        sim->launches += 1;
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    }
    cudaFree(d_poses);
    if (e != cudaSuccess) return fail(F110_ERR_CUDA, "f110_sim_reset_host: %s", cudaGetErrorString(e));
    return F110_OK;
}

int f110_step(F110Sim* sim, const F110StepIO* io, void* stream) {
    const int rc = check_step_io(sim, io);
    if (rc != F110_OK) return rc;
    Guard g(sim->cfg.device);
    return run_step(sim, *io, (cudaStream_t)stream);
}

namespace {
// One host<->device transfer of the host path.  The device mirrors of the fields present in a call are packed back to
// back in io_blob in a fixed order (see f110_step_host_async), so transfers whose HOST buffers are also exactly adjacent,
// in that order, travel as one cudaMemcpyAsync when the caller vouches for them (F110_HOST_MERGE_ADJACENT): a caller that carves its pinned buffers out of one block per direction
// (F110HostVecEnv does) pays one PCIe transaction each way per step instead of one per field.
struct Xfer { char* host; char* dev; size_t bytes; };

int run_xfers(const Xfer* x, int n, bool merge, cudaMemcpyKind kind, cudaStream_t s) {
    for (int i = 0; i < n;) {
        size_t bytes = x[i].bytes;
        int j = i + 1;
        while (merge && j < n && x[j].host == x[i].host + bytes && x[j].dev == x[i].dev + bytes) bytes += x[j++].bytes;
        if (kind == cudaMemcpyHostToDevice) CUDA_TRY(cudaMemcpyAsync(x[i].dev, x[i].host, bytes, kind, s));
        else CUDA_TRY(cudaMemcpyAsync(x[i].host, x[i].dev, bytes, kind, s));
        i = j;
    }
    return F110_OK;
}
}  // namespace

int f110_step_host_async(F110Sim* sim, const F110StepIO* hio) {
    const int rc = check_step_io(sim, hio);
    if (rc != F110_OK) return rc;
    Guard g(sim->cfg.device);
    const size_t N = sim->c.N, NA = sim->c.NA, B = sim->c.B;
    if (!sim->io_blob) {
        // room for the device mirror of every field of F110StepIO at once, allocated on first use
        sim->io_bytes = NA * 2 * 8 + NA * B * 8 + N + NA * 3 * 8 + N                       // inputs
                      + N * (B + 8) * 4 + N * 4 + N + NA * B * 8 + NA * B * 4 + NA * 7 * 8 + NA * 3 * 8  // outputs
                      + NA + NA * 4 + NA * 8 + NA * 8 + N * 8 + 4096;
        CUDA_TRY(cudaMalloc(&sim->io_blob, sim->io_bytes));
    }
    cudaStream_t s = sim->host_stream;
    F110StepIO d = *hio;
    Xfer in[5], out[12];
    int n_in = 0, n_out = 0;
    char* cur = sim->io_blob;
    // field present in the caller's struct -> next slot of io_blob; the device-side struct points there
#define SLOT(list, count, field, nbytes)                                                           \
    if (hio->field) {                                                                              \
        list[count++] = Xfer{(char*)(uintptr_t)hio->field, cur, (size_t)(nbytes)};                 \
        d.field = (decltype(d.field))cur;                                                          \
        cur += (nbytes);                                                                           \
    }
    // inputs, in merge order: actions, reset_poses, noise (8-byte multiples), reset_mask, active_mask (bytes)
    SLOT(in, n_in, actions, NA * 2 * (hio->actions_f64 ? sizeof(double) : sizeof(float)))
    SLOT(in, n_in, reset_poses, NA * 3 * sizeof(double))
    SLOT(in, n_in, noise, NA * B * sizeof(double))
    SLOT(in, n_in, reset_mask, N)
    SLOT(in, n_in, active_mask, N)
    cur = sim->io_blob + (((size_t)(cur - sim->io_blob) + 255) & ~size_t(255));
    // outputs, in merge order: the 8-byte fields, then the 4-byte ones, then the byte arrays -- no padding is ever needed
    // between two of them.  (With only obs / reward / terminated requested, obs sits at the 256-byte aligned start.)
    SLOT(out, n_out, scans_f64, NA * B * sizeof(double))
    SLOT(out, n_out, state, NA * 7 * sizeof(double))
    SLOT(out, n_out, agent_poses, NA * 3 * sizeof(double))
    SLOT(out, n_out, lap_times, NA * sizeof(double))
    SLOT(out, n_out, lap_counts, NA * sizeof(double))
    SLOT(out, n_out, time, N * sizeof(double))
    SLOT(out, n_out, obs, N * (B + 8) * sizeof(float))
    SLOT(out, n_out, scans_f32, NA * B * sizeof(float))
    SLOT(out, n_out, reward, N * sizeof(float))
    SLOT(out, n_out, toggles, NA * sizeof(int32_t))
    SLOT(out, n_out, terminated, N)
    SLOT(out, n_out, collisions, NA)
#undef SLOT
    const bool merge = (hio->host_flags & F110_HOST_MERGE_ADJACENT) != 0;
    int rc2 = run_xfers(in, n_in, merge, cudaMemcpyHostToDevice, s);
    if (rc2 != F110_OK) return rc2;
    rc2 = run_step(sim, d, s);
    if (rc2 != F110_OK) return rc2;
    return run_xfers(out, n_out, merge, cudaMemcpyDeviceToHost, s);
}

int f110_host_sync(F110Sim* sim) {
    if (!sim) return fail(F110_ERR_INVALID, "null handle");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaStreamSynchronize(sim->host_stream));
    return F110_OK;
}

int f110_step_host_multi(F110Sim* const* sims, const F110StepIO* ios, int32_t count) {
    if (!sims || !ios || count < 1) return fail(F110_ERR_INVALID, "bad arguments");
    for (int i = 0; i < count; ++i) {
        const int rc = f110_step_host_async(sims[i], &ios[i]);
        if (rc != F110_OK) return rc;
    }
    for (int i = 0; i < count; ++i) {
        const int rc = f110_host_sync(sims[i]);
        if (rc != F110_OK) return rc;
    }
    return F110_OK;
}

int f110_step_host(F110Sim* sim, const F110StepIO* hio) {
    const int rc = f110_step_host_async(sim, hio);
    if (rc != F110_OK) return rc;
    return f110_host_sync(sim);
}

// A checkpoint is a 64-byte header followed by the state arena.  The header names the layout, so that a blob from another
// build or another batch shape is refused instead of being copied over the arena.
namespace {
struct CheckpointHeader {
    uint32_t magic;      // 'F110'
    uint32_t layout;     // bumped whenever layout_state changes
    int32_t N, A, B;
    uint32_t reserved;
    uint64_t state_bytes;
    uint64_t pad[4];
};
static_assert(sizeof(CheckpointHeader) == 64, "checkpoint header is 64 bytes");
constexpr uint32_t CKPT_MAGIC = 0x30313146u, CKPT_LAYOUT = 2u;
CheckpointHeader checkpoint_header(const F110Sim* sim) {
    CheckpointHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = CKPT_MAGIC; h.layout = CKPT_LAYOUT;
    h.N = sim->c.N; h.A = sim->c.A; h.B = sim->c.B;
    h.state_bytes = sim->state_bytes;
    return h;
}
}  // namespace

int64_t f110_state_nbytes(const F110Sim* sim) { return sim ? (int64_t)(sizeof(CheckpointHeader) + sim->state_bytes) : 0; }

int f110_get_state(F110Sim* sim, void* dst, void* stream) {
    if (!sim || !dst) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    const CheckpointHeader hd = checkpoint_header(sim);
    memcpy(sim->ckpt_header_words, &hd, sizeof(hd));   // staged in the handle: the asynchronous copy reads it later
    CUDA_TRY(cudaMemcpyAsync(dst, sim->ckpt_header_words, sizeof(CheckpointHeader), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(dst) + sizeof(CheckpointHeader), sim->state_blob, sim->state_bytes,
                             cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return F110_OK;
}

int f110_set_state(F110Sim* sim, const void* src, void* stream) {
    if (!sim || !src) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    CheckpointHeader h;
    CUDA_TRY(cudaMemcpyAsync(&h, src, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    const CheckpointHeader want = checkpoint_header(sim);
    if (h.magic != want.magic) return fail(F110_ERR_INVALID, "not an f110 checkpoint (bad magic)");
    if (h.layout != want.layout) return fail(F110_ERR_INVALID, "checkpoint layout %u, this library reads layout %u", h.layout, want.layout);
    if (h.N != want.N || h.A != want.A || h.B != want.B || h.state_bytes != want.state_bytes)
        return fail(F110_ERR_INVALID, "checkpoint is for %d envs x %d agents x %d beams, this handle has %d x %d x %d", h.N, h.A, h.B,
                    want.N, want.A, want.B);
    CUDA_TRY(cudaMemcpyAsync(sim->state_blob, static_cast<const char*>(src) + sizeof(CheckpointHeader), sim->state_bytes,
                             cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return F110_OK;
}

int f110_get_stats(F110Sim* sim, double* out, int32_t reset, void* stream) {
    if (!sim || !out) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    cudaStream_t s = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(out, sim->sc.stats, sizeof(double) * F110_NUM_STATS, cudaMemcpyDeviceToDevice, s));
    if (reset) CUDA_TRY(cudaMemsetAsync(sim->sc.stats, 0, sizeof(double) * F110_NUM_STATS, s));
    return F110_OK;
}

int f110_get_lookup_count(F110Sim* sim, uint64_t* lookups, uint64_t* rays) {
    if (!sim || !lookups || !rays) return fail(F110_ERR_INVALID, "null argument");
    if (!sim->count_lookups) return fail(F110_ERR_INVALID, "handle was created without F110_FLAG_COUNT_LOOKUPS");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    unsigned long long h[4];
    CUDA_TRY(cudaMemcpy(h, sim->sc.lookups, sizeof(h), cudaMemcpyDeviceToHost));
    *lookups = h[0]; *rays = h[1];
    sim->max_lookups = h[2];
    sim->redone_rays = h[3];
    return F110_OK;
}

int64_t f110_debug_unit_timeline(F110Sim* sim, uint32_t* out, int64_t capacity_units) {
    if (!sim) return 0;
    if (!out) return sim->sc.timeline ? (int64_t)sim->sc.num_units : 0;
    if (!sim->sc.timeline || capacity_units < (int64_t)sim->sc.num_units) return fail(F110_ERR_INVALID, "no timeline (F110_FLAG_COUNT_LOOKUPS) or buffer too small");
    Guard g(sim->cfg.device);
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out, sim->sc.timeline, (size_t)sim->sc.num_units * 16, cudaMemcpyDeviceToHost));
    return (int64_t)sim->sc.num_units;
}

int f110_set_kernel_timing(F110Sim* sim, int32_t enable) {
    if (!sim) return fail(F110_ERR_INVALID, "null handle");
    sim->timing = enable != 0;
    return F110_OK;
}

int f110_get_kernel_timing(F110Sim* sim, double* ms3, int64_t* steps) {
    if (!sim || !ms3 || !steps) return fail(F110_ERR_INVALID, "null argument");
    Guard g(sim->cfg.device);
    ms3[0] = ms3[1] = ms3[2] = 0.0;
    *steps = (int64_t)(sim->tev.size() / 4);
    for (size_t i = 0; i + 3 < sim->tev.size(); i += 4) {
        CUDA_TRY(cudaEventSynchronize(sim->tev[i + 3]));
        for (int k = 0; k < 3; ++k) {
            float ms = 0.f;
            CUDA_TRY(cudaEventElapsedTime(&ms, sim->tev[i + k], sim->tev[i + k + 1]));
            ms3[k] += ms;
        }
    }
    for (cudaEvent_t e : sim->tev) cudaEventDestroy(e);
    sim->tev.clear();
    return F110_OK;
}

int64_t f110_max_lookups(const F110Sim* sim) { return sim ? (int64_t)sim->max_lookups : 0; }
int64_t f110_redone_rays(const F110Sim* sim) { return sim ? (int64_t)sim->redone_rays : 0; }
int f110_get_lidar_variant(const F110Sim* sim, int32_t out[4]) {
    if (!sim || !out) return fail(F110_ERR_INVALID, "null argument");
    if (!sim->lidar_ran) return fail(F110_ERR_INVALID, "no step has run on this handle yet");
    memcpy(out, sim->lidar_variant, sizeof(sim->lidar_variant));
    return F110_OK;
}
int64_t f110_map_generation(const F110Sim* sim) { return sim ? sim->map_generation : 0; }

int64_t f110_kernel_launches(const F110Sim* sim) { return sim ? sim->launches : 0; }

}  // extern "C"
