// f110_kernels.cuh -- device-side data model shared by the step kernels and the C ABI.
//
// Everything on the step path is fp64 evaluated in the reference's operator order with FMA
// contraction disabled (-fmad=false): numba's code for the reference contains no fused
// multiply-adds, and the ray-march's cell lookups are discontinuous in the last bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "f110_b200.h"

#define F110_PI 3.141592653589793  // numpy.pi

// Distance-transform map (laser_models.py:383-427).  Row 0 is the BOTTOM image row.
//
// Device layout: cell (r, c) of the H x W map sits at [r + 1][c + 1] of a PADDED array of prows x pitch cells whose other
// cells hold the sentinel -1.0.  prows = 2^(32 - fx_bits) is everything a 32-bit fixed-point coordinate with fx_bits
// fraction bits can address, so the lidar kernel's hot loop needs no in-map test: a lookup off the map -- including the
// negative and NaN coordinates that convert to 0, i.e. row / column 0 -- reads a sentinel, which ends the loop like any
// d <= eps, and the ray is then redone in the reference's arithmetic.  pitch = prows + 16 keeps vertically adjacent cells
// off a power-of-two stride.
struct MapView {
    const double* dt;   // [prows][pitch] metres to the nearest obstacle; sentinel outside [1, H] x [1, W]
    int H, W;
    int pitch, prows;
    int last;           // (H-1)*W + (W-1): the DENSE index numba's negative-index wrap lands on (SURVEY 7.4)
    double res;         // metres per cell
    double inv_fx;      // 2^fx_bits / res: map-frame metres -> fixed-point cells
    double fx_off;      // 2^fx_bits - guard: the fixed-point coordinates are shifted by one cell minus the guard width, so
                        //   that "fraction >= 2^fx_bits - 2 guard" alone says "within guard of a cell edge" (either edge)
    unsigned fx_bits;   // fraction bits: 32 - bit_length(max(W, H) + 1), at most 24
    unsigned guard;     // (power of two) a lookup whose fraction is within `guard` units of a cell edge is not decided by the fast path
    unsigned guard_mask;  // fraction bits above 2 guard: all of them set <=> inside the guard band
    double min_positive;  // smallest positive cell value (set_map computes it): > eps lets the march test d > 0
    double ox, oy, oc, os;
    double wres, hres;  // W*res, H*res
};

// A map set (f110_set_maps): K maps in one handle, each env on the map of its slot.  Every map is padded to the set's
// common fixed-point format (fx_bits of the largest side, so prows, pitch and guard_mask are shared) and the K padded
// blocks lie back to back at a stride of prows * pitch cells: a slot's cells start at the set MapView's dt + slot * stride.
// What differs per slot is in views[slot] (origin, resolution, inv_fx, H, W, dt of its own block) and in its direction table.
struct MapSet {
    const int32_t* env_map;   // [N] slot of each env
    const MapView* views;     // [K] per-slot descriptors
    const double2* dir_fx;    // [K][theta_dis] slot k's direction table (SimConst::dir_fx is slot 0's)
    size_t stride;            // cells between the blocks of two consecutive slots
};

// Persistent simulation state: one arena, SoA over s = env*A + agent (coalesced for one thread
// per vehicle) and over env.  Everything a checkpoint needs lives between arena and arena+nbytes.
struct SimState {
    double* x[7];       // [NA] x, y, steer, v, yaw, yaw_rate, slip        base_classes.py:97-98
    double* steer_buf0; // [NA] newest queued steering command             base_classes.py:270-278
    double* steer_buf1; // [NA] oldest queued steering command
    double* start_x;    // [NA] f110_env.py:448-450
    double* start_y;
    double* start_th;
    double* lap_times;  // [NA] f110_env.py:346-348
    double* lap_counts; // [NA]
    double* time;       // [N]  f110_env.py:406
    double* rot_c;      // [N]  cos(-start_theta[ego])                      f110_env.py:451
    double* rot_s;      // [N]  sin(-start_theta[ego])
    int32_t* steer_cnt; // [NA] entries queued in the delay FIFO (0..2)
    int32_t* toggles;   // [NA] f110_env.py:339-346
    uint32_t* step_count; // [N] steps since the env's reset (Philox counter)
    uint8_t* near_start;  // [NA]
    uint8_t* collisions;  // [NA] last step's GJK | iTTC
};

// Scratch carried between the three kernels of one step (not part of a checkpoint).
struct StepScratch {
    double* scan_x;     // [NA] lidar pose for this step (base_classes.py:420-422)
    double* scan_y;
    double* pre_yaw;    // [NA] yaw after dynamics, BEFORE iTTC zeroing (Simulator.agent_poses, :587)
    double* head;       // [NA][4] per scan, for the lidar kernel: fixed-point map-frame start X, Y; wrapped theta index of beam 0
                        //          (laser_models.py:167-172); the range above which no beam of the scan can trip the iTTC test
    int32_t* ttc_hit;   // [NA] set by the lidar kernel
    unsigned long long* lookups;  // [4] dt lookups, rays, longest ray, rays redone exactly (only with F110_FLAG_COUNT_LOOKUPS)
    double* stats;      // [F110_NUM_STATS]
    uint4* timeline;    // [num_units] or null: (start ns, end ns, longest ray, sm << 24 | queue position) of each unit in the
                        //   last lidar launch; written only by the F110_FLAG_COUNT_LOOKUPS variant (tools/unit_timeline.py)
    // work queue and launch-order history of the lidar kernel (see lidar_kernel)
    unsigned num_units;        // NA * ceil(B / 32) warp-sized work units (32 consecutive beams of one scan)
    unsigned ordered;          // 1: longest-first launch order kept (batches of up to 48 units per resident warp; beyond that the
                               //    tail it saves is below 2 % of the launch and the list atomics cost more), 0: natural order
    unsigned homes;            // segments of the unit range, each with its own queue: one per SM for launches without the
                               //   longest-first order, else one (see lidar_kernel)
    unsigned seg_units;        // units per segment: segment g is units [g seg_units, (g + 1) seg_units) (the last one may be short)
    const unsigned* home_of_sm;  // [F110_SMID_TABLE] home segment of the warps that run on SM smid (f110_create probes the ids)
    unsigned cap[3];           // capacity of the three heavy-unit lists
    unsigned* ctrl;            // [ctrl_words(homes)]: counts being recorded, parity, latched counts, the segments' queue positions
    unsigned* list[2];         // [parity][cap0 + cap1 + cap2] unit ids, heaviest class first
    unsigned* cls[2];          // [parity][num_units] class of each unit: 0..2 = on that list, >= 3 = light (natural order); 4 / 5 =
                               //   processed, alternating every second step (see lidar_kernel)
};
// the words atomics hit (the three counts being recorded, each segment's queue position) sit on 128-byte lines of their own
enum { CTRL_NEXT = 32, CTRL_NEXT_STRIDE = 32, CTRL_EPOCH = 128, CTRL_CUR = 129, CTRL_SEG = 160, SEG_STRIDE = 32,
       F110_SMID_TABLE = 1024 };
inline size_t ctrl_words(unsigned homes) { return CTRL_SEG + (size_t)homes * SEG_STRIDE; }

struct FastDiv { uint32_t mul, sh1, sh2; };   // n / d == (t + ((n - t) >> sh1)) >> sh2 with t = umulhi(n, mul)

struct SimConst {
    int N, A, B, NA;
    int theta_dis, integrator, ego;
    double fov, eps, max_range, timestep, lidar_dist, ttc_thresh, noise_std;
    double theta_inc;   // theta_dis * (fov/(B-1)) / (2 pi)               laser_models.py:367-368
    float lidar_max;
    uint64_t seed;
    uint32_t noise_key;  // Philox key derived from seed
    FastDiv div_B, div_A;
    unsigned ups;        // lidar work units per scan: ceil(B / 32)
    FastDiv div_ups;
    uint32_t philox_key[10];   // noise_key + r * 0x9E3779B9, the ten round keys of Philox2x32-10
    float obs_rcp;       // float(1 / lidar_max)
    int obs_fast_div;    // lidar_max == 30.0f: the observation's division runs through obs_rcp (see obs_lidar)
    const double* params;      // [A][18]
    const double* sim_params;  // [18] Simulator.params (construction time; base_classes.py:562)
    const double* sines;       // [theta_dis]
    const double* cosines;     // [theta_dis]
    const double* scan_angles; // [B]
    const double* beam_cos;    // [B]
    const double* side_dist;   // [B]
    const double2* beam_tt;    // [B] (beam_cos, side_dist) interleaved for the lidar kernel
    double ttc_side_max, ttc_cos_max;   // max side_dist, max |beam_cos| (+inf until the beam tables are set: nothing is pre-filtered)
    const double2* dir_fx;     // [theta_dis] table direction k rotated into the map frame and scaled to fixed point:
                               //   ((cos*oc + sin*os) * inv_fx, (-cos*os + sin*oc) * inv_fy); slot 0's table of
                               //   MapSet::dir_fx, rebuilt by set_map(s) / set_tables
};

// ms == nullptr: the handle holds one map (m); otherwise m is the set's common view (slot 0's, min_positive over the set)
cudaError_t launch_dynamics(const SimConst& c, const MapView& m, const SimState& st, const StepScratch& sc, const F110StepIO& io,
                            const MapSet* ms, cudaStream_t s);
int lidar_resident_blocks(bool single_agent);
// seen[k] = 1 for every SM id k < F110_SMID_TABLE a wave of the device's CTAs ran on (host array); synchronises
cudaError_t probe_sm_ids(unsigned char* seen);
// variant[4] (host): what the launch selected, as f110_get_lidar_variant reports it
cudaError_t launch_lidar(const SimConst& c, const MapView& m, const SimState& st, const StepScratch& sc, const F110StepIO& io,
                         const MapSet* ms, bool count_lookups, int resident_blocks, int32_t* variant, cudaStream_t s);
// env_map[e] = slots[e] for every env e with (mask == nullptr || mask[e]) and 0 <= slots[e] < count (all DEVICE pointers)
cudaError_t launch_set_env_maps(int32_t* env_map, const int32_t* slots, const uint8_t* mask, int N, int count, cudaStream_t s);
// smallest positive value of a dense device map (set_map time); synchronises the stream
cudaError_t map_min_positive(const double* dense, size_t cells, double* out, cudaStream_t s);
cudaError_t launch_post(const SimConst& c, const SimState& st, const StepScratch& sc, const F110StepIO& io, cudaStream_t s);
cudaError_t launch_sim_reset(const SimConst& c, const SimState& st, const double* poses, const uint8_t* mask, cudaStream_t s);
// dense [H][W] -> padded [prows][pitch] with the sentinel -1.0 outside the map (both DEVICE pointers)
cudaError_t launch_pad_map(const double* dense, int H, int W, double* padded, int prows, int pitch, cudaStream_t s);

// exact EDT on the device (f110_edt.cu): freemask DEVICE [H][W] (non-zero = free), dt DEVICE fp64 [H][W]; synchronises.
// The scratch (12 bytes per cell) stays with the caller's handle and is reused by the next call.
struct EdtScratch {
    void* base = nullptr;
    size_t bytes = 0;
    void* ev0 = nullptr;
    void* ev1 = nullptr;
    float kernel_ms = 0.f;   // the EDT kernels of the last call, by CUDA events
};
int edt_device(const uint8_t* freemask, int H, int W, double resolution, double* dt, EdtScratch* scratch, cudaStream_t stream);
void edt_scratch_free(EdtScratch* scratch);
int f110_set_error(int code, const char* msg);   // sets the thread-local message of f110_last_error(); returns code
