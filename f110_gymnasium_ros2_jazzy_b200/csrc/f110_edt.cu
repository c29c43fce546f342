// f110_edt.cu -- exact Euclidean distance transform on the device (SURVEY 8f row 3).
//
// The reference builds its map with scipy.ndimage.distance_transform_edt(img) * resolution on the host
// (laser_models.py:40-53,383-427; 0.3 s for a 2000 x 2000 map, 6 s for 8000 x 8000).  scipy returns sqrt(d2) of the exact
// integer squared distance d2 to the nearest obstacle pixel, so dt = resolution * sqrt((double)d2) with IEEE sqrt and
// multiply is bit-identical to the reference's array.  d2 is computed exactly, in integers, with the two-phase algorithm
// of Meijster, Roerdink & Hesselink (2000): (1) per column, the vertical distance g to the nearest obstacle; (2) per row,
// the lower envelope of the parabolas (x - i)^2 + g(i)^2.
//
// Four kernels, all but one a thread per cell or better:
//   band masks   one thread per (64-row band, column): the band's obstacle bits as one 64-bit word         H*W bytes read
//   columns      one thread per (band, column): g for the band's 64 rows from its own word (clz / ffs) and the nearest
//                non-empty words above and below; written TRANSPOSED (gT[column][row], 16 bit) so that the envelope
//                pass reads it coalesced                                                                      2 H*W written
//   envelope     one thread per row, W sequential steps (the stack algorithm is a serial chain per row: this is the
//                latency-bound kernel -- rows are the only parallelism it has, so every row gets a lane and nothing
//                else is left in it): the top of the stack lives in registers, the rest in the thread's own strip
//                of scratch; instead of the serial fill loop it leaves MARKS: marks[row][t] = 1 + stack index of the
//                parabola that takes over at column t (cleared again when that entry is popped)
//   fill         one thread per 4 cells: running maximum of the marks along the row (block scan) = the owning stack
//                entry of every cell -> d2 -> resolution * sqrt(d2), coalesced                                8 H*W written
// Scratch (band words, gT, stacks, marks: 12 bytes per cell) is kept on the handle and reused across calls.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "f110_kernels.cuh"

namespace {

constexpr int BAND = 64;

// any_obstacle: set to 1 when the band holds an obstacle (the caller clears it)
__global__ void __launch_bounds__(128) edt_band_masks_kernel(const uint8_t* __restrict__ freemask, int H, int W,
                                                             unsigned long long* __restrict__ words, unsigned* __restrict__ any_obstacle) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= W) return;
    const int r0 = blockIdx.y * BAND;
    unsigned long long m = 0;
#pragma unroll 16
    for (int j = 0; j < BAND; ++j) {
        const int r = r0 + j;
        if (r < H && freemask[(size_t)r * W + c] == 0) m |= 1ull << j;
    }
    words[(size_t)blockIdx.y * W + c] = m;
    const unsigned active = __activemask();
    if (__any_sync(active, m != 0ull) && (threadIdx.x & 31u) == (unsigned)(__ffs(active) - 1)) *any_obstacle = 1u;
}

// g(row, column) = distance along the column to the nearest obstacle (0 on one), `inf` if the column has none
__global__ void __launch_bounds__(128) edt_columns_kernel(const unsigned long long* __restrict__ words, int W, int NB, int Hp,
                                                          unsigned inf, uint16_t* __restrict__ gT) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= W) return;
    const int b = blockIdx.y;
    const unsigned long long m = words[(size_t)b * W + c];
    // U: from the row above the band to the nearest obstacle at or above it; D: likewise below.  `inf` when there is none
    // (any sum with it is capped at inf below).
    unsigned U = inf, D = inf;
    for (int bb = b - 1; bb >= 0; --bb) {
        const unsigned long long mm = words[(size_t)bb * W + c];
        if (mm) { U = (unsigned)((b - bb) * BAND - 1 - (63 - __clzll((long long)mm))); break; }
    }
    for (int bb = b + 1; bb < NB; ++bb) {
        const unsigned long long mm = words[(size_t)bb * W + c];
        if (mm) { D = (unsigned)((bb - b - 1) * BAND + (__ffsll((long long)mm) - 1)); break; }
    }
    uint4* out = reinterpret_cast<uint4*>(gT + (size_t)c * Hp + (size_t)b * BAND);
#pragma unroll
    for (int k = 0; k < BAND / 8; ++k) {
        unsigned v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int j = 8 * k + e;
            const unsigned long long up = m << (63 - j), dn = m >> j;
            const unsigned du = up ? (unsigned)__clzll((long long)up) : (unsigned)(j + 1) + U;
            const unsigned dd = dn ? (unsigned)(__ffsll((long long)dn) - 1) : (unsigned)(BAND - j) + D;
            const unsigned d = du < dd ? du : dd;
            v[e] = d < inf ? d : inf;
        }
        out[k] = make_uint4(v[0] | (v[1] << 16), v[2] | (v[3] << 16), v[4] | (v[5] << 16), v[6] | (v[7] << 16));
    }
}

// One stack entry: site s, first column t it owns, g(s).  8 bytes: {s | t << 16, g}
__device__ __forceinline__ uint2 pack_entry(int s, int t, int g) { return make_uint2((unsigned)s | ((unsigned)t << 16), (unsigned)g); }

// Lower envelope of one row (Meijster et al., phase 2, first loop).  All quantities fit 31 bits: H + W + 1 <= 32767.
__global__ void __launch_bounds__(32) edt_envelope_kernel(const uint16_t* __restrict__ gT, int H, int W, int Hp, int Wp,
                                                          uint2* __restrict__ stacks, uint16_t* __restrict__ marks) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= H) return;
    const uint16_t* g = gT + r;
    uint2* st = stacks + (size_t)r * W;
    uint16_t* mk = marks + (size_t)r * Wp;
    int q = 0, ts = 0, tt = 0, tg = g[0];          // the top of the stack, in registers
    st[0] = pack_entry(0, 0, tg);
    mk[0] = 1;
    int gnext = W > 1 ? g[(size_t)Hp] : 0;
    for (int u = 1; u < W; ++u) {
        const int gu = gnext;
        if (u + 1 < W) gnext = g[(size_t)(u + 1) * Hp];      // independent of the chain below: in flight while it runs
        const int gu2 = gu * gu;
        // pop while the top's parabola is above u's at the column where the top takes over
        for (;;) {
            const int fa = (tt - ts) * (tt - ts) + tg * tg;
            const int fb = (tt - u) * (tt - u) + gu2;
            if (fa <= fb) break;
            if (q > 0) mk[tt] = 0;
            --q;
            if (q < 0) break;
            const uint2 e = st[q];
            ts = (int)(e.x & 0xFFFFu); tt = (int)(e.x >> 16); tg = (int)e.y;
        }
        if (q < 0) {
            q = 0; ts = u; tt = 0; tg = gu;
            st[0] = pack_entry(u, 0, gu);
        } else {
            // Sep(s, u) = (u^2 - s^2 + g(u)^2 - g(s)^2) div (2 (u - s)): non-negative here
            const unsigned num = (unsigned)((u * u - ts * ts) + (gu2 - tg * tg));
            const int w = 1 + (int)(num / (unsigned)(2 * (u - ts)));
            if (w < W) {
                ++q; ts = u; tt = w; tg = gu;
                st[q] = pack_entry(u, w, gu);
                mk[w] = (uint16_t)(q + 1);
            }
        }
    }
}

constexpr int FILL_THREADS = 256;

// A mask without any obstacle: scipy's distance_transform_edt then measures every pixel from a virtual obstacle at
// (-1, 0), just outside the first row (checked against scipy 1.18 at several shapes): d2 = (row + 1)^2 + column^2.
__device__ __forceinline__ void edt_fill_row_without_obstacle(int r, int W, int x0, int step, double resolution, double* out) {
    for (int x = x0; x < W; x += step)
        out[x] = resolution * sqrt((double)((long long)(r + 1) * (r + 1) + (long long)x * x));
}

// marks -> owning entry of every cell (running maximum along the row: stack indices grow with t) -> distance
__global__ void __launch_bounds__(FILL_THREADS) edt_fill_kernel(const uint2* __restrict__ stacks, const uint16_t* __restrict__ marks,
                                                                int W, int Wp, double resolution, const unsigned* __restrict__ any_obstacle,
                                                                double* __restrict__ dt) {
    const int r = blockIdx.x;
    const uint2* st = stacks + (size_t)r * W;
    const uint16_t* mk = marks + (size_t)r * Wp;
    double* out = dt + (size_t)r * W;
    if (*any_obstacle == 0u) { edt_fill_row_without_obstacle(r, W, threadIdx.x, FILL_THREADS, resolution, out); return; }
    __shared__ unsigned s_warp[FILL_THREADS / 32];
    __shared__ unsigned s_carry;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int x0 = 0; x0 < W; x0 += 4 * FILL_THREADS) {
        const int x = x0 + 4 * threadIdx.x;
        unsigned m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        if (x < Wp) {                                   // Wp is a multiple of 4 and the pad is zero
            const uint2 v = *reinterpret_cast<const uint2*>(mk + x);
            m0 = v.x & 0xFFFFu; m1 = v.x >> 16; m2 = v.y & 0xFFFFu; m3 = v.y >> 16;
        }
        m1 = max(m1, m0); m2 = max(m2, m1); m3 = max(m3, m2);
        unsigned run = m3;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned other = __shfl_up_sync(0xffffffffu, run, o);
            if (lane >= o) run = max(run, other);
        }
        if (lane == 31) s_warp[wid] = run;
        __syncthreads();
        unsigned before = s_carry;                       // everything left of this thread's 4 cells
        for (int k = 0; k < wid; ++k) before = max(before, s_warp[k]);
        const unsigned left = __shfl_up_sync(0xffffffffu, run, 1);
        if (lane > 0) before = max(before, left);
        __syncthreads();
        if (threadIdx.x == FILL_THREADS - 1) s_carry = max(before, m3);
        const unsigned own[4] = { max(before, m0), max(before, m1), max(before, m2), max(before, m3) };
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (x + e < W) {
                const uint2 ent = st[own[e] - 1u];       // neighbours mostly share the entry: a broadcast
                const int dx = x + e - (int)(ent.x & 0xFFFFu);
                const int d2 = dx * dx + (int)(ent.y * ent.y);
                out[x + e] = resolution * sqrt((double)d2);      // -fmad=false: IEEE sqrt then IEEE multiply
            }
        }
        __syncthreads();
    }
}

// ---- the general form for maps beyond the 16-bit fast path (H + W + 1 > 32767): one thread per column, then one per row
__global__ void edt_columns_wide_kernel(const uint8_t* __restrict__ freemask, int H, int W, int* __restrict__ g, int inf,
                                        unsigned* __restrict__ any_obstacle) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= W) return;
    int d = inf;
    for (int r = 0; r < H; ++r) {
        d = freemask[(size_t)r * W + c] ? (d < inf ? d + 1 : inf) : 0;
        g[(size_t)r * W + c] = d;
    }
    if (d < inf) *any_obstacle = 1u;    // the column holds an obstacle
    d = inf;
    for (int r = H - 1; r >= 0; --r) {
        d = freemask[(size_t)r * W + c] ? (d < inf ? d + 1 : inf) : 0;
        const int up = g[(size_t)r * W + c];
        g[(size_t)r * W + c] = d < up ? d : up;
    }
}

__device__ __forceinline__ long long parab(long long x, long long i, long long gi) { return (x - i) * (x - i) + gi * gi; }

__global__ void edt_rows_wide_kernel(const int* __restrict__ g, int H, int W, int* __restrict__ s_all, int* __restrict__ t_all,
                                     double resolution, const unsigned* __restrict__ any_obstacle, double* __restrict__ dt) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= H) return;
    if (*any_obstacle == 0u) { edt_fill_row_without_obstacle(r, W, 0, 1, resolution, dt + (size_t)r * W); return; }
    const int* gr = g + (size_t)r * W;
    int* s = s_all + (size_t)r * W;
    int* t = t_all + (size_t)r * W;
    int q = 0;
    s[0] = 0; t[0] = 0;
    for (int u = 1; u < W; ++u) {
        const long long gu = gr[u];
        while (q >= 0 && parab(t[q], s[q], gr[s[q]]) > parab(t[q], u, gu)) --q;
        if (q < 0) { q = 0; s[0] = u; }
        else {
            const long long i = s[q], gi = gr[i];
            const long long w = 1 + ((long long)u * u - i * i + gu * gu - gi * gi) / (2 * ((long long)u - i));
            if (w < W) { ++q; s[q] = u; t[q] = (int)w; }
        }
    }
    for (int u = W - 1; u >= 0; --u) {
        const long long d2 = parab(u, s[q], gr[s[q]]);
        dt[(size_t)r * W + u] = resolution * sqrt((double)d2);
        if (u == t[q]) --q;
    }
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

void edt_scratch_free(EdtScratch* sc) {
    if (sc->base) cudaFree(sc->base);
    if (sc->ev0) cudaEventDestroy((cudaEvent_t)sc->ev0);
    if (sc->ev1) cudaEventDestroy((cudaEvent_t)sc->ev1);
    sc->base = nullptr; sc->bytes = 0; sc->ev0 = sc->ev1 = nullptr;
}

// freemask: DEVICE [H][W], non-zero = free space (pixel > 128 after the reference's bottom-up flip); dt: DEVICE fp64 [H][W].
// Synchronous on `stream`; sc->kernel_ms = the kernels alone (CUDA events).
int edt_device(const uint8_t* freemask, int H, int W, double resolution, double* dt, EdtScratch* sc, cudaStream_t stream) {
    const size_t cells = (size_t)H * W;
    // F110_EDT_WIDE=1 (tests, timing): force the general form on a map the 16-bit form would take
    const char* force_wide = getenv("F110_EDT_WIDE");
    const bool narrow = H + W + 1 <= 32767 && !(force_wide && force_wide[0] == '1');
    const int NB = (H + BAND - 1) / BAND, Hp = NB * BAND, Wp = (W + 7) / 8 * 8;
    size_t need;
    size_t off_words = 0, off_g = 0, off_stack = 0, off_marks = 0;
    if (narrow) {
        off_g = align_up((size_t)NB * W * sizeof(unsigned long long), 256);
        off_stack = off_g + align_up((size_t)W * Hp * sizeof(uint16_t), 256);
        off_marks = off_stack + align_up(cells * sizeof(uint2), 256);
        need = off_marks + align_up((size_t)H * Wp * sizeof(uint16_t), 256);
    } else {
        need = 3 * cells * sizeof(int);
    }
    const size_t off_any = align_up(need, 256);   // one word: does the mask hold any obstacle
    need = off_any + sizeof(unsigned);
    if (sc->bytes < need) {
        if (sc->base) cudaFree(sc->base);
        sc->base = nullptr; sc->bytes = 0;
        if (cudaMalloc(&sc->base, need) != cudaSuccess) { cudaGetLastError(); return -1; }
        sc->bytes = need;
    }
    if (!sc->ev0) {
        cudaEvent_t a, b;
        if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return -1;
        sc->ev0 = a; sc->ev1 = b;
    }
    char* base = static_cast<char*>(sc->base);
    unsigned* any_obstacle = reinterpret_cast<unsigned*>(base + off_any);
    cudaEventRecord((cudaEvent_t)sc->ev0, stream);
    cudaMemsetAsync(any_obstacle, 0, sizeof(unsigned), stream);
    if (narrow) {
        unsigned long long* words = reinterpret_cast<unsigned long long*>(base + off_words);
        uint16_t* gT = reinterpret_cast<uint16_t*>(base + off_g);
        uint2* stacks = reinterpret_cast<uint2*>(base + off_stack);
        uint16_t* marks = reinterpret_cast<uint16_t*>(base + off_marks);
        const unsigned inf = (unsigned)(H + W + 1);    // larger than any real distance
        cudaMemsetAsync(marks, 0, (size_t)H * Wp * sizeof(uint16_t), stream);
        edt_band_masks_kernel<<<dim3((W + 127) / 128, NB), 128, 0, stream>>>(freemask, H, W, words, any_obstacle);
        edt_columns_kernel<<<dim3((W + 127) / 128, NB), 128, 0, stream>>>(words, W, NB, Hp, inf, gT);
        edt_envelope_kernel<<<(H + 31) / 32, 32, 0, stream>>>(gT, H, W, Hp, Wp, stacks, marks);
        edt_fill_kernel<<<H, FILL_THREADS, 0, stream>>>(stacks, marks, W, Wp, resolution, any_obstacle, dt);
    } else {
        int* g = reinterpret_cast<int*>(base);
        int* s = g + cells;
        int* t = s + cells;
        edt_columns_wide_kernel<<<(W + 127) / 128, 128, 0, stream>>>(freemask, H, W, g, H + W + 1, any_obstacle);
        edt_rows_wide_kernel<<<(H + 63) / 64, 64, 0, stream>>>(g, H, W, s, t, resolution, any_obstacle, dt);
    }
    cudaEventRecord((cudaEvent_t)sc->ev1, stream);
    const cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return -1;
    cudaEventElapsedTime(&sc->kernel_ms, (cudaEvent_t)sc->ev0, (cudaEvent_t)sc->ev1);
    return 0;
}
