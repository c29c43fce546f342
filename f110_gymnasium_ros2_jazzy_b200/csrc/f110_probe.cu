// f110_probe.cu -- the empirical gather roofline bench.py quotes next to the lidar kernel (SURVEY 8d):
// every thread performs `chain` DEPENDENT 8-byte loads at pseudo-random cells of the handle's distance-transform
// map (the next address depends on the value just loaded), with the lidar kernel's launch shape and no other work.
// It answers "how fast can this chip chase `chain` fp64 cells per thread through a map of this size".
// Also f110_trig_probe: the dynamics kernel's sin / cos / tan, and f110_hypot_probe: the shaped reward's hypot, for the tests
// that hold those kernels to a model bit for bit.
#include <cuda_runtime.h>
#include <stdint.h>

#include "f110_b200.h"

int f110_set_error(int code, const char* msg);   // f110_capi.cu

namespace {
__global__ void __launch_bounds__(128) gather_probe_kernel(const double* __restrict__ map, unsigned mask, unsigned offset,
                                                           int chain, unsigned total, double* __restrict__ sink) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    unsigned idx = (t * 2654435761u) & mask;
    double acc = 0.0;
    for (int k = 0; k < chain; ++k) {
        const double v = __ldg(map + offset + idx);
        acc += v;
        idx = (idx * 1664525u + 1013904223u + (unsigned)__double_as_longlong(v)) & mask;
    }
    if (acc == -1.0) sink[0] = acc;   // never true: keeps the chain alive
}

// The trig calls of the dynamics kernel, compiled with the library's flags: sincos as for the heading terms, tan and cos as
// for the steering angle of the kinematic branch.
__global__ void __launch_bounds__(128) trig_probe_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    double s, c;
    sincos(v, &s, &c);
    out[i] = s;
    out[n + i] = c;
    out[2 * n + i] = tan(v);
    out[3 * n + i] = cos(v);
}

// The reward kernels' one inexact call besides sincos: hypot(ex - ox, ey - oy) of the opponent bubble.
__global__ void __launch_bounds__(128) hypot_probe_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t n,
                                                          double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = hypot(a[i], b[i]);
}
}  // namespace

extern "C" int f110_hypot_probe(const double* a_dev, const double* b_dev, int64_t n, double* out_dev, void* stream) {
    if (!a_dev || !b_dev || !out_dev || n < 0) return f110_set_error(F110_ERR_INVALID, "f110_hypot_probe: need non-null buffers and n >= 0");
    if (n == 0) return F110_OK;
    hypot_probe_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a_dev, b_dev, n, out_dev);
    return cudaGetLastError() == cudaSuccess ? F110_OK : f110_set_error(F110_ERR_CUDA, "f110_hypot_probe: kernel launch failed");
}

extern "C" int f110_trig_probe(const double* x_dev, int64_t n, double* out_dev, void* stream) {
    if (!x_dev || !out_dev || n < 0) return f110_set_error(F110_ERR_INVALID, "f110_trig_probe: need non-null buffers and n >= 0");
    if (n == 0) return F110_OK;
    trig_probe_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(x_dev, n, out_dev);
    return cudaGetLastError() == cudaSuccess ? F110_OK : f110_set_error(F110_ERR_CUDA, "f110_trig_probe: kernel launch failed");
}

extern "C" int f110_gather_probe(const double* map_dev, int64_t num_cells, int64_t window_cells, int32_t chain,
                                 int64_t num_threads, int32_t repeats, double* sink_dev, float* ms_out, void* stream) {
    if (!map_dev || !sink_dev || !ms_out || num_cells < 2 || chain < 1 || num_threads < 1 || repeats < 1) return F110_ERR_INVALID;
    int64_t w = window_cells > 0 && window_cells < num_cells ? window_cells : num_cells;
    unsigned mask = 1;
    while ((int64_t)(mask << 1) <= w) mask <<= 1;
    mask -= 1;
    const unsigned offset = (unsigned)((num_cells - (int64_t)mask - 1) / 2);
    cudaStream_t s = (cudaStream_t)stream;
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return F110_ERR_CUDA;
    const unsigned total = (unsigned)num_threads;
    const unsigned blocks = (total + 127) / 128;
    gather_probe_kernel<<<blocks, 128, 0, s>>>(map_dev, mask, offset, chain, total, sink_dev);   // warm-up
    cudaEventRecord(e0, s);
    for (int r = 0; r < repeats; ++r) gather_probe_kernel<<<blocks, 128, 0, s>>>(map_dev, mask, offset, chain, total, sink_dev);
    cudaEventRecord(e1, s);
    if (cudaEventSynchronize(e1) != cudaSuccess) return F110_ERR_CUDA;
    cudaEventElapsedTime(ms_out, e0, e1);
    *ms_out /= (float)repeats;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return F110_OK;
}
