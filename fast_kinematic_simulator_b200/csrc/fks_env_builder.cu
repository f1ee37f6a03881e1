// Device-side environment builder (SURVEY.md 8(f)-1): cuboid obstacles -> occupancy -> signed distance field ->
// surface-normal table, produced directly in the formats the simulate kernels read (fks_device_types.h DevEnv),
// without a host round trip.  Same results, bit for bit, as simulator_environment_builder::BuildCompleteEnvironment
// restated in host/environment_builder.cpp (the tests check both against the CPU restatement under oracle/):
//   BuildEnvironment + DiscretizeObstacle   simulator_environment_builder.cpp:21-46,49-160   -> rasterize_kernel
//   ExtractSignedDistanceField(+inf,{},true,false)   envb.cpp:473 (sdf_tools)                  -> edt_z_kernel, edt_line_kernel
//   BuildSurfaceNormalsGrid                 envb.cpp:258-468 (UpdateSurfaceNormalGridCell :162-187)
//                                                                 -> normals_mark / count / scan / emit kernels
// This file is compiled with --fmad=false: every product and sum is rounded separately, as on the host.
//
// Data flow in HBM (n = nx*ny*nz cells):
//   occupancy  u8[n]      written by the rasteriser (2 samples per cell and axis, envb.cpp:23), read once by the z pass
//   field      i32[n]     ONE signed buffer for both distance transforms: a free cell holds +d2(nearest filled), a filled
//                         cell holds -d2(nearest free) (squared, in cells).  Each cell needs only the transform of the
//                         opposite kind, and a cell of the opposite kind is a zero seed for it at every stage, so
//                         max(+-v, 0) recovers either partial transform.  z pass: bit scans on ballot words; y and x passes:
//                         shared-memory tiles [line position][32 consecutive cells across], windowed exact minimisation
//                         (the search radius is bounded by the current best).  The x pass writes the float SDF in place.
//   winner     u64[n]     surface pass: atomicMax of (global sample index + 1) = the LAST sample that rewrites the cell in
//                         the reference's obstacle/x/y/z loop order (ClearStoredSurfaceNormals then Insert, envb.cpp:171-181)
//   count      u8[n]      entries per cell (0..3) -> two-level exclusive scan -> cells emitted in ascending cell order

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <vector>

#include "fks_device_types.h"
#include "fks_internal.h"

using namespace fksdev;

namespace fks_host {
void finish_env_l2_window(fks_env* env);  // fks_api.cu
}

namespace {

constexpr int kInf = 1 << 29;  // "no seed": same sentinel as the host builder
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;  // cells per thread of the count / emit kernels

struct DevObstacle {
    double pose[12];
    double ext[3];
    int xc, yc, zc, _pad;
    unsigned long long sample_start;  // index of the obstacle's first discretisation sample in the global order
};

struct DevGrid {
    double inv_origin[12];
    double res, inv_res, eff;
    int nx, ny, nz, n_obstacles;
    long long ncells;
    unsigned long long total_samples;
};

__device__ __forceinline__ void iso_apply(const double* T, const double* p, double* out) {
    for (int r = 0; r < 3; r++) out[r] = T[4 * r + 0] * p[0] + T[4 * r + 1] * p[1] + T[4 * r + 2] * p[2] + T[4 * r + 3];
}
__device__ __forceinline__ void iso_rotate(const double* T, const double* v, double* out) {
    for (int r = 0; r < 3; r++) out[r] = T[4 * r + 0] * v[0] + T[4 * r + 1] * v[1] + T[4 * r + 2] * v[2];
}

// VoxelGrid::LocationToGridIndex (arc_utilities): grid-frame point * (1 / cell size), C-cast truncation
__device__ __forceinline__ bool location_to_cell(const DevGrid& g, const double* w, long long* cell) {
    double q[3];
    iso_apply(g.inv_origin, w, q);
    const long long ix = (long long)(q[0] * g.inv_res), iy = (long long)(q[1] * g.inv_res), iz = (long long)(q[2] * g.inv_res);
    if (ix < 0 || iy < 0 || iz < 0 || ix >= g.nx || iy >= g.ny || iz >= g.nz) return false;
    *cell = (ix * g.ny + iy) * g.nz + iz;
    return true;
}

// global sample index -> obstacle and (xi, yi, zi) of the nested loops of DiscretizeObstacle (envb.cpp:32-44)
__device__ __forceinline__ int decode_sample(const DevObstacle* __restrict__ obs, int n_obs, unsigned long long s, int* xi, int* yi,
                                             int* zi) {
    int lo = 0, hi = n_obs - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (obs[mid].sample_start <= s) lo = mid;
        else hi = mid - 1;
    }
    const unsigned long long local = s - obs[lo].sample_start;
    const unsigned zc = (unsigned)obs[lo].zc, yc = (unsigned)obs[lo].yc;
    if (local < 0xffffffffull) {
        const unsigned l32 = (unsigned)local, t = l32 / zc;
        *zi = (int)(l32 - t * zc);
        *xi = (int)(t / yc);
        *yi = (int)(t - (unsigned)(*xi) * yc);
    } else {
        const unsigned long long t = local / zc;
        *zi = (int)(local - t * zc);
        *xi = (int)(t / yc);
        *yi = (int)(t - (unsigned long long)(*xi) * yc);
    }
    return lo;
}

// ---- BuildEnvironment: one thread per discretisation sample (envb.cpp:32-44,85,150-155) ------------------------------
__global__ void __launch_bounds__(256) rasterize_kernel(const DevObstacle* __restrict__ obs, DevGrid g, unsigned char* __restrict__ occ) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < g.total_samples; s += stride) {
        int xi, yi, zi;
        const DevObstacle& ob = obs[decode_sample(obs, g.n_obstacles, s, &xi, &yi, &zi)];
        const double loc[3] = {-(ob.ext[0] - (g.res * 0.5)) + (g.eff * xi), -(ob.ext[1] - (g.res * 0.5)) + (g.eff * yi),
                               -(ob.ext[2] - (g.res * 0.5)) + (g.eff * zi)};
        double w[3];
        iso_apply(ob.pose, loc, w);
        long long cell;
        if (location_to_cell(g, w, &cell)) occ[cell] = 1;  // SetValue out of bounds is a no-op
    }
}

// ---- distance transform, z pass: lines are contiguous, seeds are binary -> nearest set bit on ballot words -------------
__device__ __forceinline__ int nearest_set_bit(const unsigned* __restrict__ words, int nw, int k) {
    const int wi = k >> 5, b = k & 31;
    int best = kInf;
    unsigned m = words[wi] & ((1u << b) - 1u);
    for (int j = wi;;) {
        if (m) {
            best = k - (j * 32 + 31 - __clz(m));
            break;
        }
        if (--j < 0) break;
        m = words[j];
    }
    m = (b == 31) ? 0u : (words[wi] & ~((2u << b) - 1u));
    for (int j = wi;;) {
        if (m) {
            best = min(best, (j * 32 + __ffs(m) - 1) - k);
            break;
        }
        if (++j >= nw) break;
        m = words[j];
    }
    return best;
}

constexpr int kZWarps = 8;
constexpr int kZMaxWords = 128;  // lines of up to 4096 cells

__global__ void __launch_bounds__(kZWarps * 32) edt_z_kernel(const unsigned char* __restrict__ occ, int* __restrict__ field, long long n_lines, int nz) {
    __shared__ unsigned s_filled[kZWarps][kZMaxWords];
    __shared__ unsigned s_free[kZWarps][kZMaxWords];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nw = (nz + 31) >> 5;
    for (long long line = (long long)blockIdx.x * kZWarps + warp; line < n_lines; line += (long long)gridDim.x * kZWarps) {
        const unsigned char* row = occ + line * nz;
        for (int c = 0; c < nw; c++) {
            const int k = c * 32 + lane;
            const bool in = k < nz;
            const unsigned f = __ballot_sync(0xffffffffu, in && row[k] != 0);
            const unsigned valid = __ballot_sync(0xffffffffu, in);
            if (lane == 0) {
                s_filled[warp][c] = f;
                s_free[warp][c] = ~f & valid;
            }
        }
        __syncwarp();
        for (int c = 0; c < nw; c++) {
            const int k = c * 32 + lane;
            if (k < nz) {
                const bool filled = (s_filled[warp][c] >> lane) & 1u;
                const int d = nearest_set_bit(filled ? s_free[warp] : s_filled[warp], nw, k);
                const int d2 = d >= kInf ? kInf : d * d;  // d <= 4095
                field[line * nz + k] = filled ? -d2 : d2;
            }
        }
        __syncwarp();
    }
}

// ---- distance transform, strided passes --------------------------------------------------------------------------------
// element(outer, pos, a) = field[outer * outer_stride + pos * line_stride + a], a < across.  One CTA stages the lines of W
// consecutive `a` (coalesced) for every position into shared memory, then each thread minimises h(p) + (q - p)^2 over p for
// its cells, h = max(sign * v, 0), searching outwards only while r^2 can still beat the current best (exact).
template <bool FINAL>
__global__ void __launch_bounds__(256) edt_line_kernel(int* __restrict__ field, int n, long long line_stride, long long across,
                                                        long long outer_stride, int W, double res) {
    extern __shared__ int tile[];
    const int tx = threadIdx.x % W, ty = threadIdx.x / W, TY = blockDim.x / W;
    const long long a = (long long)blockIdx.x * W + tx;
    const bool live = a < across;
    int* base = field + (long long)blockIdx.y * outer_stride + a;
    for (int pos = ty; pos < n; pos += TY) tile[pos * W + tx] = live ? base[pos * line_stride] : kInf;
    __syncthreads();
    if (!live) return;
    for (int q = ty; q < n; q += TY) {
        const int own = tile[q * W + tx];
        const int sign = own > 0 ? 1 : -1;
        int best = own * sign;
        // outwards from q while r^2 can still beat the best; past the ends of the line the index is clamped: the end cell is then
        // re-read with a larger r^2 than when it was met at its true distance, which cannot lower the minimum
        const int rmax = max(q, n - 1 - q);
        const int* col = tile + tx;
        for (int r = 1, rr = 1; r <= rmax && rr < best; rr += 2 * r + 1, r++) {
            const int lo = max(q - r, 0), hi = min(q + r, n - 1);
            const int cand = min(max(sign * col[lo * W], 0), max(sign * col[hi * W], 0)) + rr;
            best = min(best, cand);
        }
        best = min(best, kInf);
        if (FINAL) {
            // sdf = (float)(sqrt(d2_filled) * res - sqrt(d2_free) * res); one of the two is exactly zero
            const double d = sqrt((double)best) * res;
            const float f = sign > 0 ? (float)(d - 0.0) : (float)(0.0 - d);
            base[q * line_stride] = __float_as_int(f);
        } else {
            base[q * line_stride] = sign * best;
        }
    }
}

// ---- surface normals, pass 2 bookkeeping: which sample writes each cell last (envb.cpp:280-463, :162-187) ----------------
__global__ void __launch_bounds__(256) normals_mark_kernel(const DevObstacle* __restrict__ obs, DevGrid g, const float* __restrict__ sdf,
                                                            unsigned long long* __restrict__ winner) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < g.total_samples; s += stride) {
        int xi, yi, zi;
        const DevObstacle& ob = obs[decode_sample(obs, g.n_obstacles, s, &xi, &yi, &zi)];
        if (!(xi == 0 || yi == 0 || zi == 0 || xi == ob.xc - 1 || yi == ob.yc - 1 || zi == ob.zc - 1)) continue;
        const double loc[3] = {-(ob.ext[0] - g.eff) + (g.eff * xi), -(ob.ext[1] - g.eff) + (g.eff * yi), -(ob.ext[2] - g.eff) + (g.eff * zi)};
        double w[3];
        iso_apply(ob.pose, loc, w);
        long long cell;
        if (!location_to_cell(g, w, &cell)) continue;  // distance = +inf passes the test, but Clear/Insert out of bounds do nothing
        if ((double)sdf[cell] > -(g.res * 1.5)) atomicMax(&winner[cell], s + 1ull);
    }
}

// raw normals of a surface sample: the 26-way chain of envb.cpp:302-461 tests index == 0 before index == count - 1 on each
// axis and lists the axes in x, y, z order
__device__ __forceinline__ int surface_signs(const DevObstacle& ob, int xi, int yi, int zi, int* sx, int* sy, int* sz) {
    *sx = xi == 0 ? -1 : (xi == ob.xc - 1 ? 1 : 0);
    *sy = yi == 0 ? -1 : (yi == ob.yc - 1 ? 1 : 0);
    *sz = zi == 0 ? -1 : (zi == ob.zc - 1 ? 1 : 0);
    return (*sx != 0) + (*sy != 0) + (*sz != 0);
}

__global__ void __launch_bounds__(kScanThreads) normals_count_kernel(const DevObstacle* __restrict__ obs, DevGrid g, const float* __restrict__ sdf,
                                                                     const unsigned long long* __restrict__ winner,
                                                                     unsigned char* __restrict__ count,
                                                                     unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned long long s_warp[kScanThreads / 32];
    const long long base = (long long)blockIdx.x * (kScanThreads * kScanItems);
    unsigned long long local = 0;
    for (int i = 0; i < kScanItems; i++) {
        const long long cell = base + (long long)i * kScanThreads + threadIdx.x;
        if (cell >= g.ncells) break;
        int c = 0;
        const unsigned long long key = winner[cell];
        if (key) {
            int xi, yi, zi, sx, sy, sz;
            const DevObstacle& ob = obs[decode_sample(obs, g.n_obstacles, key - 1ull, &xi, &yi, &zi)];
            c = surface_signs(ob, xi, yi, zi, &sx, &sy, &sz);
        } else if (sdf[cell] < 0.0f) {  // envb.cpp:269-274
            c = 1;
        }
        count[cell] = (unsigned char)c;
        if (c) local += (1ull << 32) | (unsigned long long)c;  // {cells, entries}
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kScanThreads / 32; w++) t += s_warp[w];
        block_sums[blockIdx.x] = t;
    }
}

// exclusive scan of the per-block {cells, entries} sums (one CTA; a few thousand to a few hundred thousand values)
__global__ void __launch_bounds__(1024) scan_block_sums_kernel(unsigned long long* __restrict__ sums, long long n, unsigned long long* __restrict__ total) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (long long b = 0; b < n; b += 1024) {
        const long long i = b + threadIdx.x;
        const unsigned long long v = i < n ? sums[i] : 0ull;
        unsigned long long incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long off = s_carry, all = 0;
        for (int w = 0; w < 32; w++) {
            if (w < warp) off += s_warp[w];
            all += s_warp[w];
        }
        if (i < n) sums[i] = off + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += all;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

// EigenHelpers::SafeNormal (spcs.hpp:59,62)
__device__ __forceinline__ void safe_normal3(const double* v, double* out) {
    double s = 0.0;
    for (int i = 0; i < 3; i++) s += v[i] * v[i];
    const double nrm = sqrt(s);
    if (nrm > 2.220446049250313e-16) {
        for (int i = 0; i < 3; i++) out[i] = v[i] / nrm;
    } else {
        for (int i = 0; i < 3; i++) out[i] = v[i];
    }
}

// sdf_tools SignedDistanceField::GetGradient(x, y, z, enable_edge_gradients = true) (call site envb.cpp:272)
__device__ __forceinline__ void sdf_gradient(const float* __restrict__ sdf, const DevGrid& g, long long cell, double* out) {
    const long long sy = g.nz, sx = (long long)g.ny * g.nz;
    const int z = (int)(cell % g.nz), y = (int)((cell / g.nz) % g.ny), x = (int)(cell / sx);
    if (x > 0 && y > 0 && z > 0 && x < g.nx - 1 && y < g.ny - 1 && z < g.nz - 1) {
        const double inv_twice_res = 1.0 / (2.0 * g.res);
        out[0] = (double)(sdf[cell + sx] - sdf[cell - sx]) * inv_twice_res;
        out[1] = (double)(sdf[cell + sy] - sdf[cell - sy]) * inv_twice_res;
        out[2] = (double)(sdf[cell + 1] - sdf[cell - 1]) * inv_twice_res;
        return;
    }
    const int lx = max(0, x - 1), hx = min(g.nx - 1, x + 1), ly = max(0, y - 1), hy = min(g.ny - 1, y + 1), lz = max(0, z - 1),
              hz = min(g.nz - 1, z + 1);
    const double ix = (double)(hx - lx) * g.res, iy = (double)(hy - ly) * g.res, iz = (double)(hz - lz) * g.res;
    out[0] = out[1] = out[2] = 0.0;
    if (ix > 0.0) out[0] = ((double)sdf[cell + (hx - x) * sx] - (double)sdf[cell + (lx - x) * sx]) * (1.0 / ix);
    if (iy > 0.0) out[1] = ((double)sdf[cell + (hy - y) * sy] - (double)sdf[cell + (ly - y) * sy]) * (1.0 / iy);
    if (iz > 0.0) out[2] = ((double)sdf[cell + (hz - z)] - (double)sdf[cell + (lz - z)]) * (1.0 / iz);
}

// cells in ascending order: CSR arrays, 6-double entries and the open-addressing hash the simulate kernels probe
__global__ void __launch_bounds__(kScanThreads) normals_emit_kernel(const DevObstacle* __restrict__ obs, DevGrid g, const float* __restrict__ sdf,
                                                                    const unsigned long long* __restrict__ winner,
                                                                    const unsigned char* __restrict__ count,
                                                                    const unsigned long long* __restrict__ block_offsets,
                                                                    long long* __restrict__ cell_index, unsigned* __restrict__ cell_start,
                                                                    double* __restrict__ entries, unsigned long long* __restrict__ keys,
                                                                    unsigned long long mask) {
    __shared__ unsigned long long s_warp[kScanThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long base = (long long)blockIdx.x * (kScanThreads * kScanItems);
    unsigned long long running = block_offsets[blockIdx.x];
    for (int i = 0; i < kScanItems; i++) {
        if (base + (long long)i * kScanThreads >= g.ncells) break;  // uniform
        const long long cell = base + (long long)i * kScanThreads + threadIdx.x;
        const int c = cell < g.ncells ? (int)count[cell] : 0;
        const unsigned long long v = c ? ((1ull << 32) | (unsigned long long)c) : 0ull;
        unsigned long long incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long off = running, all = 0;
        for (int w = 0; w < kScanThreads / 32; w++) {
            if (w < warp) off += s_warp[w];
            all += s_warp[w];
        }
        __syncthreads();
        running += all;
        if (!c) continue;
        const unsigned long long excl = off + incl - v;
        const long long rank = (long long)(excl >> 32);
        const unsigned first = (unsigned)(excl & 0xffffffffull);
        cell_index[rank] = cell;
        cell_start[rank] = first;
        double* e = entries + 6ull * first;
        const unsigned long long key = winner[cell];
        if (key) {
            int xi, yi, zi, s[3];
            const DevObstacle& ob = obs[decode_sample(obs, g.n_obstacles, key - 1ull, &xi, &yi, &zi)];
            surface_signs(ob, xi, yi, zi, &s[0], &s[1], &s[2]);
            for (int axis = 0; axis < 3; axis++) {
                if (!s[axis]) continue;
                double nrm[3] = {0.0, 0.0, 0.0};
                nrm[axis] = (double)s[axis];
                const double raw_e[3] = {-nrm[0], -nrm[1], -nrm[2]};
                double rn[3], re[3];
                iso_rotate(ob.pose, nrm, rn);
                iso_rotate(ob.pose, raw_e, re);
                safe_normal3(re, e);      // entry direction (4-vector with w = 0: same norm)
                safe_normal3(rn, e + 3);  // normal
                e += 6;
            }
        } else {
            double grad[3];
            sdf_gradient(sdf, g, cell, grad);
            e[0] = e[1] = e[2] = 0.0;  // SafeNormal of the zero entry direction
            safe_normal3(grad, e + 3);
        }
        // hash slot {cell + 1, first | count << 32}
        unsigned long long h = normal_hash((unsigned long long)cell) & mask;
        while (atomicCAS(&keys[2 * h], 0ull, (unsigned long long)cell + 1ull) != 0ull) h = (h + 1) & mask;
        keys[2 * h + 1] = (unsigned long long)first | ((unsigned long long)c << 32);
    }
}

// the property link-level culling relies on (fks_env_create makes the same test on the host)
__global__ void __launch_bounds__(256) distance_field_check_kernel(const float* __restrict__ sdf, DevGrid g, double lim1, int* __restrict__ ok) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long sy = g.nz, sx = (long long)g.ny * g.nz;
    bool good = true;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < g.ncells; i += stride) {
        const int z = (int)(i % g.nz), y = (int)((i / g.nz) % g.ny), x = (int)(i / sx);
        const double v = (double)sdf[i];
        const long long nb[3] = {x + 1 < g.nx ? i + sx : i, y + 1 < g.ny ? i + sy : i, z + 1 < g.nz ? i + 1 : i};
        for (int k = 0; k < 3; k++) {
            const double w = (double)sdf[nb[k]];
            const double lim = ((v < 0.0) != (w < 0.0)) ? 2.0 * lim1 : lim1;
            if (!(fabs(v - w) <= lim)) good = false;
        }
    }
    if (!good) *ok = 0;
}

struct Temps {
    std::vector<void*> ptrs;
    std::vector<cudaEvent_t> events;
    int prev_device = -1;
    // temporaries come from the device's stream-ordered pool (no synchronising cudaMalloc / cudaFree inside the build;
    // up to 256 MiB stays cached in the pool between builds, see fks_env_build_device)
    ~Temps() {
        for (void* p : ptrs) cudaFreeAsync(p, 0);
        for (cudaEvent_t e : events) cudaEventDestroy(e);
        if (prev_device >= 0) cudaSetDevice(prev_device);
    }
    template <typename T>
    cudaError_t alloc(T** p, size_t n) {
        *p = nullptr;
        cudaError_t e = pooled_alloc((void**)p, std::max<size_t>(n, 1) * sizeof(T), 0);
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    // small blocks from the stream-ordered pool, large ones (which would make the pool grow and shrink by hundreds of MB
    // on every build) from cudaMalloc; cudaFree / cudaFreeAsync accept both kinds
    static cudaError_t pooled_alloc(void** p, size_t bytes, cudaStream_t st) {
        return bytes <= (64u << 20) ? cudaMallocAsync(p, bytes, st) : cudaMalloc(p, bytes);
    }
};

#define FKS_TRY(call)                                                                                  \
    do {                                                                                               \
        cudaError_t _e = (call);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            fks_env_destroy(env);                                                                      \
            return fail(FKS_ERR_CUDA, std::string("fks_env_build_device: " #call ": ") + cudaGetErrorString(_e)); \
        }                                                                                              \
    } while (0)

int pick_tile_width(int n) {
    int W = 32;
    while (W > 4 && (size_t)n * W * sizeof(int) > 200u * 1024u) W >>= 1;
    return W;
}

}  // namespace

extern "C" int fks_env_build_device(int device, const fks_obstacle* obstacles, size_t n_obstacles, double resolution, fks_env** out) {
    if (!out || !(resolution > 0.0) || (n_obstacles > 0 && !obstacles)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_device: invalid argument");
    *out = nullptr;
    for (size_t i = 0; i < n_obstacles; i++)
        if (obstacles[i].object_id == 0)  // envb.hpp:35,41 assert(in_object_id > 0)
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_device: obstacle object_id must be > 0");
    if (n_obstacles > (1u << 24)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_device: too many obstacles");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "fks_env_build_device: no CUDA device");
    if (device < 0 || device >= ndev) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_device: bad device index");

    fks_host::GridGeometry gg;
    int rc = fks_host::compute_grid_geometry(obstacles, n_obstacles, resolution, &gg);
    if (rc != FKS_OK) return rc;
    const long long ncells = gg.nx * gg.ny * gg.nz;
    if (ncells > (1ll << 30)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_device: more than 2^30 cells");

    Temps tmp;
    if (cudaGetDevice(&tmp.prev_device) != cudaSuccess) tmp.prev_device = -1;
    if (cudaSetDevice(device) != cudaSuccess) return fail(FKS_ERR_CUDA, "fks_env_build_device: cudaSetDevice failed");

    // obstacle table with the sample counts of DiscretizeObstacle (envb.cpp:29-31)
    const double eff = resolution * 0.5;
    std::vector<DevObstacle> hobs(std::max<size_t>(n_obstacles, 1));
    unsigned long long total_samples = 0;
    for (size_t o = 0; o < n_obstacles; o++) {
        DevObstacle& d = hobs[o];
        std::memcpy(d.pose, obstacles[o].pose, sizeof(d.pose));
        std::memcpy(d.ext, obstacles[o].extents, sizeof(d.ext));
        d.xc = (int32_t)(obstacles[o].extents[0] * 2.0 * (1.0 / eff));
        d.yc = (int32_t)(obstacles[o].extents[1] * 2.0 * (1.0 / eff));
        d.zc = (int32_t)(obstacles[o].extents[2] * 2.0 * (1.0 / eff));
        d._pad = 0;
        d.sample_start = total_samples;
        if (d.xc > 0 && d.yc > 0 && d.zc > 0) total_samples += (unsigned long long)d.xc * (unsigned long long)d.yc * (unsigned long long)d.zc;
    }
    // obstacles without samples would break the search for the owner of a sample: drop them from the device table
    // (their sample ranges are empty, so the global sample order of the others is unchanged)
    std::vector<DevObstacle> live;
    for (size_t o = 0; o < n_obstacles; o++)
        if (hobs[o].xc > 0 && hobs[o].yc > 0 && hobs[o].zc > 0) live.push_back(hobs[o]);

    fks_env* env = new (std::nothrow) fks_env();
    if (!env) return fail(FKS_ERR_OUT_OF_MEMORY, "fks_env_build_device: out of host memory");
    std::memset(env, 0, sizeof(*env));
    env->device = device;
    env->sdf_bytes = (size_t)ncells * sizeof(float);

    DevGrid g;
    std::memcpy(g.inv_origin, gg.inv_origin, sizeof(g.inv_origin));
    g.res = resolution;
    g.inv_res = 1.0 / resolution;
    g.eff = eff;
    g.nx = (int)gg.nx;
    g.ny = (int)gg.ny;
    g.nz = (int)gg.nz;
    g.n_obstacles = (int)live.size();
    g.ncells = ncells;
    g.total_samples = total_samples;

    cudaDeviceProp prop;
    FKS_TRY(cudaGetDeviceProperties(&prop, device));
    const int sms = prop.multiProcessorCount;
    {
        cudaMemPool_t pool;
        unsigned long long keep = 256ull << 20;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        cudaGetLastError();
    }
    cudaStream_t st = 0;
    for (int i = 0; i < 10; i++) {  // 8 phase boundaries + the two ends of the table-allocation gap inside phase 6
        cudaEvent_t e;
        FKS_TRY(cudaEventCreate(&e));
        tmp.events.push_back(e);
    }
    int next_event = 0;
    auto mark = [&]() { return cudaEventRecord(tmp.events[next_event++], st); };

    DevObstacle* d_obs = nullptr;
    FKS_TRY(tmp.alloc(&d_obs, live.size()));
    if (!live.empty()) FKS_TRY(cudaMemcpyAsync(d_obs, live.data(), live.size() * sizeof(DevObstacle), cudaMemcpyHostToDevice, st));
    int* d_field = nullptr;  // becomes the SDF
    FKS_TRY(cudaMalloc((void**)&d_field, (size_t)ncells * sizeof(int)));
    env->d_sdf = reinterpret_cast<float*>(d_field);
    FKS_TRY(cudaMalloc((void**)&env->d_occupancy, (size_t)ncells));

    FKS_TRY(mark());  // 0
    // ---- BuildEnvironment -----------------------------------------------------------------------------------------
    FKS_TRY(cudaMemsetAsync(env->d_occupancy, 0, (size_t)ncells, st));
    const int sample_blocks = (int)std::min<unsigned long long>((total_samples + 255) / 256, (unsigned long long)sms * 32);
    if (total_samples) rasterize_kernel<<<sample_blocks, 256, 0, st>>>(d_obs, g, env->d_occupancy);
    FKS_TRY(cudaGetLastError());
    FKS_TRY(mark());  // 1
    // ---- ExtractSignedDistanceField ---------------------------------------------------------------------------------
    {
        const long long n_lines = gg.nx * gg.ny;
        const int blocks = (int)std::min<long long>((n_lines + kZWarps - 1) / kZWarps, (long long)sms * 16);
        edt_z_kernel<<<blocks, kZWarps * 32, 0, st>>>(env->d_occupancy, d_field, n_lines, g.nz);
        FKS_TRY(cudaGetLastError());
    }
    FKS_TRY(mark());  // 2
    {
        // y pass: lines of ny with stride nz inside one x slab; across = z
        const int W = pick_tile_width(g.ny);
        const size_t smem = (size_t)g.ny * W * sizeof(int);
        FKS_TRY(cudaFuncSetAttribute(edt_line_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid((unsigned)((g.nz + W - 1) / W), (unsigned)g.nx);
        edt_line_kernel<false><<<grid, 256, smem, st>>>(d_field, g.ny, (long long)g.nz, (long long)g.nz, (long long)g.ny * g.nz, W, resolution);
        FKS_TRY(cudaGetLastError());
    }
    FKS_TRY(mark());  // 3
    {
        // x pass: lines of nx with stride ny*nz; across = the flattened (y, z) index; writes the float SDF in place
        const int W = pick_tile_width(g.nx);
        const size_t smem = (size_t)g.nx * W * sizeof(int);
        FKS_TRY(cudaFuncSetAttribute(edt_line_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const long long across = (long long)g.ny * g.nz;
        dim3 grid((unsigned)((across + W - 1) / W), 1u);
        edt_line_kernel<true><<<grid, 256, smem, st>>>(d_field, g.nx, across, across, 0ll, W, resolution);
        FKS_TRY(cudaGetLastError());
    }
    FKS_TRY(mark());  // 4
    // ---- BuildSurfaceNormalsGrid --------------------------------------------------------------------------------------
    unsigned long long* d_winner = nullptr;
    unsigned char* d_count = nullptr;
    unsigned long long *d_block_sums = nullptr, *d_total = nullptr;
    const long long cells_per_block = (long long)kScanThreads * kScanItems;
    const long long n_blocks = (ncells + cells_per_block - 1) / cells_per_block;
    FKS_TRY(tmp.alloc(&d_winner, (size_t)ncells));
    FKS_TRY(tmp.alloc(&d_count, (size_t)ncells));
    FKS_TRY(tmp.alloc(&d_block_sums, (size_t)n_blocks));
    FKS_TRY(tmp.alloc(&d_total, 1));
    FKS_TRY(cudaMemsetAsync(d_winner, 0, (size_t)ncells * sizeof(unsigned long long), st));
    if (total_samples) normals_mark_kernel<<<sample_blocks, 256, 0, st>>>(d_obs, g, env->d_sdf, d_winner);
    FKS_TRY(cudaGetLastError());
    FKS_TRY(mark());  // 5
    normals_count_kernel<<<(unsigned)n_blocks, kScanThreads, 0, st>>>(d_obs, g, env->d_sdf, d_winner, d_count, d_block_sums);
    FKS_TRY(cudaGetLastError());
    scan_block_sums_kernel<<<1, 1024, 0, st>>>(d_block_sums, n_blocks, d_total);
    FKS_TRY(cudaGetLastError());
    unsigned long long total = 0;
    FKS_TRY(cudaMemcpyAsync(&total, d_total, sizeof(total), cudaMemcpyDeviceToHost, st));
    FKS_TRY(cudaEventRecord(tmp.events[8], st));  // the stream idles from here until the table arrays are allocated
    FKS_TRY(cudaStreamSynchronize(st));
    const size_t n_normal_cells = (size_t)(total >> 32), n_entries = (size_t)(total & 0xffffffffull);
    // the table arrays also come from the stream-ordered pool (fks_env_destroy releases them with cudaFree, which accepts both)
    size_t cap = 2;
    while (cap < 2 * n_normal_cells) cap <<= 1;
    FKS_TRY(Temps::pooled_alloc((void**)&env->d_keys, 2 * cap * sizeof(unsigned long long), st));
    FKS_TRY(Temps::pooled_alloc((void**)&env->d_entries, std::max<size_t>(n_entries, 1) * 6 * sizeof(double), st));
    FKS_TRY(Temps::pooled_alloc((void**)&env->d_cell_index, std::max<size_t>(n_normal_cells, 1) * sizeof(long long), st));
    FKS_TRY(Temps::pooled_alloc((void**)&env->d_cell_start, (n_normal_cells + 1) * sizeof(unsigned), st));
    FKS_TRY(cudaEventRecord(tmp.events[9], st));
    FKS_TRY(cudaMemsetAsync(env->d_keys, 0, 2 * cap * sizeof(unsigned long long), st));
    FKS_TRY(cudaMemsetAsync(env->d_entries, 0, std::max<size_t>(n_entries, 1) * 6 * sizeof(double), st));
    normals_emit_kernel<<<(unsigned)n_blocks, kScanThreads, 0, st>>>(d_obs, g, env->d_sdf, d_winner, d_count, d_block_sums, env->d_cell_index,
                                                                     env->d_cell_start, env->d_entries, env->d_keys, (unsigned long long)(cap - 1));
    FKS_TRY(cudaGetLastError());
    const unsigned last_start = (unsigned)n_entries;
    FKS_TRY(cudaMemcpyAsync(env->d_cell_start + n_normal_cells, &last_start, sizeof(unsigned), cudaMemcpyHostToDevice, st));
    env->n_normal_cells = (long long)n_normal_cells;
    env->n_entries = n_entries;
    FKS_TRY(mark());  // 6
    // ---- culling precondition -------------------------------------------------------------------------------------------
    int* d_ok = nullptr;
    FKS_TRY(tmp.alloc(&d_ok, 1));
    const int one = 1;
    FKS_TRY(cudaMemcpyAsync(d_ok, &one, sizeof(int), cudaMemcpyHostToDevice, st));
    distance_field_check_kernel<<<sms * 8, 256, 0, st>>>(env->d_sdf, g, resolution * (1.0 + 1e-4), d_ok);
    FKS_TRY(cudaGetLastError());
    int ok = 0;
    FKS_TRY(cudaMemcpyAsync(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, st));
    FKS_TRY(mark());  // 7
    FKS_TRY(cudaStreamSynchronize(st));

    for (int i = 1; i < 8; i++) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, tmp.events[i - 1], tmp.events[i]);
        env->build_ms[i] = ms;
    }
    {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, tmp.events[0], tmp.events[7]);
        env->build_ms[0] = ms;
        // phase 6 without the host-side allocation of the table arrays (size known only after the scan; cudaMalloc of
        // hundreds of MB takes 5-20 ms and is not device work): reported separately as [8]
        cudaEventElapsedTime(&ms, tmp.events[8], tmp.events[9]);
        env->build_ms[8] = ms;
        env->build_ms[6] -= ms;
    }

    DevEnv& d = env->dev;
    std::memcpy(d.origin, gg.origin, sizeof(d.origin));
    std::memcpy(d.inv_origin, gg.inv_origin, sizeof(d.inv_origin));
    d.map_res = resolution;
    d.sdf_res = resolution;
    d.inv_sdf_res = 1.0 / resolution;
    d.inv_twice_res = 1.0 / (2.0 * resolution);
    d.nx = g.nx;
    d.ny = g.ny;
    d.nz = g.nz;
    d.oob = std::numeric_limits<float>::infinity();
    d.cull = ok ? 1 : 0;
    d.sdf = env->d_sdf;
    d.nh_keys = env->d_keys;
    d.nh_mask = (unsigned long long)(cap - 1);
    d.normal_entries = env->d_entries;
    fks_host::finish_env_l2_window(env);
    *out = env;
    return FKS_OK;
}

extern "C" int fks_env_build_timings(const fks_env* env, double* out_ms, int n) {
    if (!env || !out_ms || n < 0) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_build_timings: invalid argument");
    for (int i = 0; i < n; i++) out_ms[i] = i < 9 ? env->build_ms[i] : 0.0;
    return FKS_OK;
}

// Device environment -> host arrays in the fks_env_desc layout (parity tests, and callers that want the SDF back).
extern "C" int fks_env_download(const fks_env* env, fks_built_env** out) {
    if (!env || !out) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_download: null argument");
    *out = nullptr;
    Temps tmp;
    if (cudaGetDevice(&tmp.prev_device) != cudaSuccess) tmp.prev_device = -1;
    if (cudaSetDevice(env->device) != cudaSuccess) return fail(FKS_ERR_CUDA, "fks_env_download: cudaSetDevice failed");
    fks_built_env* b = new (std::nothrow) fks_built_env();
    if (!b) return fail(FKS_ERR_OUT_OF_MEMORY, "fks_env_download: out of host memory");
    const DevEnv& d = env->dev;
    const size_t ncells = (size_t)d.nx * (size_t)d.ny * (size_t)d.nz;
    const size_t nc = (size_t)env->n_normal_cells, ne = env->n_entries;
    cudaError_t e = cudaSuccess;
    std::vector<double> e6(std::max<size_t>(ne, 1) * 6);
    b->sdf.resize(ncells);
    b->normal_cell_index.resize(nc);
    b->normal_cell_start.resize(nc + 1, 0);
    b->normal_entries.resize(ne * 7);
    e = cudaMemcpy(b->sdf.data(), env->d_sdf, ncells * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && env->d_occupancy) {
        b->occupancy.resize(ncells);
        e = cudaMemcpy(b->occupancy.data(), env->d_occupancy, ncells, cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess && nc) e = cudaMemcpy(b->normal_cell_index.data(), env->d_cell_index, nc * sizeof(long long), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(b->normal_cell_start.data(), env->d_cell_start, (nc + 1) * sizeof(unsigned), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && ne) e = cudaMemcpy(e6.data(), env->d_entries, ne * 6 * sizeof(double), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        delete b;
        return fail(FKS_ERR_CUDA, std::string("fks_env_download: ") + cudaGetErrorString(e));
    }
    for (size_t i = 0; i < ne; i++) {  // 6 doubles on the device, 7 in the descriptor (entry direction w is always 0)
        double* dst = &b->normal_entries[7 * i];
        const double* src = &e6[6 * i];
        dst[0] = src[0];
        dst[1] = src[1];
        dst[2] = src[2];
        dst[3] = 0.0;
        dst[4] = src[3];
        dst[5] = src[4];
        dst[6] = src[5];
    }
    fks_env_desc& o = b->desc;
    std::memset(&o, 0, sizeof(o));
    std::memcpy(o.origin, d.origin, sizeof(o.origin));
    std::memcpy(o.inverse_origin, d.inv_origin, sizeof(o.inverse_origin));
    o.map_resolution = d.map_res;
    o.sdf_resolution = d.sdf_res;
    o.nx = d.nx;
    o.ny = d.ny;
    o.nz = d.nz;
    o.sdf = b->sdf.data();
    o.oob_value = d.oob;
    o.n_normal_cells = (int64_t)nc;
    o.normal_cell_index = b->normal_cell_index.data();
    o.normal_cell_start = b->normal_cell_start.data();
    o.normal_entries = b->normal_entries.data();
    *out = b;
    return FKS_OK;
}
