// Calls that consume a batch's end states on the device (include/fksgpu.h, SURVEY.md 8f-3), host and device halves: split by
// contact, pairwise distances, clustering, groups and the next batch's starts, and the nearest configurations.  The planner
// (uncertainty_planning_core.cpp:97-99) splits the returned particles by did_contact and groups them by configuration
// distance; with these calls the end-state records stay in HBM between ForwardSimulateRobots and that step.  Records are
// cfg_stride doubles + fks_result_tail.
//
// Every distance is config_distance<KIND> (fks_robot_kind.cuh), the simulate kernel's own, with the pairwise kernel's
// operand order.  Selections use one total order on keys (distance, index), with NaN read as +inf, so their results are the
// same bits for any grid, split or stream.

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "fks_internal.h"
#include "fks_robot_kind.cuh"

namespace fksdev {

constexpr int kCfgMax = kMaxDof < 12 ? 12 : kMaxDof;  // doubles of a configuration
constexpr unsigned kNoIndex = 0xffffffffu;            // the index of a key that is no candidate: after every real one

// ---- the key order and its reductions --------------------------------------------------------------------------------------
__device__ __forceinline__ bool key_less(double d, unsigned i, double e, unsigned j) { return d < e || (d == e && i < j); }

// (d, i) of the warp's smallest key, in every lane
__device__ __forceinline__ void warp_argmin(double& d, unsigned& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(FKS_FULL, d, o);
        const unsigned oi = __shfl_xor_sync(FKS_FULL, i, o);
        if (key_less(od, oi, d, i)) {
            d = od;
            i = oi;
        }
    }
}

// the CTA's smallest (d, i) over its n_warps warps' lane-uniform keys, in every lane of warp 0, where it returns true; wd / wi:
// n_warps entries of shared memory
__device__ __forceinline__ bool block_argmin(double& d, unsigned& i, unsigned n_warps, double* wd, unsigned* wi) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        wd[warp] = d;
        wi[warp] = i;
    }
    __syncthreads();
    if (warp != 0) return false;
    d = lane < n_warps ? wd[lane] : INFINITY;
    i = lane < n_warps ? wi[lane] : kNoIndex;
    warp_argmin(d, i);
    return true;
}

// the distance of a key: config_distance with NaN read as +inf
template <int KIND>
__device__ __forceinline__ double key_distance(const DevRobot& rb, const double* cur, const double* target) {
    const double d = config_distance<KIND>(rb, cur, target);
    return isnan(d) ? INFINITY : d;
}

// occupancy x SM count: the CTAs of `kernel` that run at once
template <typename Kernel>
static unsigned resident_ctas(Kernel kernel, int block, size_t smem) {
    int per_sm = 0, dev = 0, sms = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem);
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (unsigned)((per_sm > 0 ? per_sm : 1) * (sms > 0 ? sms : 1));
}

// ---------------------------------------------------------------------------------------------
// fks_end_states_partition and fks_end_states_pairwise_distance
// ---------------------------------------------------------------------------------------------
constexpr int kPartitionBlock = 1024;

__device__ __forceinline__ bool record_in_contact(const char* results, size_t rec_stride, int cfg_stride, size_t i) {
    return (reinterpret_cast<const fks_result_tail*>(results + i * rec_stride + (size_t)cfg_stride * 8)->flags & FKS_FLAG_DID_CONTACT) != 0u;
}
// pass 1: particles in contact per block of 1024 records
__global__ void __launch_bounds__(kPartitionBlock) partition_count_kernel(const char* results, size_t rec_stride, int cfg_stride, size_t n,
                                                                          unsigned* block_counts) {
    const size_t i = (size_t)blockIdx.x * kPartitionBlock + threadIdx.x;
    const int c = __syncthreads_count(i < n && record_in_contact(results, rec_stride, cfg_stride, i));
    if (threadIdx.x == 0) block_counts[blockIdx.x] = (unsigned)c;
}
// pass 2 (one block): exclusive scan of the block counts in place; totals[0] = particles without contact, totals[1] = with
__global__ void __launch_bounds__(kPartitionBlock) partition_scan_kernel(unsigned* block_counts, unsigned n_blocks, size_t n,
                                                                         unsigned long long* totals) {
    __shared__ unsigned warp_sums[32];
    __shared__ unsigned carry;
    if (threadIdx.x == 0) carry = 0u;
    __syncthreads();
    for (unsigned base = 0; base < n_blocks; base += kPartitionBlock) {
        const unsigned i = base + threadIdx.x;
        const unsigned v = i < n_blocks ? block_counts[i] : 0u;
        unsigned incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(FKS_FULL, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            unsigned w = warp_sums[threadIdx.x];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(FKS_FULL, w, o);
                if (threadIdx.x >= o) w += t;
            }
            warp_sums[threadIdx.x] = w;  // inclusive over warps
        }
        __syncthreads();
        const unsigned before = carry + ((threadIdx.x >> 5) ? warp_sums[(threadIdx.x >> 5) - 1] : 0u) + (incl - v);
        if (i < n_blocks) block_counts[i] = before;
        __syncthreads();
        if (threadIdx.x == 0) carry += warp_sums[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        totals[1] = carry;
        totals[0] = (unsigned long long)n - carry;
    }
}
// pass 3: ids without contact first, ids in contact after them, ascending inside each part
__global__ void __launch_bounds__(kPartitionBlock) partition_scatter_kernel(const char* results, size_t rec_stride, int cfg_stride, size_t n,
                                                                            const unsigned* block_offsets, const unsigned long long* totals,
                                                                            unsigned* order) {
    __shared__ unsigned warp_counts[32];
    const size_t i = (size_t)blockIdx.x * kPartitionBlock + threadIdx.x;
    const bool valid = i < n, contact = valid && record_in_contact(results, rec_stride, cfg_stride, i);
    const unsigned ballot = __ballot_sync(FKS_FULL, contact);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) warp_counts[warp] = (unsigned)__popc(ballot);
    __syncthreads();
    unsigned before_in_block = (unsigned)__popc(ballot & ((1u << lane) - 1u));
    for (int w = 0; w < warp; w++) before_in_block += warp_counts[w];
    if (!valid) return;
    const size_t contact_before = (size_t)block_offsets[blockIdx.x] + before_in_block;  // ids in contact below i
    if (contact) order[(size_t)totals[0] + contact_before] = (unsigned)i;
    else order[i - contact_before] = (unsigned)i;
}

// out[a * m + b] = distance from the configuration of record subset[a] to that of record subset[b] (subset == nullptr: identity)
template <int KIND>
__global__ void __launch_bounds__(256) pairwise_distance_kernel(const DevRobot* robot, const char* results, size_t rec_stride, int cfg_stride,
                                                                const unsigned* subset, unsigned m, double* out) {
    __shared__ double from[kCfgMax];
    const unsigned a = blockIdx.y, b = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t ia = subset ? subset[a] : a;
    if ((int)threadIdx.x < cfg_stride) from[threadIdx.x] = reinterpret_cast<const double*>(results + ia * rec_stride)[threadIdx.x];
    __syncthreads();
    if (b >= m) return;
    const size_t ib = subset ? subset[b] : b;
    out[(size_t)a * m + b] = config_distance<KIND>(*robot, from, reinterpret_cast<const double*>(results + ib * rec_stride));
}

// ---------------------------------------------------------------------------------------------
// fks_end_states_cluster: flat agglomerative clustering (single / complete linkage, distance cutoff) of every segment of a
// position range, one CTA per segment.  A segment's distances form the upper triangle of an n x n matrix D (row pitch n):
// D[p][q], p < q, is the pairwise kernel's entry [p][q] for the same records, +inf where that is NaN or the contact flags
// differ under separate_contact.  Small segments keep D in shared memory, large ones in a global slot of the CTA.
//
// Merge loop.  A cluster is named by its smallest position (its representative); only representatives' rows and columns of D
// are finite, the others are +inf.  nn[i] / nnd[i] cache the smallest (D[i][j], j) over j > i, so the smallest
// (nnd[i], i, nn[i]) over i is the smallest merge key (L, min rep, max rep).  Merging a < b writes op(D[a][k], D[b][k]) into
// a's row and column (op = min for single, max for complete linkage: the Lance-Williams update of the two, exact), sets b's
// to +inf, and repairs the cache: row a is rescanned, so is every row whose neighbour was a or b (b is gone; under complete
// linkage a's distances grew), and a row i < a with another neighbour only compares its cache with the new D[i][a] -- under
// single linkage it can only have shrunk, under complete linkage it grew from a value that already lost.
//
// Segments of up to kClusterSmallMax positions keep their distance matrix in shared memory (160^2 doubles = 200 KiB of the
// 227 KiB a CTA can have), longer ones in a global slot of n_cap^2 doubles per CTA; the per-position state of a segment (20
// bytes each) stays in shared memory, which bounds a segment at kClusterMaxSegment.
//
// Workspace (fks_sim::d_clu, u64 words): [offsets (n_segments + 1) | totals (2) | counts (n_segments), then the small and
// the large segment lists, as u32]; fks_sim::d_clu_mat: the large segments' matrix slots.
// ---------------------------------------------------------------------------------------------
constexpr unsigned kClusterSmallMax = 160;
constexpr unsigned kClusterMaxSegment = 8192;
constexpr int kClusterSmallBlock = 256;
constexpr int kClusterLargeBlock = 1024;

struct ClusterArgs {
    const DevRobot* robot;
    const char* results;
    size_t rec_stride;
    int cfg_stride;
    int complete;
    int separate_contact;
    double threshold;
    const unsigned* order;                // position -> record id, or null (identity)
    const unsigned long long* offsets;    // [n_segments + 1]
    const unsigned* segs;                 // segment ids this launch clusters
    unsigned n_segs;
    unsigned n_cap;                       // largest segment of this launch
    double* work;                         // large path: one n_cap x n_cap slot per CTA
    unsigned* labels;                     // [m]: segment-local cluster ids (the relabel kernel adds the segment's base)
    unsigned* counts;                     // [n_segments]: clusters per segment
};

// per-segment state in shared memory behind the matrix (small path) or at the start of it (large path)
struct ClusterSmem {
    unsigned* rep;   // [n_cap] representative of each position
    unsigned* nn;    // [n_cap] cached nearest j > i (n = none), reused for the ranks of the representatives at the end
    double* nnd;     // [n_cap] D[i][nn[i]]
    unsigned* list;  // [n_cap] rows to rescan
};
__host__ __device__ inline size_t cluster_state_bytes(unsigned n_cap) { return (size_t)n_cap * (8 + 4 + 4 + 4); }

struct ClusterShared {
    double wd[32];
    unsigned wi[32];
    unsigned a, b, go, n_list, carry;
};

// one warp: nn[i] / nnd[i] = smallest (D[i][j], j) over j > i (none: n / +inf)
__device__ __forceinline__ void cluster_rescan_row(const double* D, unsigned n, unsigned i, ClusterSmem& st) {
    const int lane = threadIdx.x & 31;
    const double* row = D + (size_t)i * n;
    double bd = INFINITY;
    unsigned bj = n;
    for (unsigned j = i + 1 + lane; j < n; j += 32) {
        const double d = row[j];
        if (d < bd) {
            bd = d;
            bj = j;
        }
    }
    warp_argmin(bd, bj);
    if (lane == 0) {
        st.nn[i] = bj;
        st.nnd[i] = bd;
    }
}

template <int KIND>
__device__ void cluster_segment(const ClusterArgs& a, unsigned s, double* D, ClusterSmem& st, ClusterShared& sh) {
    const unsigned begin = (unsigned)a.offsets[s], n = (unsigned)(a.offsets[s + 1] - a.offsets[s]);
    const unsigned tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, n_warps = nt >> 5;
    // distances, upper triangle, one warp per row: the operands and the inlined config_distance of pairwise_distance_kernel,
    // so the same bits
    for (unsigned p = warp; p < n; p += n_warps) {
        const size_t ip = a.order ? a.order[begin + p] : begin + p;
        const double* from = reinterpret_cast<const double*>(a.results + ip * a.rec_stride);
        const bool from_contact = record_in_contact(a.results, a.rec_stride, a.cfg_stride, ip);
        for (unsigned q = p + 1 + lane; q < n; q += 32) {
            const size_t iq = a.order ? a.order[begin + q] : begin + q;
            // NaN and the contact split in one test: key_distance here costs cluster_large_kernel<SE2> a spill
            double d = config_distance<KIND>(*a.robot, from, reinterpret_cast<const double*>(a.results + iq * a.rec_stride));
            if (isnan(d) || (a.separate_contact && record_in_contact(a.results, a.rec_stride, a.cfg_stride, iq) != from_contact)) d = INFINITY;
            D[(size_t)p * n + q] = d;
        }
    }
    for (unsigned p = tid; p < n; p += nt) st.rep[p] = p;
    __syncthreads();
    for (unsigned i = warp; i < n; i += n_warps) cluster_rescan_row(D, n, i, st);
    __syncthreads();

    unsigned merges = 0;
    for (;;) {
        // smallest (nnd[i], i)
        double bd = INFINITY;
        unsigned bi = n;
        for (unsigned i = tid; i < n; i += nt) {
            const double d = st.nnd[i];
            if (d < bd) {
                bd = d;
                bi = i;
            }
        }
        warp_argmin(bd, bi);
        if (block_argmin(bd, bi, n_warps, sh.wd, sh.wi) && lane == 0) {
            sh.go = bd < INFINITY && bd <= a.threshold;
            sh.a = bi;
            sh.b = sh.go ? st.nn[bi] : 0u;
            sh.n_list = 0;
        }
        __syncthreads();
        if (!sh.go) break;
        const unsigned ca = sh.a, cb = sh.b;
        merges++;
        // row / column a <- op(a, b); b -> +inf; b's members join a
        for (unsigned k = tid; k < n; k += nt) {
            if (st.rep[k] == cb) st.rep[k] = ca;
            if (k == ca) continue;
            const size_t bk = k < cb ? (size_t)k * n + cb : (size_t)cb * n + k;
            if (k == cb) {
                D[(size_t)ca * n + cb] = INFINITY;
                continue;
            }
            const size_t ak = k < ca ? (size_t)k * n + ca : (size_t)ca * n + k;
            const double x = D[ak], y = D[bk];
            D[ak] = a.complete ? fmax(x, y) : fmin(x, y);
            D[bk] = INFINITY;
        }
        __syncthreads();
        // cache repair (rows of merged-away positions are all +inf and stay out of the argmin through nnd = +inf)
        for (unsigned i = tid; i < n; i += nt) {
            if (i == cb) {
                st.nnd[i] = INFINITY;
                st.nn[i] = n;
                continue;
            }
            if (st.rep[i] != i) continue;
            const unsigned j = st.nn[i];
            bool rescan = i == ca || j == cb;
            if (i < ca && !rescan) {
                if (j == ca) {
                    rescan = true;
                } else {
                    const double d = D[(size_t)i * n + ca];
                    if (key_less(d, ca, st.nnd[i], j)) {
                        st.nnd[i] = d;
                        st.nn[i] = ca;
                    }
                }
            }
            if (rescan) st.list[atomicAdd(&sh.n_list, 1u)] = i;
        }
        __syncthreads();
        for (unsigned r = warp; r < sh.n_list; r += n_warps) cluster_rescan_row(D, n, st.list[r], st);
        __syncthreads();
    }

    // dense ids in representative order: exclusive count of representatives below each position
    if (tid == 0) sh.carry = 0;
    __syncthreads();
    for (unsigned base = 0; base < n; base += nt) {
        const unsigned p = base + tid;
        const bool is_rep = p < n && st.rep[p] == p;
        const unsigned ballot = __ballot_sync(FKS_FULL, is_rep);
        if (lane == 0) sh.wi[warp] = (unsigned)__popc(ballot);
        __syncthreads();
        unsigned before = sh.carry + (unsigned)__popc(ballot & ((1u << lane) - 1u));
        for (unsigned w = 0; w < warp; w++) before += sh.wi[w];
        if (p < n) st.nn[p] = before;
        __syncthreads();
        if (tid == 0)
            for (unsigned w = 0; w < n_warps; w++) sh.carry += sh.wi[w];
        __syncthreads();
    }
    for (unsigned p = tid; p < n; p += nt) a.labels[begin + p] = st.nn[st.rep[p]];
    if (tid == 0) a.counts[s] = n - merges;
    __syncthreads();  // the next segment reuses the shared state
}

// segments of at most kClusterSmallMax positions: D, then the per-position state, in dynamic shared memory
template <int KIND>
__global__ void __launch_bounds__(kClusterSmallBlock) cluster_small_kernel(ClusterArgs a) {
    extern __shared__ __align__(16) unsigned char cluster_smem[];
    __shared__ ClusterShared sh;
    double* D = reinterpret_cast<double*>(cluster_smem);
    const unsigned n_cap = a.n_cap;
    ClusterSmem st;
    st.nnd = D + (size_t)n_cap * n_cap;
    st.rep = reinterpret_cast<unsigned*>(st.nnd + n_cap);
    st.nn = st.rep + n_cap;
    st.list = st.nn + n_cap;
    for (unsigned t = blockIdx.x; t < a.n_segs; t += gridDim.x) cluster_segment<KIND>(a, a.segs[t], D, st, sh);
}

// larger segments: D in the CTA's slot of the global workspace, the per-position state in dynamic shared memory
template <int KIND>
__global__ void __launch_bounds__(kClusterLargeBlock) cluster_large_kernel(ClusterArgs a) {
    extern __shared__ __align__(16) unsigned char cluster_smem[];
    __shared__ ClusterShared sh;
    const unsigned n_cap = a.n_cap;
    double* D = a.work + (size_t)blockIdx.x * n_cap * n_cap;
    ClusterSmem st;
    st.nnd = reinterpret_cast<double*>(cluster_smem);
    st.rep = reinterpret_cast<unsigned*>(st.nnd + n_cap);
    st.nn = st.rep + n_cap;
    st.list = st.nn + n_cap;
    for (unsigned t = blockIdx.x; t < a.n_segs; t += gridDim.x) cluster_segment<KIND>(a, a.segs[t], D, st, sh);
}

// labels of segment s += the clusters of the segments before it (exclusive scan of the counts)
__global__ void __launch_bounds__(256) cluster_relabel_kernel(const unsigned long long* offsets, unsigned n_segments, const unsigned* base,
                                                              unsigned* labels) {
    for (unsigned s = blockIdx.x; s < n_segments; s += gridDim.x) {
        const unsigned add = base[s];
        for (unsigned long long p = offsets[s] + threadIdx.x; p < offsets[s + 1]; p += blockDim.x) labels[p] += add;
    }
}

// one clustering kernel over the segments of `a` (none: no launch): a resident grid, at most one CTA per segment and, when
// max_grid > 0, at most max_grid CTAs
template <typename Kernel>
static int cluster_launch(Kernel k, const ClusterArgs& a, int block, size_t smem, int max_grid, cudaStream_t stream) {
    if (a.n_segs == 0) return 0;
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return (int)err;
    long long grid = resident_ctas(k, block, smem);
    if (grid > (long long)a.n_segs) grid = a.n_segs;
    if (max_grid > 0 && grid > max_grid) grid = max_grid;
    k<<<(unsigned)grid, block, smem, stream>>>(a);
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// fks_end_states_groups: the clusters of a labelled position range as particle groups.  Members: a stable counting sort by
// label -- count, the partition's one-block scan, a scatter in arrival order, then each group sorted by position in shared
// memory, so the result does not depend on the order of the scatter's atomics.  Representative: the member with the smallest
// (r, position), r(p) = max over the other members q of d(min(p,q), max(p,q)), d = the pairwise kernel's entry (same
// inlined config_distance, same operands), NaN as +inf.  Every pair is evaluated in both rows, so a row's maximum is a plain
// warp reduction; max over non-NaN values and the (r, position) argmin are exact in any order, so every result is.
//
// Clusters of up to kGroupSmallMax members get their representative from one CTA each, larger ones (up to
// kClusterMaxSegment, the largest cluster fks_end_states_cluster makes) from row chunks spread over the grid.  A call makes
// kGroupLaunches launches whatever the number and sizes of its clusters: count, scan, scatter, sort + small search, large
// rows, large argmin.
//
// Workspace (fks_sim::d_grp, u64 words): [totals (2) | row maxima (m doubles) | cursors (n_clusters), state as u32].
// ---------------------------------------------------------------------------------------------
constexpr int kGroupBlock = 256;
constexpr unsigned kGroupWarps = kGroupBlock / 32;
constexpr unsigned kGroupRowsPerTask = 32;  // rows of a large cluster per task of the row pass
constexpr unsigned kGroupSmallMax = 256;
constexpr unsigned kGroupErrLabel = 1, kGroupErrEmpty = 2, kGroupErrLarge = 4;  // bits of GroupsLaunch::state[1]
constexpr int kGroupLaunches = 6;

struct GroupsLaunch {
    const DevRobot* robot;
    const char* results;
    size_t rec_stride;
    int cfg_stride;
    const unsigned* order;          // device, or null
    const unsigned* labels;         // device [m]
    unsigned m, n_clusters;
    unsigned* offsets;              // device [n_clusters + 1] (the caller's)
    unsigned* members;              // device [m] (the caller's)
    unsigned* reps;                 // device [n_clusters]
    double* radius;                 // device [n_clusters]
    unsigned long long* totals;     // workspace [2]
    double* row_max;                // workspace [m]: r of every member of a large cluster, by slot
    unsigned* cursor;               // workspace [n_clusters], zeroed
    unsigned* state;                // workspace [2 + m / (kGroupSmallMax + 1) + 1], zeroed: large clusters, error bits, their list
};

// pass 1: members per label into offsets[0 .. n_clusters) (zeroed), error bit for labels out of range
__global__ void __launch_bounds__(kGroupBlock) groups_count_kernel(const unsigned* labels, unsigned m, unsigned n_clusters, unsigned* counts,
                                                                   unsigned* state) {
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (size_t)gridDim.x * blockDim.x) {
        const unsigned l = labels[p];
        if (l < n_clusters) atomicAdd(&counts[l], 1u);
        else atomicOr(&state[1], kGroupErrLabel);
    }
}

// pass 3 (after the scan): positions into their group's range in arrival order; offsets[n_clusters] = positions with a valid label
__global__ void __launch_bounds__(kGroupBlock) groups_scatter_kernel(const unsigned* labels, unsigned m, unsigned n_clusters, unsigned* offsets,
                                                                     const unsigned long long* totals, unsigned* cursor, unsigned* members) {
    if (blockIdx.x == 0 && threadIdx.x == 0) offsets[n_clusters] = (unsigned)totals[1];
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (size_t)gridDim.x * blockDim.x) {
        const unsigned l = labels[p];
        if (l < n_clusters) members[offsets[l] + atomicAdd(&cursor[l], 1u)] = (unsigned)p;
    }
}

// one warp: r of member i of a group whose record ids are ids[0 .. k), in position order (every lane gets it)
template <int KIND>
__device__ __forceinline__ double group_row_max(const GroupsLaunch& g, const unsigned* ids, unsigned k, unsigned i) {
    const unsigned lane = threadIdx.x & 31;
    const double* rec_i = reinterpret_cast<const double*>(g.results + (size_t)ids[i] * g.rec_stride);
    double r = -INFINITY;
    for (unsigned j = lane; j < k; j += 32) {
        if (j == i) continue;
        const double* rec_j = reinterpret_cast<const double*>(g.results + (size_t)ids[j] * g.rec_stride);
        const double d = key_distance<KIND>(*g.robot, j > i ? rec_i : rec_j, j > i ? rec_j : rec_i);
        if (d > r) r = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(FKS_FULL, r, o);
        if (x > r) r = x;
    }
    return k == 1 ? 0.0 : r;
}

// pass 4, one CTA per group: check its size, sort its positions (bitonic, padded to a power of two), write its record ids;
// groups of up to kGroupSmallMax members get their representative here, larger ones go on the list of the row pass
template <int KIND>
__global__ void __launch_bounds__(kGroupBlock) groups_sort_small_kernel(GroupsLaunch g) {
    __shared__ unsigned key[kClusterMaxSegment];
    __shared__ double wd[kGroupWarps];
    __shared__ unsigned wi[kGroupWarps];
    const unsigned tid = threadIdx.x, warp = tid >> 5;
    for (unsigned c = blockIdx.x; c < g.n_clusters; c += gridDim.x) {
        const unsigned begin = g.offsets[c], k = g.offsets[c + 1] - begin;
        if (k == 0 || k > kClusterMaxSegment) {
            if (tid == 0) atomicOr(&g.state[1], k == 0 ? kGroupErrEmpty : kGroupErrLarge);
            continue;
        }
        unsigned n2 = 1;
        while (n2 < k) n2 <<= 1;
        for (unsigned i = tid; i < n2; i += kGroupBlock) key[i] = i < k ? g.members[begin + i] : 0xffffffffu;
        __syncthreads();
        for (unsigned size = 2; size <= n2; size <<= 1) {
            for (unsigned stride = size >> 1; stride > 0; stride >>= 1) {
                for (unsigned t = tid; t < n2 / 2; t += kGroupBlock) {
                    const unsigned i = 2 * stride * (t / stride) + t % stride, j = i + stride;
                    const unsigned x = key[i], y = key[j];
                    if ((x > y) == ((i & size) == 0)) {
                        key[i] = y;
                        key[j] = x;
                    }
                }
                __syncthreads();
            }
        }
        for (unsigned i = tid; i < k; i += kGroupBlock) {
            const unsigned id = g.order ? g.order[key[i]] : key[i];
            key[i] = id;
            g.members[begin + i] = id;
        }
        __syncthreads();
        if (k > kGroupSmallMax) {
            if (tid == 0) g.state[2 + atomicAdd(&g.state[0], 1u)] = c;
            continue;
        }
        double bd = INFINITY;
        unsigned bi = k;
        for (unsigned i = warp; i < k; i += kGroupWarps) {
            const double r = group_row_max<KIND>(g, key, k, i);
            if (key_less(r, i, bd, bi)) {
                bd = r;
                bi = i;
            }
        }
        block_argmin(bd, bi, kGroupWarps, wd, wi);
        if (tid == 0) {
            g.reps[c] = key[bi];
            g.radius[c] = bd;
        }
        __syncthreads();  // the next group reuses key, wd, wi
    }
}

// pass 5: r of every member of the listed groups.  Group e's rows form tasks of kGroupRowsPerTask rows, numbered on from the
// tasks of the groups before it; task T goes to CTA T mod gridDim.x.
template <int KIND>
__global__ void __launch_bounds__(kGroupBlock) groups_large_rows_kernel(GroupsLaunch g) {
    const unsigned n_large = g.state[0], warp = threadIdx.x >> 5, lane = threadIdx.x & 31, G = gridDim.x;
    unsigned shift = 0;  // (tasks of the groups before e) mod G
    for (unsigned e = 0; e < n_large; e++) {
        const unsigned c = g.state[2 + e], begin = g.offsets[c], k = g.offsets[c + 1] - begin;
        const unsigned n_tasks = (k + kGroupRowsPerTask - 1) / kGroupRowsPerTask;
        for (unsigned t = (blockIdx.x + G - shift) % G; t < n_tasks; t += G) {
            const unsigned end = min(k, (t + 1) * kGroupRowsPerTask);
            for (unsigned i = t * kGroupRowsPerTask + warp; i < end; i += kGroupWarps) {
                const double r = group_row_max<KIND>(g, g.members + begin, k, i);
                if (lane == 0) g.row_max[begin + i] = r;
            }
        }
        shift = (shift + n_tasks) % G;
    }
}

// pass 6: one CTA per listed group, the smallest (r, position)
__global__ void __launch_bounds__(kGroupBlock) groups_large_argmin_kernel(GroupsLaunch g) {
    __shared__ double wd[kGroupWarps];
    __shared__ unsigned wi[kGroupWarps];
    const unsigned n_large = g.state[0];
    for (unsigned e = blockIdx.x; e < n_large; e += gridDim.x) {
        const unsigned c = g.state[2 + e], begin = g.offsets[c], k = g.offsets[c + 1] - begin;
        double bd = INFINITY;
        unsigned bi = k;
        for (unsigned i = threadIdx.x; i < k; i += kGroupBlock) {
            const double r = g.row_max[begin + i];
            if (key_less(r, i, bd, bi)) {
                bd = r;
                bi = i;
            }
        }
        warp_argmin(bd, bi);
        block_argmin(bd, bi, kGroupWarps, wd, wi);
        if (threadIdx.x == 0) {
            g.reps[c] = g.members[begin + bi];
            g.radius[c] = bd;
        }
        __syncthreads();
    }
}

// fks_end_states_gather_starts: value v of the outputs is component v mod cfg_stride of slot v / cfg_stride
__global__ void __launch_bounds__(256) gather_starts_kernel(const char* results, size_t rec_stride, int cfg_stride, const unsigned* offsets,
                                                            const unsigned* members, const unsigned* selected, unsigned per_group,
                                                            size_t n_values, const double* group_targets, double* starts, double* targets) {
    for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_values; v += (size_t)gridDim.x * blockDim.x) {
        const unsigned slot = (unsigned)(v / (unsigned)cfg_stride), t = (unsigned)(v % (unsigned)cfg_stride);
        const unsigned s = slot / per_group, j = slot % per_group;
        const unsigned g = selected[s], begin = offsets[g], k = offsets[g + 1] - begin;
        starts[v] = k ? reinterpret_cast<const double*>(results + (size_t)members[begin + j % k] * rec_stride)[t] : NAN;
        if (targets) targets[v] = group_targets[(size_t)s * cfg_stride + t];
    }
}

// ---------------------------------------------------------------------------------------------
// fks_nearest_configurations: per query the k <= kNearestMaxK smallest keys (d, i), d = config_distance<KIND>(candidate i,
// query) -- the pairwise kernel's inlined distance with the candidate as `cur`, as in its entry [i][m + j] -- NaN as +inf.
// A warp keeps a query's running list sorted by key over 64 positions, position p in lane p mod 32 (slot p / 32); a key
// enters only if it is below the one at position k - 1.  Keys are a total order, so the k smallest of a union are the k
// smallest of the parts' k smallest: any split of the candidates and any merge order give the same bits.
//
// With n_split == 1 one scan launch writes the output (the query-tiled path); with n_split > 1 each query's candidates are
// cut into n_split chunks of `chunk`, the scan writes a list per (query, chunk) to the workspace (fks_sim::near:
// [distances | ids as u32]) and a second launch merges them.
// ---------------------------------------------------------------------------------------------
constexpr unsigned kNearestMaxK = 64;
constexpr int kNearestBlock = 256;
constexpr unsigned kNearestWarps = kNearestBlock / 32;  // queries per CTA of the scan
constexpr unsigned kNearestTileDoubles = 4096;          // the candidate tile in shared memory (32 KiB)
constexpr unsigned kNearestCtasPerSm = 4;     // the scan's grid the split aims at
constexpr unsigned kNearestMinChunk = 2048;   // fewest candidates per chunk of a split

struct NearestLaunch {
    const DevRobot* robot;
    const double* candidates;  // device [m][cfg_stride]
    const double* queries;     // device [n_queries][cfg_stride]
    int cfg_stride;
    unsigned m, n_queries, k;
    unsigned n_split, chunk;
    unsigned* ids;             // device [n_queries * k] (the caller's)
    double* distances;         // device [n_queries * k] (the caller's)
    double* part_d;            // workspace [n_queries * n_split * k] when n_split > 1
    unsigned* part_i;          // workspace [n_queries * n_split * k] when n_split > 1
};

struct NearestList {
    double d0, d1;    // keys at positions lane, 32 + lane
    unsigned i0, i1;
};

struct NearestShared {
    double d[kNearestWarps][kNearestMaxK];
    unsigned i[kNearestWarps][kNearestMaxK];
};

__device__ __forceinline__ void nearest_list_init(NearestList& L, double& kd, unsigned& ki) {
    L.d0 = L.d1 = kd = INFINITY;
    L.i0 = L.i1 = ki = kNoIndex;
}

// (d, i), the same in every lane, goes to its rank; the key at position 63 drops out.  kd / ki = the key at position k - 1.
__device__ __forceinline__ void nearest_insert(NearestList& L, unsigned k, double& kd, unsigned& ki, double d, unsigned i) {
    const unsigned lane = threadIdx.x & 31;
    const unsigned pos = __popc(__ballot_sync(FKS_FULL, key_less(L.d0, L.i0, d, i))) +
                         __popc(__ballot_sync(FKS_FULL, key_less(L.d1, L.i1, d, i)));
    const double up_d0 = __shfl_up_sync(FKS_FULL, L.d0, 1), last_d0 = __shfl_sync(FKS_FULL, L.d0, 31);
    const unsigned up_i0 = __shfl_up_sync(FKS_FULL, L.i0, 1), last_i0 = __shfl_sync(FKS_FULL, L.i0, 31);
    double up_d1 = __shfl_up_sync(FKS_FULL, L.d1, 1);
    unsigned up_i1 = __shfl_up_sync(FKS_FULL, L.i1, 1);
    if (lane == 0) {
        up_d1 = last_d0;
        up_i1 = last_i0;
    }
    if (lane == pos) {
        L.d0 = d;
        L.i0 = i;
    } else if (lane > pos) {
        L.d0 = up_d0;
        L.i0 = up_i0;
    }
    if (lane + 32 == pos) {
        L.d1 = d;
        L.i1 = i;
    } else if (lane + 32 > pos) {
        L.d1 = up_d1;
        L.i1 = up_i1;
    }
    kd = __shfl_sync(FKS_FULL, k > 32 ? L.d1 : L.d0, (k - 1) & 31);
    ki = __shfl_sync(FKS_FULL, k > 32 ? L.i1 : L.i0, (k - 1) & 31);
}

// every lane offers one key; those below the k-th enter in lane order (invalid lanes offer (+inf, kNoIndex))
__device__ __forceinline__ void nearest_offer(NearestList& L, unsigned k, double& kd, unsigned& ki, double d, unsigned i) {
    unsigned mask = __ballot_sync(FKS_FULL, key_less(d, i, kd, ki));
    while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const double bd = __shfl_sync(FKS_FULL, d, src);
        const unsigned bi = __shfl_sync(FKS_FULL, i, src);
        if (key_less(bd, bi, kd, ki)) nearest_insert(L, k, kd, ki, bd, bi);
    }
}

// the first k keys of a stored list
__device__ __forceinline__ void nearest_offer_list(NearestList& L, unsigned k, double& kd, unsigned& ki, const double* d, const unsigned* id) {
    const unsigned lane = threadIdx.x & 31;
    for (unsigned p0 = 0; p0 < k; p0 += 32) {
        const unsigned p = p0 + lane;
        nearest_offer(L, k, kd, ki, p < k ? d[p] : INFINITY, p < k ? id[p] : kNoIndex);
    }
}

__device__ __forceinline__ void nearest_store(const NearestList& L, unsigned k, double* d, unsigned* id) {
    const unsigned lane = threadIdx.x & 31;
    if (lane < k) {
        d[lane] = L.d0;
        id[lane] = L.i0;
    }
    if (lane + 32 < k) {
        d[lane + 32] = L.d1;
        id[lane + 32] = L.i1;
    }
}

// warps q + s * n_lists, 0 < s < per, hand their lists to warp q through shared memory (per is the same in the whole CTA)
__device__ __forceinline__ void nearest_block_merge(NearestList& L, unsigned k, double& kd, unsigned& ki, unsigned n_lists, unsigned per,
                                                    NearestShared& sh) {
    const unsigned warp = threadIdx.x >> 5;
    if (per == 1) return;
    if (warp >= n_lists && warp < n_lists * per) nearest_store(L, k, sh.d[warp], sh.i[warp]);
    __syncthreads();
    if (warp < n_lists)
        for (unsigned s = 1; s < per; s++) nearest_offer_list(L, k, kd, ki, sh.d[warp + s * n_lists], sh.i[warp + s * n_lists]);
}

// CTA (x, y): queries 8x .. 8x + qt - 1 against chunk y of the candidates, streamed through shared memory in coalesced tiles.
// With qt < 8 queries, per = 8 / qt warps share a query, each taking every per-th group of 32 candidates of a tile.
template <int KIND>
__global__ void __launch_bounds__(kNearestBlock) nearest_scan_kernel(NearestLaunch a) {
    __shared__ double cand[kNearestTileDoubles];
    __shared__ double qry[kNearestWarps * kCfgMax];
    __shared__ NearestShared sh;
    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, S = (unsigned)a.cfg_stride;
    const unsigned q0 = blockIdx.x * kNearestWarps, qt = min(kNearestWarps, a.n_queries - q0), per = kNearestWarps / qt;
    const unsigned qi = warp % qt, sub = warp / qt;
    for (unsigned t = tid; t < qt * S; t += kNearestBlock) qry[t] = a.queries[(size_t)q0 * S + t];
    const unsigned c_begin = blockIdx.y * a.chunk, c_end = (unsigned)min((size_t)a.m, (size_t)c_begin + a.chunk), tile = kNearestTileDoubles / S;
    NearestList L;
    double kd;
    unsigned ki;
    nearest_list_init(L, kd, ki);
    for (unsigned c0 = c_begin, n; c0 < c_end; c0 += n) {
        n = min(tile, c_end - c0);
        __syncthreads();  // the previous tile is consumed (and the queries are in place)
        const double* src = a.candidates + (size_t)c0 * S;
        for (unsigned t = tid; t < n * S; t += kNearestBlock) cand[t] = src[t];
        __syncthreads();
        if (sub >= per) continue;
        for (unsigned b = sub * 32; b < n; b += 32 * per) {
            const unsigned c = b + lane;
            double d = INFINITY;
            unsigned id = kNoIndex;
            if (c < n) {
                d = key_distance<KIND>(*a.robot, cand + c * S, qry + qi * S);
                id = c0 + c;
            }
            nearest_offer(L, a.k, kd, ki, d, id);
        }
    }
    nearest_block_merge(L, a.k, kd, ki, qt, per, sh);
    if (warp >= qt) return;
    const size_t q = q0 + qi;
    if (a.n_split == 1) nearest_store(L, a.k, a.distances + q * a.k, a.ids + q * a.k);
    else nearest_store(L, a.k, a.part_d + (q * a.n_split + blockIdx.y) * a.k, a.part_i + (q * a.n_split + blockIdx.y) * a.k);
}

// one CTA per query: warp w takes the chunk lists w, w + 8, ..., then warp 0 takes the other warps' lists
__global__ void __launch_bounds__(kNearestBlock) nearest_merge_kernel(NearestLaunch a) {
    __shared__ NearestShared sh;
    const unsigned warp = threadIdx.x >> 5;
    const size_t q = blockIdx.x;
    NearestList L;
    double kd;
    unsigned ki;
    nearest_list_init(L, kd, ki);
    for (unsigned s = warp; s < a.n_split; s += kNearestWarps)
        nearest_offer_list(L, a.k, kd, ki, a.part_d + (q * a.n_split + s) * a.k, a.part_i + (q * a.n_split + s) * a.k);
    nearest_block_merge(L, a.k, kd, ki, 1, kNearestWarps, sh);
    if (warp == 0) nearest_store(L, a.k, a.distances + q * a.k, a.ids + q * a.k);
}

// Split only when the query tiles would fill at most half of a kNearestCtasPerSm grid: then up to the grid's worth of
// chunks per tile, none below kNearestMinChunk candidates.
static unsigned nearest_split(unsigned m, unsigned n_queries, int num_sms) {
    const size_t tiles = ((size_t)n_queries + kNearestWarps - 1) / kNearestWarps;
    const size_t target = (size_t)kNearestCtasPerSm * (size_t)(num_sms > 0 ? num_sms : 1);
    if (tiles == 0 || 2 * tiles > target) return 1;
    const size_t by_m = ((size_t)m + kNearestMinChunk - 1) / kNearestMinChunk;
    const size_t s = target / tiles < by_m ? target / tiles : by_m;
    return s > 1 ? (unsigned)s : 1u;
}

}  // namespace fksdev

using namespace fksdev;

int fks_host::StreamBuffer::acquire(size_t bytes, cudaStream_t stream) {
    if (!done) FKS_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    if (pending && bytes > cap) FKS_CUDA(cudaEventSynchronize(done));
    const int rc = ensure(&ptr, &cap, bytes);
    if (rc != FKS_OK) return rc;
    if (pending) FKS_CUDA(cudaStreamWaitEvent(stream, done, 0));
    return FKS_OK;
}

int fks_host::StreamBuffer::release(cudaStream_t stream) {
    FKS_CUDA(cudaEventRecord(done, stream));
    pending = true;
    return FKS_OK;
}

void fks_host::StreamBuffer::destroy() {
    if (pending) cudaEventSynchronize(done);
    cudaFree(ptr);
    if (done) cudaEventDestroy(done);
}

extern "C" {

int fks_end_states_partition(fks_sim* s, const void* d_results, size_t n, uint32_t* d_order, uint64_t* counts, void* cuda_stream) {
    if (!s || !counts) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_partition: null argument");
    counts[0] = counts[1] = 0;
    if (n == 0) return FKS_OK;
    if (!d_results || !d_order || n > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_partition: bad buffer or count");
    NvtxRange range("fks_end_states_partition");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_partition: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const char* results = (const char*)d_results;
    const size_t rec_stride = fks_sim_result_stride(s);
    const int cfg_stride = s->robot->stride;
    const unsigned n_blocks = (unsigned)((n + kPartitionBlock - 1) / kPartitionBlock);
    // workspace (fks_sim::d_part, u32 words): [totals (2 x u64) | block counts]
    const int rc = ensure(&s->d_part, &s->cap_part, n_blocks + 4);
    if (rc != FKS_OK) return rc;
    unsigned long long* totals = reinterpret_cast<unsigned long long*>(s->d_part);
    unsigned* block_counts = s->d_part + 4;
    partition_count_kernel<<<n_blocks, kPartitionBlock, 0, stream>>>(results, rec_stride, cfg_stride, n, block_counts);
    partition_scan_kernel<<<1, kPartitionBlock, 0, stream>>>(block_counts, n_blocks, n, totals);
    partition_scatter_kernel<<<n_blocks, kPartitionBlock, 0, stream>>>(results, rec_stride, cfg_stride, n, block_counts, totals, d_order);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return cuda_fail(err, "fks_end_states_partition: launch");
    s->launches += 3;
    unsigned long long host[2] = {0, 0};
    FKS_CUDA(cudaMemcpyAsync(host, totals, sizeof(host), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaStreamSynchronize(stream));
    counts[0] = host[0];
    counts[1] = host[1];
    return FKS_OK;
}

int fks_end_states_pairwise_distance(fks_sim* s, const void* d_results, const uint32_t* d_subset, size_t m, double* d_out, void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_pairwise_distance: null simulator");
    if (m == 0) return FKS_OK;
    if (!d_results || !d_out || m > 65535) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_pairwise_distance: bad buffer, or more than 65535 records");
    NvtxRange range("fks_end_states_pairwise_distance");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_pairwise_distance: cudaSetDevice failed");
    const int rc = for_kind(s->robot->host.kind, [&](auto K) {
        pairwise_distance_kernel<decltype(K)::value><<<dim3((unsigned)(m + 255) / 256, (unsigned)m), 256, 0, (cudaStream_t)cuda_stream>>>(
            s->robot->d_robot, (const char*)d_results, fks_sim_result_stride(s), s->robot->stride, d_subset, (unsigned)m, d_out);
        return (int)cudaGetLastError();
    });
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_pairwise_distance: launch");
    s->launches += 1;
    return FKS_OK;
}

int fks_end_states_cluster(fks_sim* s, const void* d_results, const uint32_t* d_order, const uint64_t* segment_offsets, size_t n_segments,
                           int linkage, double max_cluster_distance, int separate_contact, uint32_t* d_labels, uint64_t* cluster_counts,
                           void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: null simulator");
    if (std::isnan(max_cluster_distance)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: max_cluster_distance is NaN");
    if (linkage != FKS_LINKAGE_SINGLE && linkage != FKS_LINKAGE_COMPLETE) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: unknown linkage");
    if (n_segments == 0) return FKS_OK;
    if (!segment_offsets || !cluster_counts) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: null segment offsets or counts");
    if (n_segments > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: more than 2^32 - 1 segments");
    if (segment_offsets[0] != 0) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: segment_offsets[0] must be 0");
    std::vector<uint32_t> small_segs, large_segs;
    unsigned small_cap = 0, large_cap = 0;
    for (size_t i = 0; i < n_segments; i++) {
        if (segment_offsets[i + 1] < segment_offsets[i]) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: segment_offsets decrease");
        const uint64_t len = segment_offsets[i + 1] - segment_offsets[i];
        if (len > kClusterMaxSegment)
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: a segment is longer than " + std::to_string(kClusterMaxSegment) + " positions");
        if (len == 0) continue;
        if (len <= kClusterSmallMax) {
            small_segs.push_back((uint32_t)i);
            small_cap = std::max(small_cap, (unsigned)len);
        } else {
            large_segs.push_back((uint32_t)i);
            large_cap = std::max(large_cap, (unsigned)len);
        }
    }
    const uint64_t m = segment_offsets[n_segments];
    if (m > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: 2^32 or more positions");
    std::fill(cluster_counts, cluster_counts + n_segments, (uint64_t)0);
    if (m == 0) return FKS_OK;
    if (!d_results || !d_labels) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_cluster: null records or labels");
    NvtxRange range("fks_end_states_cluster");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_cluster: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;

    // one upload of the workspace's head, with the counts zeroed
    const size_t n_u32 = n_segments + small_segs.size() + large_segs.size();
    std::vector<unsigned long long> meta(n_segments + 3 + (n_u32 + 1) / 2, 0ull);
    std::memcpy(meta.data(), segment_offsets, (n_segments + 1) * sizeof(uint64_t));
    uint32_t* meta32 = reinterpret_cast<uint32_t*>(meta.data() + n_segments + 3);
    std::copy(small_segs.begin(), small_segs.end(), meta32 + n_segments);
    std::copy(large_segs.begin(), large_segs.end(), meta32 + n_segments + small_segs.size());
    int rc;
    if ((rc = ensure(&s->d_clu, &s->cap_clu, meta.size())) != FKS_OK) return rc;
    // large segments: one matrix slot per CTA, as many CTAs as SMs, segments and a 1 GiB workspace allow (at least one)
    int large_slots = 0;
    if (!large_segs.empty()) {
        const size_t slot = (size_t)large_cap * large_cap;
        large_slots = (int)std::max<size_t>(1, std::min<size_t>({large_segs.size(), (size_t)s->num_sms, ((size_t)1 << 30) / (slot * sizeof(double))}));
        if ((rc = ensure(&s->d_clu_mat, &s->cap_clu_mat, slot * large_slots)) != FKS_OK) return rc;
    }
    FKS_CUDA(cudaMemcpyAsync(s->d_clu, meta.data(), meta.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, stream));
    unsigned* counts = reinterpret_cast<unsigned*>(s->d_clu + n_segments + 3);
    unsigned long long* totals = s->d_clu + n_segments + 1;
    ClusterArgs small;
    small.robot = s->robot->d_robot;
    small.results = (const char*)d_results;
    small.rec_stride = fks_sim_result_stride(s);
    small.cfg_stride = s->robot->stride;
    small.complete = linkage == FKS_LINKAGE_COMPLETE;
    small.separate_contact = separate_contact != 0;
    small.threshold = max_cluster_distance;
    small.order = d_order;
    small.offsets = s->d_clu;
    small.segs = counts + n_segments;
    small.n_segs = (unsigned)small_segs.size();
    small.n_cap = small_cap;
    small.work = nullptr;
    small.labels = d_labels;
    small.counts = counts;
    ClusterArgs large = small;
    large.segs = small.segs + small_segs.size();
    large.n_segs = (unsigned)large_segs.size();
    large.n_cap = large_cap;
    large.work = s->d_clu_mat;
    rc = for_kind(s->robot->host.kind, [&](auto K) {
        constexpr int KIND = decltype(K)::value;
        const int e = cluster_launch(cluster_small_kernel<KIND>, small, kClusterSmallBlock,
                                     (size_t)small_cap * small_cap * 8 + cluster_state_bytes(small_cap), 0, stream);
        if (e != 0) return e;
        return cluster_launch(cluster_large_kernel<KIND>, large, kClusterLargeBlock, cluster_state_bytes(large_cap), large_slots, stream);
    });
    if (rc == 0) {
        // base of every segment's ids: partition's exclusive scan, in place over the counts (totals[1] = all clusters)
        partition_scan_kernel<<<1, kPartitionBlock, 0, stream>>>(counts, (unsigned)n_segments, 0, totals);
        const unsigned relabel_grid = n_segments < 65535u ? (unsigned)n_segments : 65535u;
        cluster_relabel_kernel<<<relabel_grid, 256, 0, stream>>>(s->d_clu, (unsigned)n_segments, counts, d_labels);
        rc = (int)cudaGetLastError();
    }
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_cluster: launch");
    s->launches += 2 + (small_segs.empty() ? 0 : 1) + (large_segs.empty() ? 0 : 1);
    std::vector<unsigned> base(n_segments);
    unsigned long long total = 0;
    FKS_CUDA(cudaMemcpyAsync(base.data(), counts, n_segments * sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaMemcpyAsync(&total, totals + 1, sizeof(total), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaStreamSynchronize(stream));
    for (size_t i = 0; i < n_segments; i++) cluster_counts[i] = (i + 1 < n_segments ? base[i + 1] : total) - base[i];
    return FKS_OK;
}

int fks_end_states_groups(fks_sim* s, const void* d_results, const uint32_t* d_order, size_t m, const uint32_t* d_labels, size_t n_clusters,
                          uint32_t* d_group_offsets, uint32_t* d_members, uint32_t* d_representatives, double* d_radius,
                          uint64_t* group_sizes, void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: null simulator");
    if (m > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: 2^32 or more positions");
    if (n_clusters > m) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: more clusters than positions");
    if (m == 0) return FKS_OK;
    if (!d_results || !d_labels || !d_group_offsets || !d_members || !d_representatives || !d_radius || !group_sizes)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: null buffer");
    if (n_clusters == 0) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: a label is not below n_clusters");
    NvtxRange range("fks_end_states_groups");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_groups: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const size_t n_state = 2 + m / (kGroupSmallMax + 1) + 1;
    int rc;
    if ((rc = ensure(&s->d_grp, &s->cap_grp, 2 + m + (n_clusters + n_state + 1) / 2)) != FKS_OK) return rc;
    GroupsLaunch g;
    g.robot = s->robot->d_robot;
    g.results = (const char*)d_results;
    g.rec_stride = fks_sim_result_stride(s);
    g.cfg_stride = s->robot->stride;
    g.order = d_order;
    g.labels = d_labels;
    g.m = (unsigned)m;
    g.n_clusters = (unsigned)n_clusters;
    g.offsets = d_group_offsets;
    g.members = d_members;
    g.reps = d_representatives;
    g.radius = d_radius;
    g.totals = s->d_grp;
    g.row_max = reinterpret_cast<double*>(s->d_grp + 2);
    g.cursor = reinterpret_cast<unsigned*>(s->d_grp + 2 + m);
    g.state = g.cursor + n_clusters;
    FKS_CUDA(cudaMemsetAsync(d_group_offsets, 0, n_clusters * sizeof(uint32_t), stream));
    FKS_CUDA(cudaMemsetAsync(g.cursor, 0, (n_clusters + 2) * sizeof(uint32_t), stream));
    rc = for_kind(s->robot->host.kind, [&](auto K) {
        constexpr int KIND = decltype(K)::value;
        const size_t blocks = (m + kGroupBlock - 1) / kGroupBlock;
        const unsigned grid = blocks < 65535 ? (unsigned)blocks : 65535u;
        // the host does not know how many groups are large: the row and argmin passes run a full grid and read the list
        const unsigned resident = resident_ctas(groups_sort_small_kernel<KIND>, kGroupBlock, 0);
        const unsigned rows_grid = resident_ctas(groups_large_rows_kernel<KIND>, kGroupBlock, 0);
        groups_count_kernel<<<grid, kGroupBlock, 0, stream>>>(g.labels, g.m, g.n_clusters, g.offsets, g.state);
        partition_scan_kernel<<<1, kPartitionBlock, 0, stream>>>(g.offsets, g.n_clusters, g.m, g.totals);
        groups_scatter_kernel<<<grid, kGroupBlock, 0, stream>>>(g.labels, g.m, g.n_clusters, g.offsets, g.totals, g.cursor, g.members);
        groups_sort_small_kernel<KIND><<<g.n_clusters < resident ? g.n_clusters : resident, kGroupBlock, 0, stream>>>(g);
        groups_large_rows_kernel<KIND><<<rows_grid, kGroupBlock, 0, stream>>>(g);
        groups_large_argmin_kernel<<<rows_grid, kGroupBlock, 0, stream>>>(g);
        return (int)cudaGetLastError();
    });
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_groups: launch");
    s->launches += kGroupLaunches;
    std::vector<uint32_t> offsets(n_clusters + 1);
    uint32_t err = 0;
    FKS_CUDA(cudaMemcpyAsync(offsets.data(), d_group_offsets, offsets.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaMemcpyAsync(&err, g.state + 1, sizeof(err), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaStreamSynchronize(stream));
    if (err & kGroupErrLabel) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: a label is not below n_clusters");
    if (err & kGroupErrEmpty) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: a cluster has no member");
    if (err & kGroupErrLarge)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_groups: a cluster has more than " + std::to_string(kClusterMaxSegment) + " members");
    for (size_t c = 0; c < n_clusters; c++) group_sizes[c] = offsets[c + 1] - offsets[c];
    return FKS_OK;
}

int fks_end_states_gather_starts(fks_sim* s, const void* d_results, const uint32_t* d_group_offsets, const uint32_t* d_members,
                                 size_t n_clusters, const uint32_t* selected, size_t n_selected, size_t per_group,
                                 const double* d_group_targets, double* d_starts, double* d_targets, void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: null simulator");
    if (per_group == 0) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: per_group is 0");
    if ((d_targets == nullptr) != (d_group_targets == nullptr))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: d_targets and d_group_targets go together");
    if (n_selected == 0) return FKS_OK;
    if (n_selected > 0xffffffffull / per_group) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: 2^32 or more starts");
    if (!d_results || !d_group_offsets || !d_members || !selected || !d_starts)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: null buffer");
    for (size_t i = 0; i < n_selected; i++)
        if (selected[i] >= n_clusters) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_gather_starts: a selected group is not below n_clusters");
    NvtxRange range("fks_end_states_gather_starts");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_gather_starts: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    // the selected group ids go through the workspace fks_sim::sel
    int rc;
    if ((rc = s->sel.acquire(n_selected * sizeof(uint32_t), stream)) != FKS_OK) return rc;
    const unsigned* d_sel = reinterpret_cast<const unsigned*>(s->sel.ptr);
    FKS_CUDA(cudaMemcpyAsync(s->sel.ptr, selected, n_selected * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    const int cfg_stride = s->robot->stride;
    const size_t n_values = n_selected * per_group * (size_t)cfg_stride;
    const size_t grid = (n_values + 255) / 256 < 65535 ? (n_values + 255) / 256 : 65535;
    gather_starts_kernel<<<(unsigned)grid, 256, 0, stream>>>((const char*)d_results, fks_sim_result_stride(s), cfg_stride, d_group_offsets,
                                                             d_members, d_sel, (unsigned)per_group, n_values, d_group_targets, d_starts, d_targets);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return cuda_fail(err, "fks_end_states_gather_starts: launch");
    s->launches += 1;
    return s->sel.release(stream);
}

int fks_nearest_configurations(fks_sim* s, const double* d_candidates, size_t m, const double* d_queries, size_t n_queries, size_t k,
                               uint32_t* d_ids, double* d_distances, void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_nearest_configurations: null simulator");
    if (k == 0 || k > kNearestMaxK) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_nearest_configurations: k is 0 or above " + std::to_string(kNearestMaxK));
    if (m > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_nearest_configurations: 2^32 or more candidates");
    if (n_queries > 0xffffffffull / k) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_nearest_configurations: n_queries * k is 2^32 or more");
    if (n_queries == 0) return FKS_OK;
    if (!d_queries || !d_ids || !d_distances || (m > 0 && !d_candidates))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_nearest_configurations: null buffer");
    NvtxRange range("fks_nearest_configurations");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_nearest_configurations: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    NearestLaunch a;
    a.robot = s->robot->d_robot;
    a.candidates = d_candidates;
    a.queries = d_queries;
    a.cfg_stride = s->robot->stride;
    a.m = (unsigned)m;
    a.n_queries = (unsigned)n_queries;
    a.k = (unsigned)k;
    a.n_split = nearest_split(a.m, a.n_queries, s->num_sms);
    a.chunk = (unsigned)((m + a.n_split - 1) / a.n_split);
    if (a.n_split > 1) a.n_split = (unsigned)((m + a.chunk - 1) / a.chunk);  // no empty chunk
    a.ids = d_ids;
    a.distances = d_distances;
    a.part_d = nullptr;
    a.part_i = nullptr;
    if (a.n_split > 1) {
        const size_t n_keys = n_queries * a.n_split * k;
        const int rc = s->near.acquire(n_keys * sizeof(double) + n_keys * sizeof(unsigned), stream);
        if (rc != FKS_OK) return rc;
        a.part_d = reinterpret_cast<double*>(s->near.ptr);
        a.part_i = reinterpret_cast<unsigned*>(a.part_d + n_keys);
    }
    const int rc = for_kind(s->robot->host.kind, [&](auto K) {
        if (a.cfg_stride > kCfgMax) return (int)cudaErrorInvalidValue;
        const dim3 grid((a.n_queries + kNearestWarps - 1) / kNearestWarps, a.n_split);
        nearest_scan_kernel<decltype(K)::value><<<grid, kNearestBlock, 0, stream>>>(a);
        if (a.n_split > 1) nearest_merge_kernel<<<a.n_queries, kNearestBlock, 0, stream>>>(a);
        return (int)cudaGetLastError();
    });
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_nearest_configurations: launch");
    s->launches += a.n_split > 1 ? 2 : 1;
    return a.n_split > 1 ? s->near.release(stream) : FKS_OK;
}

}  // extern "C"
