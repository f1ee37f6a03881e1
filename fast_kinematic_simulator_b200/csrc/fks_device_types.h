// Device-side data model of the particle contact simulator (shared by fks_kernels.cu and fks_api.cu).
//
// Layout in HBM (uploaded once per environment / robot, read-only afterwards):
//   SDF            float[nx*ny*nz], x-major (same linear index as VoxelGrid), L2-persisting window
//   normal table   open-addressing hash  (cell index + 1) -> (first entry, entry count); entries are
//                  6 doubles (entry direction xyz, normal xyz)
//   robot          one DevRobot struct + point arrays ({x,y}[], {z,link}[]), staged into shared
//                  memory once by every CTA of the persistent kernel
//   particles      starts/targets as flat doubles (cfg_stride per particle), results as fixed records
//   scratch        one slot per resident warp: stacked Jacobian (column major) + self-collision work
#ifndef FKS_DEVICE_TYPES_H
#define FKS_DEVICE_TYPES_H

#include <stdint.h>

#include "fksgpu.h"

namespace fksdev {

constexpr int kMaxDof = 16;
constexpr int kMaxLinks = 16;
constexpr int kMaxJoints = 16;
constexpr int kMaxPairs = (kMaxLinks * (kMaxLinks - 1)) / 2;
constexpr int kMaxSelfPartners = kMaxLinks - 1;
constexpr int kPairChunks = (kMaxPairs + 31) / 32;
// 24 warps per CTA: 80 registers per thread instead of the 64 that 32 warps leave (fewer spills in the solver) and a
// bigger shared-memory block per warp; measured 3-9 % faster than 32 on the contact workloads, 2 % slower in free flight
// (profiles/r2_kernel_experiments.md)
#ifndef FKS_MAX_WARPS
#define FKS_MAX_WARPS 24
#endif
constexpr int kWarpsPerBlock = FKS_MAX_WARPS;  // upper bound of warps per CTA (launch bounds); the CTA's warps run in lock step
constexpr int kThreadsPerBlock = kWarpsPerBlock * 32;

struct DevAxis {
    double kp, ki, kd, iclamp;  // |.| already applied (pid.hpp:104-113)
    double vlim;                // |velocity_limit| (unc.hpp:61)
    double pnoise, mnoise;      // |.| applied
    double sigma;
};

struct DevJoint {
    int parent, child, type, active;  // active = index among non-fixed joints, -1 if fixed
    double T[12];
    double axis[3];
    double lo, hi, weight;
    // M_j(q) = T + s1 C1 + s2 C2 with (s1, s2) = (sin q, 1 - cos q) for revolute / continuous joints (C1 = T K, C2 = T K^2,
    // K = [axis]x: Rodrigues' form of T R(q)), (q, 0) for prismatic ones (C1 = [0 | T axis]); filled by fks_robot_create
    double C1[12], C2[12];
};

struct DevRobot {
    int kind, L, J, D, P, n_pairs;
    double base[12];
    double pos_w, rot_w;
    DevAxis axes[kMaxDof];
    DevJoint joints[kMaxJoints];
    unsigned long long joint_parents, joint_children;  // link indices of joint j in bits 4j .. 4j+3 (kMaxLinks = kMaxJoints = 16)
    int active_joint[kMaxDof];        // active dof -> joint index
    int link_begin[kMaxLinks + 1];
    unsigned link_ancestors[kMaxLinks];  // bit j: joint j is on the path from the root to this link
    unsigned disallowed[kMaxLinks];      // bit j: self collision between this link and j is NOT allowed
    unsigned char pair_a[kMaxPairs], pair_b[kMaxPairs];  // the disallowed pairs, a < b
    double cap_p0[kMaxLinks][3], cap_p1[kMaxLinks][3];  // bounding capsule of the link's points (link frame)
    double cap_radius[kMaxLinks];
    double sph_center[kMaxLinks][3];  // bounding sphere of the link's points (link frame): link-level SDF culling
    double sph_radius[kMaxLinks];
    double link_mass[kMaxLinks];         // cumulative point counts (spcs.hpp:1244-1255)
};

struct DevEnv {
    double origin[12];
    double inv_origin[12];
    double map_res, sdf_res;
    double inv_sdf_res;      // 1.0 / sdf_res (VoxelGrid multiplies by the inverse cell size)
    double inv_twice_res;    // 1.0 / (2.0 * sdf_res)
    int nx, ny, nz;
    float oob;
    int cull;                // 1: the SDF is a true distance field (checked at upload): link-level culling is exact
    int _pad;
    const float* sdf;
    // normal hash: 16-byte entries {linear cell index + 1 (0 = empty slot), first entry | entry count << 32}
    const unsigned long long* nh_keys;
    unsigned long long nh_mask;
    const double* normal_entries;  // 6 doubles: entry direction xyz, normal xyz
};

struct DevSolver {
    double interval;          // 1 / frequency, sign kept (spcs.hpp:427)
    double shortcut_distance;
    double check_tolerance;
    double decay_rate, initial_step, min_scaling;
    unsigned max_iters, decay_iters, n_steps;
    int failed_ends_motion;
};

// hash of a linear cell index into the normal table (same function on host and device)
inline __host__ __device__ unsigned long long normal_hash(unsigned long long cell) {
    unsigned long long h = cell * 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}

// per-particle bookkeeping of a warp, kept in shared memory (uniform across lanes)
struct WarpVars {
    unsigned long long pid, tape_pos, tape_end;
    unsigned long long dec_pos, dec_end;  // decision tape (parity mode): next / one-past-last record of this particle
    double scaling;
    double m_result;  // last motion estimate
    unsigned step, micro, number_microsteps, resolver_iterations, flags, n_micro_total, n_iter_total, n_steps;
    int collided, any_resolve_failed, step_collided, step_failed, step_stopped;
    // control state of the particle's state machine (registers while a phase runs, here in between: the context may be
    // picked up by another warp): what to do next (after), the pending operation of phase A / B, the ping-pong indices of
    // the current / previous kinematic state, the last collision bits, and whether the next thing it needs is a contact solve
    int after, op, op_in, op_out, op_u, op_tn, op_derive, measure, cur, prev, want_solve;
    unsigned cc;
    // leg of a sequence call the particle is in, top bit: the next leg is due (used by the sequence kernel only).  Here,
    // behind the fields above: inserted among them it shifts their offsets, and the single-call kernel's spill code with them
    unsigned leg;
    int ctx;        // index of this context in the CTA's pool (fixed: its slot of the global context store)
};
constexpr int kWarpVarsDoubles = (int)((sizeof(WarpVars) + 7) / 8);

// ---- per-warp shared memory layout (offsets in doubles from the start of the warp's block) -----
// Three kinematic states X = 0, 1, 2: configuration cfg + X*S and link transforms T + X*L12.  States 0 / 1
// ping-pong between "previous" and "current" configuration of a microstep, state 2 is the scratch state of
// the motion estimates.  G / caps are derived from the CURRENT state only.
// The stacked Jacobian of a contact solve lives in shared memory when it is small (jsm): the region aliases what is dead
// between the collision check and the motion estimate of the correction -- the scratch state's transforms, the joint
// matrices and the capsule end points (all rebuilt before they are read again) -- plus whatever shared memory the robot
// leaves free (jsm_extra).  Once the corrections are COLLECTED the world->voxel transforms, the joint axes / origins and the
// candidate list are dead as well (the next apply rebuilds what is needed): a system that outgrew the small store is moved
// from the warp's global scratch slot into this larger one (jsm_big_ld) for the solve.  Only systems taller than that are
// factored in global memory, where every load of the in-place update is an L2 round trip.
struct WarpLayout {
    int S;        // vector slot (doubles) >= max(cfg_stride, D), even
    int L12;      // 12 * links
    int cfg;      // 3 * S
    int T;        // 3 * L12; state 2 is the LAST one and starts the jsm region
    int G;        // L12: per link, (1/res) * inverse_origin * T_link  (world -> voxel coordinates in one transform); after the jsm store
    int caps;     // 6 * L: world end points of every link's bounding capsule
    int M;        // 16 * J: joint_transform * motion(value), by columns
    int jsm;      // start of the shared-memory Jacobian store (= T + 2 * L12)
    int jsm_ld;   // its leading dimension
    int jsm_big_ld;  // leading dimension of the larger store that opens up once the corrections are collected (see below)
    int jaxis, jorig;  // 3 * J each
    int target, scfg, act, ru, du, raw, stepv;  // S each
    int tn;       // noise_batch * S: truncated-normal draws of the next noise_batch microsteps
    int qr;       // S doubles: the actuated twist of the SE(3) robot (apply_control)
    int cand;     // 32 doubles = 32 candidate records of collect_corrections
    int vars;     // WarpVars (kWarpVarsDoubles) + 2 * S doubles of PID state (inside [target, save2_end): parked with the context)
    int flags;    // 1 (u32 FKS_FLAG_* bits raised by any lane)
    int save2_end;  // a particle's context = [cfg, T + 2 L12) + [G, G + L12) + [target, save2_end): what has to survive between phases
                    // (parked as whole 16-byte units: the third range also carries qr[0], which is dead between phases)
    int stats;    // FKS_NUM_STATS u64 counters of this WARP (not part of a context)
    int total;
    int noise_batch;
};

inline __host__ __device__ WarpLayout make_warp_layout(int L, int J, int D, int stride, int jsm_extra = 0) {
    WarpLayout w;
    int S = stride > D ? stride : D;
    S = (S + 1) & ~1;
    w.S = S;
    w.L12 = 12 * L;
    w.noise_batch = 32 / D < 1 ? 1 : (32 / D > 8 ? 8 : 32 / D);
    int o = 0;
    w.cfg = o; o += 3 * S;
    w.T = o; o += 3 * w.L12;
    w.jsm = w.T + 2 * w.L12;
    w.M = o; o += 16 * J;  // joint matrices, TRANSPOSED and padded: element (row k, column c) of joint j at 16 j + 4 c + k
    w.caps = o; o += 6 * L;
    o += jsm_extra;
    // (D + 1) columns of ld doubles.  The solver's lane 4 g + i reads rows = i (mod 4) of column g: a leading dimension
    // = 4 (mod 16) puts the 16 lanes of a half warp on 16 different bank pairs; take it when it costs at most a quarter
    // of the rows
    // Even in any case: columns are moved between shared and global memory as bulk copies, which start on 16 bytes
    auto pick_ld = [](int doubles, int columns) {
        const int cap = doubles / columns;
        int ld = cap & ~1;
        const int pref = cap - ((cap - 4) & 15);
        if (cap >= 20 && pref >= 20 && pref * 4 >= cap * 3) ld = pref;
        return ld < 0 ? 0 : ld;
    };
    w.jsm_ld = pick_ld(o - w.jsm, D + 1);
    // kinematics<LINKED> runs the T chain (lanes 0..11) and the G chain (lanes 12..23) in the same instructions: their row loads
    // must not share banks, so T starts 2 doubles (mod 16 = one bank cycle) after a multiple of 16 from G
    o += (14 + 16 - (o - w.T) % 16) % 16;
    w.G = o; o += w.L12;
    w.jaxis = o; o += 3 * J;
    w.jorig = o; o += 3 * J;
    o = (o + 1) & ~1;
    w.cand = o; o += 32;
    w.jsm_big_ld = pick_ld(o - w.jsm, D + 1);
    w.target = o; o += S;
    w.scfg = o; o += S;
    w.act = o; o += S;
    w.ru = o; o += S;
    w.du = o; o += S;
    w.raw = o; o += S;
    w.stepv = o; o += S;
    w.tn = o; o += w.noise_batch * S;
    w.vars = o; o += kWarpVarsDoubles + 2 * S;
    w.flags = o; o += 1;
    w.save2_end = o;  // [target, save2_end): third saved range of a context
    w.qr = o; o += S;
    w.stats = o; o += FKS_NUM_STATS;
    w.total = (o + 1) & ~1;
    return w;
}

// ---- global scratch (bytes): a small slot per particle context and a big one per warp -----------------------------------
// the global store of a stacked Jacobian too tall for shared memory (collected in one solve phase, factored in a later
// one -- possibly by another warp) and the self-collision corrections (found by a collision check, consumed by the next
// solve phase)
struct ScratchLayout {
    // per particle CONTEXT (written by the collision check of a round, read by the collect of the following solve, possibly
    // on another warp):
    unsigned long long selfcorr;  // 3*P doubles
    unsigned long long selfwork;  // small dense solve workspace
    unsigned long long keys;      // P packed 64-bit cell keys
    unsigned long long sflag;     // P bytes
    unsigned long long total;     // bytes of a context's slot
    // per WARP (written and consumed inside one solve task):
    unsigned long long jstore;    // offset 0 of the warp's slot: (D+1) * ldj doubles, then P u64 (candidate list of collect_corrections)
    unsigned long long jtotal;    // bytes of a warp's slot
    int ldj;
    int _pad;
};

constexpr int kSelfWorkDoubles = kMaxSelfPartners * 5 + 4 + kMaxSelfPartners * (2 * kMaxSelfPartners) +
                                 kMaxSelfPartners * kMaxSelfPartners + 2 * kMaxSelfPartners;

inline __host__ __device__ ScratchLayout make_scratch_layout(int D, int P) {
    ScratchLayout s;
    s.ldj = ((3 * P + 3) / 4) * 4;
    s._pad = 0;
    unsigned long long o = 0;
    s.selfcorr = o; o += (unsigned long long)3 * P * 8;
    s.selfwork = o; o += (unsigned long long)kSelfWorkDoubles * 8;
    s.keys = o; o += (unsigned long long)P * 8;
    s.sflag = o; o += (((unsigned long long)P + 7) / 8) * 8;
    s.total = ((o + 127) / 128) * 128;
    s.jstore = 0;
    s.jtotal = ((((unsigned long long)(D + 1) * s.ldj * 8 + (unsigned long long)P * 8) + 127) / 128) * 128;
    return s;
}

// one collision point in shared memory: 32 bytes -> two conflict-free 16-byte arrays
struct PointZL {
    double z;
    int link;
    int _pad;
};

// Kernel parameter block.  The kernel copies it (and the robot) into a shared-memory Frame so that every
// device function reads uniform data with LDS at fixed offsets.
struct LaunchArgs {
    DevEnv env;
    DevSolver sp;
    WarpLayout wl;
    ScratchLayout sl;
    const DevRobot* robot;
    const double2* pxy;      // [P] link-relative x, y
    const PointZL* pzl;      // [P] z and the link index
    const double* starts;
    const double* targets;
    const double* tape;
    const unsigned long long* tape_off;
    const unsigned long long* dec_tape;  // decision tape (parity mode, fksgpu.h): records of 2 + D words, or null
    const unsigned long long* dec_off;   // [n + 1] first record of each particle
    char* results;
    unsigned long long* stats;
    unsigned int* counter;
    char* scratch;                   // global scratch, one slot per context of every CTA's pool (self-collision lists)
    char* jscratch;                  // global store of stacked systems too tall for shared memory, one slot per warp
    // Context pool: every CTA keeps `pool` particles in flight for its warps_per_block warps (fks_kernels.cu, simulate_kernel).
    // A context that no warp has loaded lives in ctx_store (ctx_stride bytes each, pool per CTA).
    char* ctx_store;
    int pool, ctx_stride;
    unsigned long long n_particles, n_targets, seed, first_id;
    // sequence calls (fks_forward_simulate_sequence): every particle runs n_legs consecutive legs; leg k of particle i draws
    // Philox noise as particle first_id + k * leg_id_stride + i (leg_id_stride = the whole batch, also for one device's shard)
    unsigned long long leg_id_stride;
    int n_legs;
    int allow_contacts, noise_mode, cfg_stride, rec_stride;
    int P, warps_per_block;
    int pts_off, warps_off;          // byte offsets of the point arrays / the warp blocks in dynamic shared memory
    int sync_off;                    // byte offset of the CTA-level synchronisation word
    int cull_mode;                   // link-level SDF culling: 0 never, 1 always, 2 only while the particle is collision free
    // step trace of a single-particle call (fks_forward_simulate_traced); null on the batch path
    char* trace;                     // records of trace_stride bytes: fks_trace_header + trace_width doubles
    unsigned int* trace_count;       // records produced (may exceed the capacity: the excess is not stored)
    unsigned int trace_capacity;
    int trace_width;                 // doubles per record = max(cfg_stride, D)
};

constexpr int kMaxPool = 64;  // contexts per CTA (two per warp)

struct Frame {
    LaunchArgs a;
    DevRobot rb;
    double gbase[12];  // (1 / sdf_res) * inverse_origin * base: root of the world->voxel chain (linked robots)
    // per disallowed link pair: (half lengths + radii of the two bounding capsules + cell diagonal)^2 -- capsule midpoints
    // further apart than that cannot bring two points of the links into one cell (self-collision broad phase)
    double pair_reach_sq[kMaxPairs];
};

// launch interface implemented in fks_kernels.cu
struct KernelInfo {
    int regs, static_smem, local_bytes, max_blocks_per_sm;
    size_t dyn_smem;
};
int simulate_kernel_info(int kind, size_t dyn_smem, int warps_per_block, KernelInfo* out);
int launch_simulate(int kind, const LaunchArgs& args, int grid, size_t dyn_smem, void* stream,
                    const void* l2_window_base, size_t l2_window_bytes);
// bytes of one particle context in the global context store for this layout
size_t context_bytes(const WarpLayout& wl);
// bytes of CTA-level scheduling state behind the warp blocks in dynamic shared memory: a flag word (16), what every context
// waits for (kMaxPool), which context each warp holds (kMaxPool), then one mbarrier per warp for its bulk loads
constexpr size_t kSyncBytes = 16 + 2 * kMaxPool + 4 * kMaxPool;
constexpr size_t kSyncBarOff = 16 + 2 * kMaxPool;
static_assert(kSyncBarOff % 8 == 0 && kSyncBarOff + 8 * kWarpsPerBlock <= kSyncBytes, "one mbarrier per warp in the sync area");
// fills args.wl / pts_off / warps_off / warps_per_block and returns the dynamic shared memory size, or 0 when a range that the
// kernel moves with bulk copies does not sit on 16-byte boundaries
size_t simulate_smem_plan(LaunchArgs* args, int L, int J, int D, int P, int stride, int warps_per_block, size_t smem_limit);
int launch_check_config(int kind, const LaunchArgs& args, int grid, size_t dyn_smem, void* stream, double inflation_ratio, unsigned char* out);
int launch_qr_solve(double* work, const unsigned long long* offsets, const int* rows, int cols, int n, double* x_out, unsigned* flags_out,
                    void* stream);
int launch_partition(const char* results, size_t rec_stride, int cfg_stride, size_t n, unsigned* block_counts, unsigned long long* totals,
                     unsigned* order, void* stream);
int launch_pairwise_distance(int kind, const DevRobot* robot, const char* results, size_t rec_stride, int cfg_stride, const unsigned* subset,
                             unsigned m, double* out, void* stream);
// fks_end_states_cluster: segments of up to kClusterSmallMax positions keep their distance matrix in shared memory (160^2
// doubles = 200 KiB of the 227 KiB a CTA can have), longer ones in a global slot of large_cap^2 doubles per CTA; the
// per-position state of a segment (20 bytes each) stays in shared memory, which bounds a segment at kClusterMaxSegment.
constexpr unsigned kClusterSmallMax = 160;
constexpr unsigned kClusterMaxSegment = 8192;
struct ClusterLaunch {
    const DevRobot* robot;
    const char* results;
    size_t rec_stride;
    int cfg_stride;
    int complete, separate_contact;
    double threshold;
    const unsigned* order;              // device, or null
    const unsigned long long* offsets;  // device [n_segments + 1]
    unsigned n_segments;
    const unsigned* small_segs;         // device: the non-empty segments of at most kClusterSmallMax positions
    unsigned n_small, small_cap;        // their number and the longest one
    const unsigned* large_segs;         // device: the longer segments
    unsigned n_large, large_cap;
    double* work;                       // large_slots * large_cap^2 doubles
    int large_slots;
    unsigned* labels;                   // [m]
    unsigned* counts;                   // device [n_segments], zeroed: clusters per segment, then their exclusive scan
    unsigned long long* totals;         // device [2]: totals[1] = all clusters
};
// the launches of one call: the two clustering kernels (those with segments), the scan of the counts and the relabel pass
int launch_cluster(int kind, const ClusterLaunch& c, void* stream);
// fks_end_states_groups: clusters of up to kGroupSmallMax members get their minimax representative from one CTA each, larger
// ones (up to kClusterMaxSegment, the largest cluster fks_end_states_cluster makes) from row chunks spread over the grid.
constexpr unsigned kGroupSmallMax = 256;
constexpr unsigned kGroupErrLabel = 1, kGroupErrEmpty = 2, kGroupErrLarge = 4;  // bits of GroupsLaunch::state[1]
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
// the launches of one call, whatever the number and sizes of the clusters: count, scan, scatter, sort + small search,
// large rows, large argmin
constexpr int kGroupLaunches = 6;
int launch_groups(int kind, const GroupsLaunch& g, void* stream);
// fks_end_states_gather_starts: one launch
int launch_gather_starts(const char* results, size_t rec_stride, int cfg_stride, const unsigned* offsets, const unsigned* members,
                         const unsigned* selected, unsigned n_selected, unsigned per_group, const double* group_targets, double* starts,
                         double* targets, void* stream);
int launch_dbg_copy(unsigned long long* out, void* stream);  // developer counters of the FKS_PHASE_TIMERS build
int launch_fp64_peak(double* out, int grid, int iters, void* stream);
int launch_gather(const float* data, unsigned long long n_mask, float* out, int grid, int iters, void* stream);

}  // namespace fksdev

#endif
