// C ABI of libfksgpu.so (include/fksgpu.h): uploads, launch plumbing, statistics.
// The computation itself is in fks_kernels.cu; the environment builder in host/environment_builder.cpp.
// There is NO CPU fallback: every compute entry point fails with FKS_ERR_NO_DEVICE / FKS_ERR_CUDA when
// the device path cannot run.

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only: named host ranges for Nsight Systems / ncu --nvtx, free without a tool attached

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "fks_device_types.h"
#include "fks_internal.h"

using namespace fksdev;

namespace fks_host {
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

// keep the SDF resident in L2 when it fits the persisting carve-out (the current device is env->device)
void finish_env_l2_window(fks_env* env) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, env->device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
        const size_t want = std::min<size_t>(env->sdf_bytes, (size_t)prop.persistingL2CacheMaxSize);
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess && env->sdf_bytes <= (size_t)prop.persistingL2CacheMaxSize)
            env->l2_window_bytes = std::min<size_t>(env->sdf_bytes, (size_t)prop.accessPolicyMaxWindowSize);
    }
    cudaGetLastError();
}
}  // namespace fks_host

namespace {

int fail(int code, const std::string& msg) {
    fks_host::set_last_error(msg);
    return code;
}
int cuda_fail(cudaError_t err, const char* what) {
    return fail(FKS_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(err));
}
#define FKS_CUDA(call)                                        \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) return cuda_fail(_e, #call);   \
    } while (0)

struct DeviceGuard {
    int prev;
    bool ok;
    explicit DeviceGuard(int dev) : prev(-1), ok(false) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

template <typename T>
int upload(T** dst, const T* src, size_t n) {
    *dst = nullptr;
    if (n == 0) n = 1;
    FKS_CUDA(cudaMalloc((void**)dst, n * sizeof(T)));
    if (src) FKS_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return FKS_OK;
}

template <typename T>
int ensure(T** ptr, size_t* cap, size_t need) {
    if (need <= *cap) return FKS_OK;
    cudaFree(*ptr);
    *ptr = nullptr;
    *cap = 0;
    const size_t want = need + need / 4;
    FKS_CUDA(cudaMalloc((void**)ptr, want * sizeof(T)));
    *cap = want;
    return FKS_OK;
}

}  // namespace

struct fks_robot {
    int device;
    DevRobot host;
    DevRobot* d_robot;
    double2* d_pxy;
    PointZL* d_pzl;
    int stride;
};

struct fks_sim {
    int device;
    const fks_env* env;
    const fks_robot* robot;
    DevSolver sp;
    uint64_t seed;
    int32_t debug_level;
    cudaStream_t stream;
    int grid_max, num_sms;
    size_t dyn_smem;
    KernelInfo kinfo;
    LaunchArgs plan;  // layouts and shared-memory offsets (simulate_smem_plan)
    char* d_scratch;
    char* d_jscratch = nullptr;
    unsigned long long* d_stats;
    unsigned int* d_counter;
    // staging for the host-buffer entry point (grown on demand)
    double *d_starts, *d_targets, *d_tape;
    unsigned long long *d_tape_off, *d_dec, *d_dec_off;
    char* d_results;
    size_t cap_starts, cap_targets, cap_tape, cap_tape_off, cap_results, cap_dec, cap_dec_off;
    unsigned int* d_part = nullptr;  // fks_end_states_partition: totals + per-block counts
    size_t cap_part = 0;
    // fks_end_states_cluster: [offsets | totals | counts, segment lists] and the distance matrices of the large segments
    unsigned long long* d_clu = nullptr;
    size_t cap_clu = 0;
    double* d_clu_mat = nullptr;
    size_t cap_clu_mat = 0;
    // fks_end_states_groups: [totals (2) | row maxima (m doubles) | cursors, state as u32]
    unsigned long long* d_grp = nullptr;
    size_t cap_grp = 0;
    // fks_end_states_gather_starts: the selected group ids, and when the last launch that reads them is done
    unsigned* d_sel = nullptr;
    size_t cap_sel = 0;
    cudaEvent_t sel_read = nullptr;
    bool has_sel = false;
    unsigned long long* d_trace_buf = nullptr;  // fks_forward_simulate_traced: [counter word | records], grown on demand
    size_t cap_trace_buf = 0;
    size_t smem_limit;
    // context pool of the simulate kernel: global store of parked particle contexts and their scratch slots
    char* d_ctx_store;
    int pool;
    int pool_eighths = 16;
    // device time of the simulate kernel of the last batch call (fks_sim_kernel_times), recorded only after
    // fks_sim_enable_kernel_timing
    cudaEvent_t tev[2];
    int timing, timed_kernels;
    // launches of one simulator share its particle counter, scratch slots and statistics: a launch on another stream waits
    // for the previous one (fks_forward_simulate_device takes the caller's stream)
    cudaEvent_t last_done;
    cudaStream_t last_stream;
    bool has_last;
    uint64_t launches;
    std::string info;
    // set by fks_forward_simulate_traced around its launch, null otherwise
    char* d_trace;
    unsigned int* d_trace_count;
    unsigned int trace_capacity;
};

extern "C" {

namespace {
struct NvtxRange {  // one named range per C-ABI call and per stage inside it
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};
}  // namespace

int fks_abi_version(void) { return FKS_ABI_VERSION; }

const char* fks_last_error_string(void) { return fks_host::g_last_error.c_str(); }

int fks_device_count(int* count) {
    if (!count) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_device_count: null argument");
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess) {
        *count = 0;
        return fail(FKS_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(err));
    }
    *count = n;
    return FKS_OK;
}

void fks_default_solver_params(fks_solver_params* out) {
    if (!out) return;
    out->forward_simulation_time = 1.0;
    out->simulation_shortcut_distance = 0.0;
    out->environment_collision_check_tolerance = 0.001;
    out->resolve_correction_step_scaling_decay_rate = 0.5;
    out->resolve_correction_initial_step_size = 1.0;
    out->resolve_correction_min_step_scaling = 0.03125;
    out->max_resolver_iterations = 25;
    out->resolve_correction_step_scaling_decay_iterations = 5;
    out->failed_resolves_end_motion = 1;
    out->_pad = 0;
}

// ---------------------------------------------------------------------------------------------
// environment
// ---------------------------------------------------------------------------------------------
int fks_env_create(int device, const fks_env_desc* desc, fks_env** out) {
    if (!desc || !out) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: null argument");
    *out = nullptr;
    if (!desc->sdf || desc->nx <= 0 || desc->ny <= 0 || desc->nz <= 0 || desc->nx > 65535 || desc->ny > 65535 ||
        desc->nz > 65535 || (double)desc->nx * (double)desc->ny * (double)desc->nz >= 2147483648.0 || !(desc->sdf_resolution > 0.0) || !(desc->map_resolution > 0.0))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: bad grid description");
    if (desc->n_normal_cells < 0 || (desc->n_normal_cells > 0 && (!desc->normal_cell_index || !desc->normal_cell_start || !desc->normal_entries)))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: bad surface-normal table");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "fks_env_create: no CUDA device");
    if (device < 0 || device >= ndev) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: bad device index");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_env_create: cudaSetDevice failed");

    fks_env* env = new (std::nothrow) fks_env();
    if (!env) return fail(FKS_ERR_OUT_OF_MEMORY, "fks_env_create: out of host memory");
    std::memset(env, 0, sizeof(*env));
    env->device = device;
    const size_t ncells = (size_t)desc->nx * (size_t)desc->ny * (size_t)desc->nz;
    env->sdf_bytes = ncells * sizeof(float);
    int rc = upload(&env->d_sdf, desc->sdf, ncells);
    if (rc != FKS_OK) { fks_env_destroy(env); return rc; }

    // surface normals: open-addressing hash, load factor <= 0.5, linear probing
    const size_t ncell_n = (size_t)desc->n_normal_cells;
    size_t cap = 2;
    while (cap < 2 * ncell_n) cap <<= 1;
    std::vector<unsigned long long> keys(2 * cap, 0ull);  // {key, start | count << 32} pairs
    const size_t nentries = ncell_n ? (size_t)desc->normal_cell_start[ncell_n] : 0;
    for (size_t i = 0; i < ncell_n; i++) {
        const int64_t li = desc->normal_cell_index[i];
        if (li < 0 || (size_t)li >= ncells || desc->normal_cell_start[i + 1] < desc->normal_cell_start[i]) {
            fks_env_destroy(env);
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: surface-normal cell out of range");
        }
        size_t h = (size_t)(normal_hash((unsigned long long)li) & (cap - 1));
        while (keys[2 * h] != 0ull) {
            if (keys[2 * h] == (unsigned long long)li + 1ull) {
                fks_env_destroy(env);
                return fail(FKS_ERR_INVALID_ARGUMENT, "fks_env_create: duplicate surface-normal cell");
            }
            h = (h + 1) & (cap - 1);
        }
        keys[2 * h] = (unsigned long long)li + 1ull;
        keys[2 * h + 1] = (unsigned long long)desc->normal_cell_start[i] |
                          ((unsigned long long)(desc->normal_cell_start[i + 1] - desc->normal_cell_start[i]) << 32);
    }
    std::vector<double> entries(std::max<size_t>(nentries, 1) * 6, 0.0);
    for (size_t en = 0; en < nentries; en++) {
        const double* src = desc->normal_entries + 7 * en;  // entry direction xyzw (w == 0), normal xyz
        entries[6 * en + 0] = src[0];
        entries[6 * en + 1] = src[1];
        entries[6 * en + 2] = src[2];
        entries[6 * en + 3] = src[4];
        entries[6 * en + 4] = src[5];
        entries[6 * en + 5] = src[6];
    }
    rc = upload(&env->d_keys, keys.data(), 2 * cap);
    if (rc == FKS_OK) rc = upload(&env->d_entries, entries.data(), entries.size());
    // ordered view kept for fks_env_download
    static_assert(sizeof(long long) == sizeof(int64_t), "cell index width");
    const uint32_t zero_start = 0;
    if (rc == FKS_OK) rc = upload(&env->d_cell_index, reinterpret_cast<const long long*>(desc->normal_cell_index), ncell_n);
    if (rc == FKS_OK) rc = upload(&env->d_cell_start, ncell_n ? desc->normal_cell_start : &zero_start, ncell_n + 1);
    env->n_normal_cells = (long long)ncell_n;
    env->n_entries = nentries;
    if (rc != FKS_OK) { fks_env_destroy(env); return rc; }

    DevEnv& d = env->dev;
    std::memcpy(d.origin, desc->origin, sizeof(d.origin));
    std::memcpy(d.inv_origin, desc->inverse_origin, sizeof(d.inv_origin));
    d.map_res = desc->map_resolution;
    d.sdf_res = desc->sdf_resolution;
    d.inv_sdf_res = 1.0 / desc->sdf_resolution;
    d.inv_twice_res = 1.0 / (2.0 * desc->sdf_resolution);
    d.nx = (int)desc->nx;
    d.ny = (int)desc->ny;
    d.nz = (int)desc->nz;
    d.oob = desc->oob_value;
    // Link-level culling (fks_kernels.cu: active_links) relies on the SDF being a distance field: neighbouring cells
    // differ by at most one cell size inside a sign region and by at most two across the surface.  Verified here;
    // an SDF that is not (hand-made, inflated, ...) simply runs without culling.
    {
        const int64_t nx = desc->nx, ny = desc->ny, nz = desc->nz;
        const double lim1 = desc->sdf_resolution * (1.0 + 1e-4), lim2 = 2.0 * lim1;
        bool ok = std::isinf(desc->oob_value) && desc->oob_value > 0.0f;
        const float* f = desc->sdf;
#pragma omp parallel for schedule(static) reduction(&& : ok)
        for (int64_t x = 0; x < nx; x++)
            for (int64_t y = 0; y < ny && ok; y++)
                for (int64_t z = 0; z < nz; z++) {
                    const size_t i = (size_t)((x * ny + y) * nz + z);
                    const double v = (double)f[i];
                    const size_t nb[3] = {x + 1 < nx ? i + (size_t)(ny * nz) : i, y + 1 < ny ? i + (size_t)nz : i, z + 1 < nz ? i + 1 : i};
                    for (int k = 0; k < 3; k++) {
                        const double w = (double)f[nb[k]];
                        const double lim = ((v < 0.0) != (w < 0.0)) ? lim2 : lim1;
                        if (!(std::fabs(v - w) <= lim)) ok = false;
                    }
                }
        d.cull = ok ? 1 : 0;
    }
    d.sdf = env->d_sdf;
    d.nh_keys = env->d_keys;
    d.nh_mask = (unsigned long long)(cap - 1);
    d.normal_entries = env->d_entries;

    fks_host::finish_env_l2_window(env);
    *out = env;
    return FKS_OK;
}

void fks_env_destroy(fks_env* env) {
    if (!env) return;
    DeviceGuard guard(env->device);
    cudaFree(env->d_sdf);
    cudaFree(env->d_keys);
    cudaFree(env->d_entries);
    cudaFree(env->d_cell_index);
    cudaFree(env->d_cell_start);
    cudaFree(env->d_occupancy);
    delete env;
}

// ---------------------------------------------------------------------------------------------
// robot
// ---------------------------------------------------------------------------------------------
int fks_robot_create(int device, const fks_robot_desc* r, fks_robot** out) {
    if (!r || !out) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: null argument");
    *out = nullptr;
    if (r->kind != FKS_ROBOT_SE2 && r->kind != FKS_ROBOT_SE3 && r->kind != FKS_ROBOT_LINKED)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: unknown robot kind");
    if (r->n_points <= 0 || r->n_points > (1 << 20) || !r->points_xyz || !r->point_link || !r->axes)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: bad point/axis arrays");
    const int L = r->n_links, J = r->n_joints, D = r->n_dof;
    if (L < 1 || L > kMaxLinks || J < 0 || J > kMaxJoints || D < 1 || D > kMaxDof - 1)  // the solver keeps D + 1 <= 16 columns
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: link/joint/dof count out of range");
    if (r->kind == FKS_ROBOT_SE2 && (L != 1 || D != 3)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: SE2 needs 1 link, 3 dof");
    if (r->kind == FKS_ROBOT_SE3 && (L != 1 || D != 6)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: SE3 needs 1 link, 6 dof");
    if (r->kind == FKS_ROBOT_LINKED && (J < 1 || !r->joints)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: linked robot needs joints");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "fks_robot_create: no CUDA device");
    if (device < 0 || device >= ndev) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: bad device index");

    fks_robot* rob = new (std::nothrow) fks_robot();
    if (!rob) return fail(FKS_ERR_OUT_OF_MEMORY, "fks_robot_create: out of host memory");
    std::memset(rob, 0, sizeof(*rob));
    rob->device = device;
    DevRobot& h = rob->host;
    h.kind = r->kind;
    h.L = L;
    h.J = (r->kind == FKS_ROBOT_LINKED) ? J : 0;
    h.D = D;
    h.P = (int)r->n_points;
    std::memcpy(h.base, r->base_transform, sizeof(h.base));
    h.pos_w = r->position_distance_weight;
    h.rot_w = r->rotation_distance_weight;
    for (int i = 0; i < D; i++) {
        const fks_axis_params& a = r->axes[i];
        DevAxis& d = h.axes[i];
        d.kp = std::fabs(a.kp);  // pid.hpp:104-113
        d.ki = std::fabs(a.ki);
        d.kd = std::fabs(a.kd);
        d.iclamp = std::fabs(a.integral_clamp);
        d.vlim = std::fabs(a.velocity_limit);          // unc.hpp:61
        d.pnoise = std::fabs(a.proportional_noise);
        d.mnoise = std::fabs(a.minimum_noise);
        d.sigma = a.noise_sigma;
    }
    // points: link-major, point-minor
    std::vector<double> px((size_t)h.P), py((size_t)h.P), pz((size_t)h.P);
    std::vector<int> plink((size_t)h.P);
    for (int l = 0; l <= L; l++) h.link_begin[l] = 0;
    for (int i = 0; i < h.P; i++) {
        const int l = r->point_link[i];
        if (l < 0 || l >= L || (i > 0 && l < r->point_link[i - 1])) {
            delete rob;
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: point_link must be non-decreasing and < n_links");
        }
        px[(size_t)i] = r->points_xyz[3 * i];
        py[(size_t)i] = r->points_xyz[3 * i + 1];
        pz[(size_t)i] = r->points_xyz[3 * i + 2];
        plink[(size_t)i] = l;
        h.link_begin[l + 1]++;
    }
    for (int l = 0; l < L; l++) h.link_begin[l + 1] += h.link_begin[l];
    // joints (kinematic order: a joint's parent link must already have a transform)
    int link_parent_joint[kMaxLinks];
    for (int l = 0; l < L; l++) link_parent_joint[l] = -1;
    int active = 0;
    for (int j = 0; j < h.J; j++) {
        const fks_joint_desc& jd = r->joints[j];
        if (jd.parent_link < 0 || jd.parent_link >= L || jd.child_link <= 0 || jd.child_link >= L || jd.type < 0 || jd.type > 3 ||
            (jd.parent_link != 0 && link_parent_joint[jd.parent_link] < 0) || link_parent_joint[jd.child_link] >= 0) {
            delete rob;
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: joints must form a tree rooted at link 0, in kinematic order");
        }
        DevJoint& d = h.joints[j];
        d.parent = jd.parent_link;
        d.child = jd.child_link;
        d.type = jd.type;
        d.active = (jd.type == FKS_JOINT_FIXED) ? -1 : active++;
        std::memcpy(d.T, jd.transform, sizeof(d.T));
        std::memcpy(d.axis, jd.axis, sizeof(d.axis));
        d.lo = jd.lower_limit;
        d.hi = jd.upper_limit;
        d.weight = jd.distance_weight;
        if (d.active >= 0 && d.active < kMaxDof) h.active_joint[d.active] = j;
        link_parent_joint[jd.child_link] = j;
    }
    for (int l = 1; l < L; l++)
        if (link_parent_joint[l] < 0) {  // a link no joint leads to would keep an uninitialised transform on the device
            delete rob;
            return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: every link other than link 0 needs a parent joint");
        }
    if (r->kind == FKS_ROBOT_LINKED && active != D) {  // tnuva.hpp:503-516 throws std::invalid_argument
        delete rob;
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: number of axis parameter sets != number of active joints");
    }
    for (int l = 0; l < L; l++) {
        unsigned anc = 0u;
        int j = link_parent_joint[l];
        while (j >= 0) {
            anc |= 1u << j;
            j = link_parent_joint[h.joints[j].parent];
        }
        h.link_ancestors[l] = anc;
    }
    // self-collision table
    h.n_pairs = 0;
    for (int a = 0; a < L; a++) h.disallowed[a] = 0u;
    if (L > 1 && r->allowed_self_collision) {
        for (int a = 0; a < L; a++)
            for (int b = a + 1; b < L; b++) {
                const bool ab = r->allowed_self_collision[a * L + b] != 0, ba = r->allowed_self_collision[b * L + a] != 0;
                if (ab != ba) {
                    delete rob;
                    return fail(FKS_ERR_INVALID_ARGUMENT, "fks_robot_create: allowed_self_collision must be symmetric");
                }
                if (!ab) {
                    h.disallowed[a] |= 1u << b;
                    h.disallowed[b] |= 1u << a;
                    h.pair_a[h.n_pairs] = (unsigned char)a;
                    h.pair_b[h.n_pairs] = (unsigned char)b;
                    h.n_pairs++;
                }
            }
    }
    // bounding spheres (slightly inflated) and cumulative masses (spcs.hpp:1244-1255)
    double acc = 0.0;
    for (int l = L - 1; l >= 0; l--) {
        const double m = (double)(h.link_begin[l + 1] - h.link_begin[l]);
        h.link_mass[l] = m + acc;
        acc += m;
    }
    for (int l = 0; l < L; l++) {
        // bounding capsule: segment along the longest bounding-box axis through the box centre
        double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
        for (int p = h.link_begin[l]; p < h.link_begin[l + 1]; p++) {
            const double v[3] = {px[(size_t)p], py[(size_t)p], pz[(size_t)p]};
            for (int k = 0; k < 3; k++) {
                if (p == h.link_begin[l] || v[k] < lo[k]) lo[k] = v[k];
                if (p == h.link_begin[l] || v[k] > hi[k]) hi[k] = v[k];
            }
        }
        int ax = 0;
        for (int k = 1; k < 3; k++)
            if (hi[k] - lo[k] > hi[ax] - lo[ax]) ax = k;
        for (int k = 0; k < 3; k++) {
            const double mid = 0.5 * (lo[k] + hi[k]);
            h.cap_p0[l][k] = (k == ax) ? lo[k] : mid;
            h.cap_p1[l][k] = (k == ax) ? hi[k] : mid;
        }
        double rad = 0.0;
        for (int p = h.link_begin[l]; p < h.link_begin[l + 1]; p++) {
            const double v[3] = {px[(size_t)p], py[(size_t)p], pz[(size_t)p]};
            double d2 = 0.0;
            for (int k = 0; k < 3; k++) {
                const double c = (k == ax) ? std::min(std::max(v[k], lo[k]), hi[k]) : h.cap_p0[l][k];
                d2 += (v[k] - c) * (v[k] - c);
            }
            rad = std::max(rad, std::sqrt(d2));
        }
        h.cap_radius[l] = rad * (1.0 + 1e-9) + 1e-12;
        double srad = 0.0;
        for (int k = 0; k < 3; k++) h.sph_center[l][k] = 0.5 * (lo[k] + hi[k]);
        for (int p = h.link_begin[l]; p < h.link_begin[l + 1]; p++) {
            const double dx = px[(size_t)p] - h.sph_center[l][0], dy = py[(size_t)p] - h.sph_center[l][1], dz = pz[(size_t)p] - h.sph_center[l][2];
            srad = std::max(srad, std::sqrt(dx * dx + dy * dy + dz * dz));
        }
        h.sph_radius[l] = srad * (1.0 + 1e-9) + 1e-12;
    }
    rob->stride = (r->kind == FKS_ROBOT_SE2) ? 3 : (r->kind == FKS_ROBOT_SE3 ? 12 : D);

    DeviceGuard guard(device);
    if (!guard.ok) { delete rob; return fail(FKS_ERR_CUDA, "fks_robot_create: cudaSetDevice failed"); }
    std::vector<double2> pxy((size_t)h.P);
    std::vector<PointZL> pzl((size_t)h.P);
    for (int i = 0; i < h.P; i++) {
        pxy[(size_t)i] = make_double2(px[(size_t)i], py[(size_t)i]);
        pzl[(size_t)i].z = pz[(size_t)i];
        pzl[(size_t)i].link = plink[(size_t)i];
        pzl[(size_t)i]._pad = 0;
    }
    // Joint matrix as a function of the joint value (linked robots): M_j(q) = J_t R(q) with Rodrigues' form
    // R = I + sin q K + (1 - cos q) K^2, K = [axis]x  ->  M_j = J_t + sin q (J_t K) + (1 - cos q) (J_t K^2); prismatic:
    // M_j = J_t + q [0 | J_t axis].  The two constant 3x4 matrices per joint are formed here once (algebraically the same
    // entries as Eigen's AngleAxis -> quaternion -> matrix path the reference takes, for any axis length).
    for (int j = 0; j < h.J; j++) {
        DevJoint& d = h.joints[j];
        const double ax = d.axis[0], ay = d.axis[1], az = d.axis[2];
        double* C1 = d.C1;
        double* C2 = d.C2;
        for (int i = 0; i < 12; i++) C1[i] = C2[i] = 0.0;
        if (d.active < 0) continue;
        if (d.type == FKS_JOINT_PRISMATIC) {
            for (int r = 0; r < 3; r++) C1[4 * r + 3] = d.T[4 * r + 0] * ax + d.T[4 * r + 1] * ay + d.T[4 * r + 2] * az;
        } else {
            const double K[9] = {0.0, -az, ay, az, 0.0, -ax, -ay, ax, 0.0};
            double K2[9];
            for (int r = 0; r < 3; r++)
                for (int c = 0; c < 3; c++) K2[3 * r + c] = K[3 * r + 0] * K[c] + K[3 * r + 1] * K[3 + c] + K[3 * r + 2] * K[6 + c];
            for (int r = 0; r < 3; r++)
                for (int c = 0; c < 3; c++) {
                    C1[4 * r + c] = d.T[4 * r + 0] * K[c] + d.T[4 * r + 1] * K[3 + c] + d.T[4 * r + 2] * K[6 + c];
                    C2[4 * r + c] = d.T[4 * r + 0] * K2[c] + d.T[4 * r + 1] * K2[3 + c] + d.T[4 * r + 2] * K2[6 + c];
                }
        }
    }
    static_assert(kMaxLinks <= 16 && kMaxJoints <= 16, "joint_parents / joint_children pack one nibble per joint");
    h.joint_parents = h.joint_children = 0ull;
    for (int j = 0; j < h.J; j++) {
        h.joint_parents |= (unsigned long long)h.joints[j].parent << (4 * j);
        h.joint_children |= (unsigned long long)h.joints[j].child << (4 * j);
    }
    int rc = upload(&rob->d_robot, &rob->host, 1);
    if (rc == FKS_OK) rc = upload(&rob->d_pxy, pxy.data(), pxy.size());
    if (rc == FKS_OK) rc = upload(&rob->d_pzl, pzl.data(), pzl.size());
    if (rc != FKS_OK) { fks_robot_destroy(rob); return rc; }
    *out = rob;
    return FKS_OK;
}

void fks_robot_destroy(fks_robot* robot) {
    if (!robot) return;
    DeviceGuard guard(robot->device);
    cudaFree(robot->d_robot);
    cudaFree(robot->d_pxy);
    cudaFree(robot->d_pzl);
    delete robot;
}

int fks_robot_config_stride(const fks_robot* robot) { return robot ? robot->stride : 0; }

// ---------------------------------------------------------------------------------------------
// simulator
// ---------------------------------------------------------------------------------------------
int fks_sim_create(const fks_env* env, const fks_robot* robot, const fks_solver_params* params,
                   double simulation_controller_frequency, uint64_t prng_seed, int32_t debug_level, fks_sim** out) {
    if (!env || !robot || !params || !out) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_create: null argument");
    *out = nullptr;
    if (env->device != robot->device) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_create: environment and robot live on different devices");
    if (simulation_controller_frequency == 0.0 || std::isnan(simulation_controller_frequency))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_create: controller frequency must be non-zero");
    if (params->resolve_correction_step_scaling_decay_iterations == 0)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_create: decay iterations must be > 0");
    DeviceGuard guard(env->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_sim_create: cudaSetDevice failed");
    fks_sim* s = new (std::nothrow) fks_sim();
    if (!s) return fail(FKS_ERR_OUT_OF_MEMORY, "fks_sim_create: out of host memory");
    s->device = env->device;
    s->env = env;
    s->robot = robot;
    s->seed = prng_seed;
    s->debug_level = debug_level;
    s->stream = nullptr;
    s->d_scratch = nullptr;
    s->d_stats = nullptr;
    s->d_counter = nullptr;
    s->d_starts = s->d_targets = s->d_tape = nullptr;
    s->d_tape_off = s->d_dec = s->d_dec_off = nullptr;
    s->d_results = nullptr;
    s->cap_starts = s->cap_targets = s->cap_tape = s->cap_tape_off = s->cap_results = s->cap_dec = s->cap_dec_off = 0;
    s->d_ctx_store = nullptr;
    s->pool = 0;
    for (int i = 0; i < 2; i++) s->tev[i] = nullptr;
    s->timing = 0;
    s->timed_kernels = 0;
    s->last_done = nullptr;
    s->last_stream = nullptr;
    s->has_last = false;
    {
        int lim = 0;
        if (cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, env->device) != cudaSuccess || lim <= 0) lim = 48 * 1024;
        s->smem_limit = (size_t)lim;
    }
    s->launches = 0;
    s->d_trace = nullptr;
    s->d_trace_count = nullptr;
    s->trace_capacity = 0;
    const double freq = std::fabs(simulation_controller_frequency);  // spcs.hpp:426
    s->sp.interval = 1.0 / simulation_controller_frequency;          // spcs.hpp:427 (sign kept)
    s->sp.shortcut_distance = params->simulation_shortcut_distance;
    s->sp.check_tolerance = params->environment_collision_check_tolerance;
    s->sp.decay_rate = params->resolve_correction_step_scaling_decay_rate;
    s->sp.initial_step = params->resolve_correction_initial_step_size;
    s->sp.min_scaling = params->resolve_correction_min_step_scaling;
    s->sp.max_iters = params->max_resolver_iterations;
    s->sp.decay_iters = params->resolve_correction_step_scaling_decay_iterations;
    s->sp.n_steps = std::max((uint32_t)(params->forward_simulation_time * freq), 1u);  // spcs.hpp:856
    s->sp.failed_ends_motion = params->failed_resolves_end_motion ? 1 : 0;

    const DevRobot& h = robot->host;
    std::memset(&s->plan, 0, sizeof(s->plan));
    int wpb = kWarpsPerBlock;
    if (const char* ev = std::getenv("FKS_WARPS_PER_BLOCK")) {  // developer knob: warps per lock-step CTA, 1..kWarpsPerBlock
        const int v = std::atoi(ev);
        if (v >= 1 && v <= kWarpsPerBlock) wpb = v;
    }
    // largest lock-step CTA whose shared memory fits the SM (robots with many links / points get fewer warps per CTA)
    int rc = 0;
    for (;; wpb = (wpb > 4) ? wpb - 4 : wpb - 1) {
        s->dyn_smem = simulate_smem_plan(&s->plan, h.L, h.J, h.D, h.P, robot->stride, wpb, s->smem_limit);
        if (s->dyn_smem == 0) break;
        s->kinfo.max_blocks_per_sm = 0;
        rc = simulate_kernel_info(h.kind, s->dyn_smem, wpb, &s->kinfo);
        if ((rc == 0 && s->kinfo.max_blocks_per_sm >= 1) || wpb <= 1) break;
        cudaGetLastError();
    }
    s->plan.cull_mode = 1;
    s->plan.trace = nullptr;
    s->plan.trace_count = nullptr;
    s->plan.trace_capacity = 0;
    s->plan.trace_width = 0;
    if (const char* ev = std::getenv("FKS_CULL")) s->plan.cull_mode = std::atoi(ev);  // developer knob
    if (s->dyn_smem == 0) { delete s; return fail(FKS_ERR_UNSUPPORTED, "fks_sim_create: warp block layout not 16-byte aligned for bulk copies"); }
    if (rc != 0) { delete s; return cuda_fail((cudaError_t)rc, "fks_sim_create: kernel attributes"); }
    if (s->kinfo.max_blocks_per_sm < 1) { delete s; return fail(FKS_ERR_UNSUPPORTED, "fks_sim_create: robot does not fit one CTA's shared memory"); }
    cudaDeviceProp prop;
    cudaError_t err = cudaGetDeviceProperties(&prop, s->device);
    if (err != cudaSuccess) { delete s; return cuda_fail(err, "cudaGetDeviceProperties"); }
    s->grid_max = prop.multiProcessorCount * s->kinfo.max_blocks_per_sm;
    s->num_sms = prop.multiProcessorCount;
    s->pool_eighths = 16;  // contexts per warp, in eighths (2 per warp)
    if (const char* ev = std::getenv("FKS_POOL_EIGHTHS")) s->pool_eighths = std::max(8, std::atoi(ev));  // developer knob
    s->pool = std::min((s->pool_eighths * wpb + 7) / 8, kMaxPool);
    const size_t scratch_bytes = (size_t)s->grid_max * s->pool * s->plan.sl.total;  // one small slot per context
    const size_t jscratch_bytes = (size_t)s->grid_max * wpb * s->plan.sl.jtotal;    // one tall-system slot per warp
    s->plan.pool = s->pool;
    s->plan.ctx_stride = (int)context_bytes(s->plan.wl);
    const size_t ctx_bytes = (size_t)s->grid_max * s->pool * (size_t)s->plan.ctx_stride;

    if ((err = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (err = cudaEventCreateWithFlags(&s->last_done, cudaEventDisableTiming)) != cudaSuccess ||
        (err = cudaMalloc((void**)&s->d_scratch, scratch_bytes)) != cudaSuccess ||
        (err = cudaMalloc((void**)&s->d_jscratch, jscratch_bytes)) != cudaSuccess ||
        (err = cudaMalloc((void**)&s->d_ctx_store, ctx_bytes)) != cudaSuccess ||
        (err = cudaMalloc((void**)&s->d_stats, 128 * sizeof(unsigned long long))) != cudaSuccess ||
        (err = cudaMalloc((void**)&s->d_counter, 4 * sizeof(unsigned int))) != cudaSuccess ||
        (err = cudaMemset(s->d_stats, 0, 128 * sizeof(unsigned long long))) != cudaSuccess) {
        fks_sim_destroy(s);
        return cuda_fail(err, "fks_sim_create: allocation");
    }
    char buf[512];
    std::snprintf(buf, sizeof(buf),
                  "simulate_kernel<kind=%d>: %d regs/thread, %zu B dynamic smem/CTA, %d B local/thread, %d threads/CTA, "
                  "%d CTAs/SM x %d SMs (persistent grid %d), scratch %llu B/warp, L2 window %zu B",
                  h.kind, s->kinfo.regs, s->dyn_smem, s->kinfo.local_bytes, 32 * wpb, s->kinfo.max_blocks_per_sm,
                  prop.multiProcessorCount, s->grid_max, (unsigned long long)s->plan.sl.jtotal, env->l2_window_bytes);
    s->info = buf;
    *out = s;
    return FKS_OK;
}

void fks_sim_destroy(fks_sim* s) {
    if (!s) return;
    DeviceGuard guard(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->has_last) cudaEventSynchronize(s->last_done);
    cudaFree(s->d_scratch);
    cudaFree(s->d_jscratch);
    cudaFree(s->d_stats);
    cudaFree(s->d_counter);
    cudaFree(s->d_starts);
    cudaFree(s->d_targets);
    cudaFree(s->d_tape);
    cudaFree(s->d_tape_off);
    cudaFree(s->d_dec);
    cudaFree(s->d_dec_off);
    cudaFree(s->d_trace_buf);
    cudaFree(s->d_part);
    cudaFree(s->d_clu);
    cudaFree(s->d_clu_mat);
    if (s->has_sel) cudaEventSynchronize(s->sel_read);
    cudaFree(s->d_grp);
    cudaFree(s->d_sel);
    if (s->sel_read) cudaEventDestroy(s->sel_read);
    cudaFree(s->d_ctx_store);
    cudaFree(s->d_results);
    if (s->last_done) cudaEventDestroy(s->last_done);
    for (int i = 0; i < 2; i++)
        if (s->tev[i]) cudaEventDestroy(s->tev[i]);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

size_t fks_sim_result_stride(const fks_sim* sim) {
    return sim ? (size_t)sim->robot->stride * 8 + sizeof(fks_result_tail) : 0;
}

// n_legs consecutive legs per particle (1: a single ForwardSimulateRobots call); d_targets and d_results are leg-major
static int simulate_on_stream(fks_sim* s, const double* d_starts, const double* d_targets, size_t n, size_t n_targets, size_t n_legs,
                              uint64_t leg_id_stride, int allow_contacts, int noise_mode, const double* d_tape, const uint64_t* d_tape_off,
                              const uint64_t* d_dec, const uint64_t* d_dec_off,
                              uint64_t first_particle_id, void* d_results, cudaStream_t stream) {
    if (n == 0) return FKS_OK;
    if (n > 0xFFFFFF00ull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: too many particles for one call");
    LaunchArgs a = s->plan;
    a.env = s->env->dev;
    a.sp = s->sp;
    a.robot = s->robot->d_robot;
    a.pxy = s->robot->d_pxy;
    a.pzl = s->robot->d_pzl;
    a.starts = d_starts;
    a.targets = d_targets;
    a.tape = d_tape;
    a.tape_off = (const unsigned long long*)d_tape_off;
    a.dec_tape = (noise_mode == FKS_NOISE_INJECTED) ? (const unsigned long long*)d_dec : nullptr;
    a.dec_off = (const unsigned long long*)d_dec_off;
    a.results = (char*)d_results;
    a.stats = s->d_stats;
    a.counter = s->d_counter;
    a.scratch = s->d_scratch;
    a.jscratch = s->d_jscratch;
    a.n_particles = n;
    a.n_targets = n_targets;
    a.seed = s->seed;
    a.first_id = first_particle_id;
    a.leg_id_stride = leg_id_stride;
    a.n_legs = (int)n_legs;
    a.allow_contacts = allow_contacts ? 1 : 0;
    a.noise_mode = noise_mode;
    a.cfg_stride = s->robot->stride;
    a.rec_stride = (int)fks_sim_result_stride(s);
    a.trace = s->d_trace;
    a.trace_count = s->d_trace_count;
    a.trace_capacity = s->trace_capacity;
    a.trace_width = std::max(s->robot->stride, s->robot->host.D);
    // small batches: fewer warps per CTA so that the particles spread over all SMs (one warp per particle)
    const size_t per_sm = (n + (size_t)s->num_sms - 1) / (size_t)s->num_sms;
    const int wpb = (int)std::max<size_t>(1, std::min<size_t>((size_t)s->plan.warps_per_block, per_sm));
    a.warps_per_block = wpb;
    a.sync_off = a.warps_off + wpb * a.wl.total * 8;
    const size_t dyn_smem = (size_t)a.sync_off + kSyncBytes;
    const size_t blocks_needed = (n + (size_t)wpb - 1) / (size_t)wpb;
    const int grid = (int)std::min<size_t>((size_t)s->grid_max, blocks_needed);
    if (s->has_last && stream != s->last_stream) FKS_CUDA(cudaStreamWaitEvent(stream, s->last_done, 0));
    FKS_CUDA(cudaMemsetAsync(s->d_counter, 0, 4 * sizeof(unsigned int), stream));
    const void* l2_base = s->env->l2_window_bytes ? s->env->d_sdf : nullptr;
    a.ctx_store = s->d_ctx_store;
    a.pool = std::max(wpb, std::min((s->pool_eighths * wpb + 7) / 8, s->pool));
    if (s->timing) FKS_CUDA(cudaEventRecord(s->tev[0], stream));
    const int rc = launch_simulate(s->robot->host.kind, a, grid, dyn_smem, stream, l2_base, s->env->l2_window_bytes);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "simulate kernel launch");
    if (s->timing) FKS_CUDA(cudaEventRecord(s->tev[1], stream));
    s->timed_kernels = s->timing ? 1 : 0;
    FKS_CUDA(cudaEventRecord(s->last_done, stream));
    s->last_stream = stream;
    s->has_last = true;
    s->launches++;
    return FKS_OK;
}

static int check_batch(const fks_sim* sim, const void* starts, const void* targets, size_t n, size_t n_targets, int noise_mode,
                       const void* tape_draws, const void* tape_off, const void* results) {
    if (!sim) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: null simulator");
    if (n == 0) return FKS_OK;
    if (!starts || !targets || !results) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: null buffer");
    // assert((target_positions.size() == 1) || (target_positions.size() == start_positions.size())) spcs.hpp:790-793
    if (!(n_targets == 1 || n_targets == n)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: need 1 target or one per start");
    if (noise_mode != FKS_NOISE_PHILOX && noise_mode != FKS_NOISE_INJECTED && noise_mode != FKS_NOISE_NONE)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: unknown noise mode");
    if (noise_mode == FKS_NOISE_INJECTED && (!tape_draws || !tape_off))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate: injected noise needs a tape");
    return FKS_OK;
}

}  // extern "C"

int fks_host::check_sequence(const char* fn, const void* targets, size_t n, size_t n_legs, uint64_t first_particle_id) {
    if (n_legs == 0 || !targets) return fail(FKS_ERR_INVALID_ARGUMENT, std::string(fn) + ": need at least one leg and its targets");
    // the kernel counts legs in 31 bits (the top bit of WarpVars::leg marks a pending leg)
    if (n_legs > 0x7FFFFFFFull) return fail(FKS_ERR_INVALID_ARGUMENT, std::string(fn) + ": more than 2^31 - 1 legs");
    if (n != 0 && (n_legs > UINT64_MAX / n || (uint64_t)(n_legs * n) > UINT64_MAX - first_particle_id))
        return fail(FKS_ERR_INVALID_ARGUMENT, std::string(fn) + ": first_particle_id + n_legs * n_particles overflows 64 bits");
    return FKS_OK;
}

// (fks_internal.h) the pitches let one device's shard of a multi-GPU call read and write its slices of the caller's arrays in place
int fks_host::simulate_host_async(fks_sim* s, const double* starts, const double* targets, size_t targets_pitch, size_t n,
                                  size_t n_targets, size_t n_legs, uint64_t leg_id_stride, int allow_contacts, int noise_mode,
                                  const fks_noise_tape* tape, uint64_t first_particle_id, void* results, size_t results_pitch) {
    if (n == 0) return FKS_OK;
    int rc = FKS_OK;
    NvtxRange range("fks_forward_simulate");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_forward_simulate: cudaSetDevice failed");
    const size_t stride = (size_t)s->robot->stride;
    const size_t rec = fks_sim_result_stride(s);
    const size_t leg_targets = n_targets * stride;  // doubles of one leg's targets on the device
    size_t n_draws = 0;
    if (noise_mode == FKS_NOISE_INJECTED) n_draws = (size_t)tape->offsets[n];
    if ((rc = ensure(&s->d_starts, &s->cap_starts, n * stride)) != FKS_OK) return rc;
    if ((rc = ensure(&s->d_targets, &s->cap_targets, n_legs * leg_targets)) != FKS_OK) return rc;
    if ((rc = ensure(&s->d_results, &s->cap_results, n_legs * n * rec)) != FKS_OK) return rc;
    const bool with_decisions = noise_mode == FKS_NOISE_INJECTED && tape->decisions && tape->decision_offsets;
    size_t n_dec_words = 0;
    if (noise_mode == FKS_NOISE_INJECTED) {
        if ((rc = ensure(&s->d_tape, &s->cap_tape, std::max<size_t>(n_draws, 1))) != FKS_OK) return rc;
        if ((rc = ensure(&s->d_tape_off, &s->cap_tape_off, n + 1)) != FKS_OK) return rc;
        if (with_decisions) {
            n_dec_words = (size_t)tape->decision_offsets[n] * (size_t)(2 + s->robot->host.D);
            if ((rc = ensure(&s->d_dec, &s->cap_dec, std::max<size_t>(n_dec_words, 1))) != FKS_OK) return rc;
            if ((rc = ensure(&s->d_dec_off, &s->cap_dec_off, n + 1)) != FKS_OK) return rc;
        }
    }
    {
        NvtxRange h2d("fks: H2D starts / targets / tape");
        FKS_CUDA(cudaMemcpyAsync(s->d_starts, starts, n * stride * 8, cudaMemcpyHostToDevice, s->stream));
        if (n_legs == 1 || targets_pitch == leg_targets)
            FKS_CUDA(cudaMemcpyAsync(s->d_targets, targets, n_legs * leg_targets * 8, cudaMemcpyHostToDevice, s->stream));
        else
            FKS_CUDA(cudaMemcpy2DAsync(s->d_targets, leg_targets * 8, targets, targets_pitch * 8, leg_targets * 8, n_legs,
                                       cudaMemcpyHostToDevice, s->stream));
        if (noise_mode == FKS_NOISE_INJECTED) {
            if (n_draws) FKS_CUDA(cudaMemcpyAsync(s->d_tape, tape->draws, n_draws * 8, cudaMemcpyHostToDevice, s->stream));
            FKS_CUDA(cudaMemcpyAsync(s->d_tape_off, tape->offsets, (n + 1) * 8, cudaMemcpyHostToDevice, s->stream));
            if (with_decisions) {
                if (n_dec_words) FKS_CUDA(cudaMemcpyAsync(s->d_dec, tape->decisions, n_dec_words * 8, cudaMemcpyHostToDevice, s->stream));
                FKS_CUDA(cudaMemcpyAsync(s->d_dec_off, tape->decision_offsets, (n + 1) * 8, cudaMemcpyHostToDevice, s->stream));
            }
        }
    }
    {
        NvtxRange launch("fks: simulate kernel");
        rc = simulate_on_stream(s, s->d_starts, s->d_targets, n, n_targets, n_legs, leg_id_stride, allow_contacts, noise_mode, s->d_tape,
                                (const uint64_t*)s->d_tape_off, with_decisions ? (const uint64_t*)s->d_dec : nullptr,
                                with_decisions ? (const uint64_t*)s->d_dec_off : nullptr, first_particle_id, s->d_results, s->stream);
    }
    if (rc != FKS_OK) return rc;
    NvtxRange d2h("fks: D2H records");
    if (n_legs == 1 || results_pitch == n * rec)
        FKS_CUDA(cudaMemcpyAsync(results, s->d_results, n_legs * n * rec, cudaMemcpyDeviceToHost, s->stream));
    else
        FKS_CUDA(cudaMemcpy2DAsync(results, results_pitch, s->d_results, n * rec, n * rec, n_legs, cudaMemcpyDeviceToHost, s->stream));
    return FKS_OK;
}

extern "C" {

int fks_forward_simulate_async(fks_sim* s, const double* starts, const double* targets, size_t n, size_t n_targets,
                         int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                         void* results) {
    const int rc = check_batch(s, starts, targets, n, n_targets, noise_mode, tape ? tape->draws : nullptr, tape ? tape->offsets : nullptr, results);
    if (rc != FKS_OK || n == 0) return rc;
    return fks_host::simulate_host_async(s, starts, targets, n_targets * (size_t)s->robot->stride, n, n_targets, 1, n, allow_contacts,
                                         noise_mode, tape, first_particle_id, results, n * fks_sim_result_stride(s));
}

int fks_forward_simulate_sequence(fks_sim* s, const double* starts, const double* targets, size_t n, size_t n_targets, size_t n_legs,
                                  int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                                  void* results) {
    int rc = fks_host::check_sequence("fks_forward_simulate_sequence", targets, n, n_legs, first_particle_id);
    if (rc == FKS_OK)
        rc = check_batch(s, starts, targets, n, n_targets, noise_mode, tape ? tape->draws : nullptr, tape ? tape->offsets : nullptr, results);
    if (rc != FKS_OK || n == 0) return rc;
    rc = fks_host::simulate_host_async(s, starts, targets, n_targets * (size_t)s->robot->stride, n, n_targets, n_legs, n, allow_contacts,
                                       noise_mode, tape, first_particle_id, results, n * fks_sim_result_stride(s));
    if (rc != FKS_OK) return rc;
    return fks_sim_synchronize(s);
}

int fks_sim_synchronize(fks_sim* s) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_synchronize: null simulator");
    NvtxRange range("fks_sim_synchronize");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_sim_synchronize: cudaSetDevice failed");
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    return FKS_OK;
}

int fks_forward_simulate(fks_sim* s, const double* starts, const double* targets, size_t n, size_t n_targets,
                         int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                         void* results) {
    const int rc = fks_forward_simulate_async(s, starts, targets, n, n_targets, allow_contacts, noise_mode, tape, first_particle_id, results);
    if (rc != FKS_OK || n == 0) return rc;
    return fks_sim_synchronize(s);
}

size_t fks_sim_trace_stride(const fks_sim* s) {
    return s ? sizeof(fks_trace_header) + (size_t)std::max(s->robot->stride, s->robot->host.D) * 8 : 0;
}

// ForwardSimulateRobot(..., trace, enable_tracing = true, ...) (spcs.hpp:824-829) for one particle
int fks_forward_simulate_traced(fks_sim* s, const double* start, const double* target, int allow_contacts, int noise_mode,
                                const fks_noise_tape* tape, uint64_t particle_id, void* result, void* trace_records,
                                size_t trace_capacity, size_t* n_records) {
    if (!s || !n_records || (trace_capacity > 0 && !trace_records) || trace_capacity > 0x7fffffffull)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_forward_simulate_traced: bad argument");
    *n_records = 0;
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_forward_simulate_traced: cudaSetDevice failed");
    const size_t rec = fks_sim_trace_stride(s);
    NvtxRange range("fks_forward_simulate_traced");
    // the trace buffer and its counter belong to the simulator and grow on demand (no allocation per call)
    int rc = FKS_OK;
    if ((rc = ensure(&s->d_trace_buf, &s->cap_trace_buf, (std::max<size_t>(trace_capacity, 1) * rec + 7) / 8 + 1)) != FKS_OK) return rc;
    char* d_trace = reinterpret_cast<char*>(s->d_trace_buf) + 8;
    unsigned int* d_count = reinterpret_cast<unsigned int*>(s->d_trace_buf);
    FKS_CUDA(cudaMemsetAsync(d_count, 0, sizeof(unsigned int), s->stream));
    s->d_trace = d_trace;
    s->d_trace_count = d_count;
    s->trace_capacity = (unsigned int)trace_capacity;
    rc = fks_forward_simulate(s, start, target, 1, 1, allow_contacts, noise_mode, tape, particle_id, result);
    s->d_trace = nullptr;
    s->d_trace_count = nullptr;
    s->trace_capacity = 0;
    if (rc != FKS_OK) return rc;
    unsigned int count = 0;
    FKS_CUDA(cudaMemcpyAsync(&count, d_count, sizeof(count), cudaMemcpyDeviceToHost, s->stream));
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    if (trace_capacity && count) {
        FKS_CUDA(cudaMemcpyAsync(trace_records, d_trace, std::min<size_t>(count, trace_capacity) * rec, cudaMemcpyDeviceToHost, s->stream));
        FKS_CUDA(cudaStreamSynchronize(s->stream));
    }
    *n_records = count;
    return FKS_OK;
}

int fks_reverse_simulate(fks_sim* s, const double* starts, const double* targets, size_t n, size_t n_targets,
                         int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                         void* results) {
    // ReverseSimulateMutableRobot forwards to ForwardSimulateMutableRobot (spcs.hpp:838-841)
    return fks_forward_simulate(s, starts, targets, n, n_targets, allow_contacts, noise_mode, tape, first_particle_id, results);
}

int fks_forward_simulate_device(fks_sim* s, const double* d_starts, const double* d_targets, size_t n, size_t n_targets,
                                int allow_contacts, int noise_mode, const double* d_tape_draws,
                                const uint64_t* d_tape_offsets, uint64_t first_particle_id, void* d_results,
                                void* cuda_stream) {
    int rc = check_batch(s, d_starts, d_targets, n, n_targets, noise_mode, d_tape_draws, d_tape_offsets, d_results);
    if (rc != FKS_OK || n == 0) return rc;
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_forward_simulate_device: cudaSetDevice failed");
    return simulate_on_stream(s, d_starts, d_targets, n, n_targets, 1, n, allow_contacts, noise_mode, d_tape_draws, d_tape_offsets,
                              nullptr, nullptr, first_particle_id, d_results, (cudaStream_t)cuda_stream);
}

int fks_forward_simulate_sequence_device(fks_sim* s, const double* d_starts, const double* d_targets, size_t n, size_t n_targets,
                                         size_t n_legs, int allow_contacts, int noise_mode, const double* d_tape_draws,
                                         const uint64_t* d_tape_offsets, uint64_t first_particle_id, void* d_results, void* cuda_stream) {
    int rc = fks_host::check_sequence("fks_forward_simulate_sequence_device", d_targets, n, n_legs, first_particle_id);
    if (rc == FKS_OK) rc = check_batch(s, d_starts, d_targets, n, n_targets, noise_mode, d_tape_draws, d_tape_offsets, d_results);
    if (rc != FKS_OK || n == 0) return rc;
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_forward_simulate_sequence_device: cudaSetDevice failed");
    return simulate_on_stream(s, d_starts, d_targets, n, n_targets, n_legs, n, allow_contacts, noise_mode, d_tape_draws, d_tape_offsets,
                              nullptr, nullptr, first_particle_id, d_results, (cudaStream_t)cuda_stream);
}

int fks_check_config_collision(fks_sim* s, const double* configs, size_t n, double inflation_ratio, uint8_t* out) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_check_config_collision: null simulator");
    if (n == 0) return FKS_OK;
    if (!configs || !out || std::isnan(inflation_ratio)) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_check_config_collision: bad argument");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_check_config_collision: cudaSetDevice failed");
    const size_t stride = (size_t)s->robot->stride;
    int rc;
    if ((rc = ensure(&s->d_starts, &s->cap_starts, n * stride)) != FKS_OK) return rc;
    if ((rc = ensure(&s->d_results, &s->cap_results, n)) != FKS_OK) return rc;
    FKS_CUDA(cudaMemcpyAsync(s->d_starts, configs, n * stride * 8, cudaMemcpyHostToDevice, s->stream));
    LaunchArgs a = s->plan;
    a.env = s->env->dev;
    a.sp = s->sp;
    a.robot = s->robot->d_robot;
    a.pxy = s->robot->d_pxy;
    a.pzl = s->robot->d_pzl;
    a.starts = s->d_starts;
    a.scratch = s->d_scratch;
    a.jscratch = s->d_jscratch;
    a.ctx_store = s->d_ctx_store;
    a.n_particles = n;
    a.cfg_stride = s->robot->stride;
    const size_t per_sm = (n + (size_t)s->num_sms - 1) / (size_t)s->num_sms;
    const int wpb = (int)std::max<size_t>(1, std::min<size_t>((size_t)s->plan.warps_per_block, per_sm));
    a.warps_per_block = wpb;
    a.pool = wpb;  // (check_config keeps no context pool; scratch slots are per warp)
    a.sync_off = a.warps_off + wpb * a.wl.total * 8;
    const size_t dyn_smem = (size_t)a.sync_off + kSyncBytes;
    const int grid = (int)std::min<size_t>((size_t)s->grid_max, (n + (size_t)wpb - 1) / (size_t)wpb);
    rc = launch_check_config(s->robot->host.kind, a, grid, dyn_smem, s->stream, inflation_ratio, (unsigned char*)s->d_results);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "check_config kernel launch");
    s->launches++;
    FKS_CUDA(cudaMemcpyAsync(out, s->d_results, n, cudaMemcpyDeviceToHost, s->stream));
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    return FKS_OK;
}

// waits for the simulator's own work only: its stream and the last launch made on a caller's stream
static int sync_simulator(fks_sim* s) {
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    if (s->has_last) FKS_CUDA(cudaEventSynchronize(s->last_done));
    return FKS_OK;
}

int fks_get_statistics(fks_sim* s, uint64_t* out) {
    if (!s || !out) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_get_statistics: null argument");
    DeviceGuard guard(s->device);
    int rc = sync_simulator(s);
    if (rc != FKS_OK) return rc;
    FKS_CUDA(cudaMemcpyAsync(out, s->d_stats, FKS_NUM_STATS * sizeof(uint64_t), cudaMemcpyDeviceToHost, s->stream));
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    return FKS_OK;
}

// Measurement aid (bench.py): device time of the simulate kernel of the last batch call.
int fks_sim_enable_kernel_timing(fks_sim* s, int enable) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_enable_kernel_timing: null simulator");
    DeviceGuard guard(s->device);
    if (enable)
        for (int i = 0; i < 2; i++)
            if (!s->tev[i]) FKS_CUDA(cudaEventCreate(&s->tev[i]));
    s->timing = enable ? 1 : 0;
    s->timed_kernels = 0;
    return FKS_OK;
}

// out_ms[0] = device milliseconds of the simulate kernel of the last call; *n_kernels = 1 when it was timed.  Waits for the call.
int fks_sim_kernel_times(fks_sim* s, double* out_ms, int* n_kernels) {
    if (!s || !out_ms || !n_kernels) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_sim_kernel_times: null argument");
    DeviceGuard guard(s->device);
    *n_kernels = s->timed_kernels;
    for (int i = 0; i < s->timed_kernels; i++) {
        FKS_CUDA(cudaEventSynchronize(s->tev[i + 1]));
        float ms = 0.f;
        FKS_CUDA(cudaEventElapsedTime(&ms, s->tev[i], s->tev[i + 1]));
        out_ms[i] = (double)ms;
    }
    return FKS_OK;
}

int fks_reset_statistics(fks_sim* s) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_reset_statistics: null argument");
    DeviceGuard guard(s->device);
    int rc = sync_simulator(s);
    if (rc != FKS_OK) return rc;
    FKS_CUDA(cudaMemsetAsync(s->d_stats, 0, 128 * sizeof(uint64_t), s->stream));
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    return FKS_OK;
}

uint64_t fks_sim_launch_count(const fks_sim* s) { return s ? s->launches : 0; }

// developer aid (not in the public header): per-phase clock totals of builds made with -DFKS_PHASE_TIMERS
int fks_debug_phase_cycles(fks_sim* s, uint64_t* out16) {
    if (!s || !out16) return FKS_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(s->device);
    FKS_CUDA(cudaDeviceSynchronize());
    FKS_CUDA(cudaMemcpy(out16, s->d_stats + 16, 48 * sizeof(uint64_t), cudaMemcpyDeviceToHost));  // 48 values
    launch_dbg_copy(s->d_stats + 64, nullptr);  // (timers build: 64 more developer counters behind them)
    FKS_CUDA(cudaDeviceSynchronize());
    FKS_CUDA(cudaMemcpy(out16 + 48, s->d_stats + 64, 64 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return FKS_OK;
}

const char* fks_sim_kernel_info(fks_sim* s) { return s ? s->info.c_str() : ""; }

// ---------------------------------------------------------------------------------------------
// first consumer of a batch on the device (fksgpu.h, SURVEY.md 8f-3)
// ---------------------------------------------------------------------------------------------
int fks_end_states_partition(fks_sim* s, const void* d_results, size_t n, uint32_t* d_order, uint64_t* counts, void* cuda_stream) {
    if (!s || !counts) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_partition: null argument");
    counts[0] = counts[1] = 0;
    if (n == 0) return FKS_OK;
    if (!d_results || !d_order || n > 0xffffffffull) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_end_states_partition: bad buffer or count");
    NvtxRange range("fks_end_states_partition");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_end_states_partition: cudaSetDevice failed");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    int rc;
    const size_t n_blocks = (n + 1023) / 1024;
    if ((rc = ensure(&s->d_part, &s->cap_part, n_blocks + 4)) != FKS_OK) return rc;  // [2 x u64 totals | block counts]
    unsigned long long* totals = reinterpret_cast<unsigned long long*>(s->d_part);
    rc = launch_partition((const char*)d_results, fks_sim_result_stride(s), s->robot->stride, n, s->d_part + 4, totals, d_order, stream);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_partition: launch");
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
    const int rc = launch_pairwise_distance(s->robot->host.kind, s->robot->d_robot, (const char*)d_results, fks_sim_result_stride(s),
                                            s->robot->stride, d_subset, (unsigned)m, d_out, cuda_stream);
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

    // one upload: [offsets (n + 1) | totals (2) | counts (n, zero), small segments, large segments as u32]
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
    unsigned* d32 = reinterpret_cast<unsigned*>(s->d_clu + n_segments + 3);
    ClusterLaunch c;
    c.robot = s->robot->d_robot;
    c.results = (const char*)d_results;
    c.rec_stride = fks_sim_result_stride(s);
    c.cfg_stride = s->robot->stride;
    c.complete = linkage == FKS_LINKAGE_COMPLETE;
    c.separate_contact = separate_contact != 0;
    c.threshold = max_cluster_distance;
    c.order = d_order;
    c.offsets = s->d_clu;
    c.n_segments = (unsigned)n_segments;
    c.small_segs = d32 + n_segments;
    c.n_small = (unsigned)small_segs.size();
    c.small_cap = small_cap;
    c.large_segs = d32 + n_segments + small_segs.size();
    c.n_large = (unsigned)large_segs.size();
    c.large_cap = large_cap;
    c.work = s->d_clu_mat;
    c.large_slots = large_slots;
    c.labels = d_labels;
    c.counts = d32;
    c.totals = s->d_clu + n_segments + 1;
    rc = launch_cluster(s->robot->host.kind, c, stream);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_cluster: launch");
    s->launches += 2 + (small_segs.empty() ? 0 : 1) + (large_segs.empty() ? 0 : 1);
    std::vector<unsigned> base(n_segments);
    unsigned long long total = 0;
    FKS_CUDA(cudaMemcpyAsync(base.data(), d32, n_segments * sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    FKS_CUDA(cudaMemcpyAsync(&total, c.totals + 1, sizeof(total), cudaMemcpyDeviceToHost, stream));
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
    rc = launch_groups(s->robot->host.kind, g, stream);
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
    if (!s->sel_read) FKS_CUDA(cudaEventCreateWithFlags(&s->sel_read, cudaEventDisableTiming));
    // the ids go through one buffer: a launch of an earlier call, perhaps on another stream, must have read it first
    if (s->has_sel && n_selected > s->cap_sel) FKS_CUDA(cudaEventSynchronize(s->sel_read));
    int rc;
    if ((rc = ensure(&s->d_sel, &s->cap_sel, n_selected)) != FKS_OK) return rc;
    if (s->has_sel) FKS_CUDA(cudaStreamWaitEvent(stream, s->sel_read, 0));
    FKS_CUDA(cudaMemcpyAsync(s->d_sel, selected, n_selected * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    rc = launch_gather_starts((const char*)d_results, fks_sim_result_stride(s), s->robot->stride, d_group_offsets, d_members, s->d_sel,
                              (unsigned)n_selected, (unsigned)per_group, d_group_targets, d_starts, d_targets, stream);
    if (rc != 0) return cuda_fail((cudaError_t)rc, "fks_end_states_gather_starts: launch");
    s->launches += 1;
    FKS_CUDA(cudaEventRecord(s->sel_read, stream));
    s->has_sel = true;
    return FKS_OK;
}

// ---------------------------------------------------------------------------------------------
// test entry: the device's stacked-Jacobian solver on caller-provided systems (fksgpu.h)
// ---------------------------------------------------------------------------------------------
int fks_debug_qr_solve(int device, const double* systems, const uint64_t* offsets, const int32_t* rows, int32_t cols, size_t n,
                       double* solutions, uint32_t* flags) {
    if (n == 0) return FKS_OK;
    if (!systems || !offsets || !rows || !solutions || !flags || cols < 1 || cols >= kMaxDof)
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_debug_qr_solve: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "no CUDA device");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "cudaSetDevice failed");
    const size_t total = (size_t)offsets[n];
    double *d_work = nullptr, *d_x = nullptr;
    unsigned long long* d_off = nullptr;
    int* d_rows = nullptr;
    unsigned* d_flags = nullptr;
    int rc = upload(&d_work, systems, total);
    if (rc == FKS_OK) rc = upload(&d_off, (const unsigned long long*)offsets, n + 1);
    if (rc == FKS_OK) rc = upload(&d_rows, (const int*)rows, n);
    if (rc == FKS_OK) rc = upload(&d_x, (const double*)nullptr, n * (size_t)cols);
    if (rc == FKS_OK) rc = upload(&d_flags, (const unsigned*)nullptr, n);
    if (rc == FKS_OK) {
        const int lrc = launch_qr_solve(d_work, d_off, d_rows, cols, (int)n, d_x, d_flags, nullptr);
        cudaError_t err = lrc ? (cudaError_t)lrc : cudaDeviceSynchronize();
        if (err == cudaSuccess) err = cudaMemcpy(solutions, d_x, n * (size_t)cols * 8, cudaMemcpyDeviceToHost);
        if (err == cudaSuccess) err = cudaMemcpy(flags, d_flags, n * 4, cudaMemcpyDeviceToHost);
        if (err != cudaSuccess) rc = cuda_fail(err, "fks_debug_qr_solve");
    }
    cudaFree(d_work);
    cudaFree(d_off);
    cudaFree(d_rows);
    cudaFree(d_x);
    cudaFree(d_flags);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// roofline micro-benchmarks
// ---------------------------------------------------------------------------------------------
int fks_measure_fp64_peak(int device, double* flops_per_s) {
    if (!flops_per_s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_measure_fp64_peak: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "no CUDA device");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    FKS_CUDA(cudaGetDeviceProperties(&prop, device));
    double* d_out = nullptr;
    FKS_CUDA(cudaMalloc((void**)&d_out, 8));
    const int grid = prop.multiProcessorCount * 8, iters = 1 << 16;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, 0);
        int rc = launch_fp64_peak(d_out, grid, iters, nullptr);
        cudaEventRecord(e1, 0);
        cudaError_t err = cudaEventSynchronize(e1);
        if (rc != 0 || err != cudaSuccess) {
            cudaFree(d_out);
            return cuda_fail(rc ? (cudaError_t)rc : err, "fp64 peak kernel");
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = 2.0 * 8.0 * (double)iters * 256.0 * (double)grid;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_out);
    *flops_per_s = best;
    return FKS_OK;
}

int fks_measure_gather_rate(int device, size_t bytes, double* gathers_per_s) {
    if (!gathers_per_s || bytes < 4096) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_measure_gather_rate: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(FKS_ERR_NO_DEVICE, "no CUDA device");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    FKS_CUDA(cudaGetDeviceProperties(&prop, device));
    size_t n = 1;
    while (n * 2 * 4 <= bytes) n <<= 1;  // power-of-two element count
    float *d_data = nullptr, *d_out = nullptr;
    FKS_CUDA(cudaMalloc((void**)&d_data, n * 4));
    FKS_CUDA(cudaMalloc((void**)&d_out, 4));
    FKS_CUDA(cudaMemset(d_data, 0, n * 4));
    const int grid = prop.multiProcessorCount * 8, iters = 2048;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, 0);
        int rc = launch_gather(d_data, (unsigned long long)(n - 1), d_out, grid, iters, nullptr);
        cudaEventRecord(e1, 0);
        cudaError_t err = cudaEventSynchronize(e1);
        if (rc != 0 || err != cudaSuccess) {
            cudaFree(d_data);
            cudaFree(d_out);
            return cuda_fail(rc ? (cudaError_t)rc : err, "gather kernel");
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double gathers = 4.0 * (double)iters * 256.0 * (double)grid;
        if (rep > 0) best = std::max(best, gathers / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_data);
    cudaFree(d_out);
    *gathers_per_s = best;
    return FKS_OK;
}

}  // extern "C"
