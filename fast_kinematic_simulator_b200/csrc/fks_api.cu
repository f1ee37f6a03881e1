// C ABI of libfksgpu.so (include/fksgpu.h): uploads, launch plumbing, statistics.
// The computation itself is in fks_kernels.cu, the calls that consume a batch on the device in fks_consumers.cu, the
// environment builder in host/environment_builder.cpp.
// There is NO CPU fallback: every compute entry point fails with FKS_ERR_NO_DEVICE / FKS_ERR_CUDA when
// the device path cannot run.

#include <cuda_runtime.h>

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

template <typename T>
int upload(T** dst, const T* src, size_t n) {
    *dst = nullptr;
    if (n == 0) n = 1;
    FKS_CUDA(cudaMalloc((void**)dst, n * sizeof(T)));
    if (src) FKS_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return FKS_OK;
}

// The launches of one simulator share its particle counter, statistics and scratch slots (the simulate kernel's contexts and
// check_config_kernel's warps both use d_scratch), so they never overlap: the one kernel `enqueue` puts on `stream` waits for
// the previous launch when that was on another stream, and the next launch waits for it.  `enqueue` returns FKS_OK or a code.
template <typename Enqueue>
int serialised_launch(fks_sim* s, cudaStream_t stream, Enqueue&& enqueue) {
    if (s->has_last && stream != s->last_stream) FKS_CUDA(cudaStreamWaitEvent(stream, s->last_done, 0));
    const int rc = enqueue();
    if (rc != FKS_OK) return rc;
    FKS_CUDA(cudaEventRecord(s->last_done, stream));
    s->last_stream = stream;
    s->has_last = true;
    s->launches++;
    return FKS_OK;
}

}  // namespace

extern "C" {

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
    cudaFree(s->d_grp);
    s->sel.destroy();
    s->near.destroy();
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
    const void* l2_base = s->env->l2_window_bytes ? s->env->d_sdf : nullptr;
    a.ctx_store = s->d_ctx_store;
    a.pool = std::max(wpb, std::min((s->pool_eighths * wpb + 7) / 8, s->pool));
    return serialised_launch(s, stream, [&]() -> int {
        FKS_CUDA(cudaMemsetAsync(s->d_counter, 0, 4 * sizeof(unsigned int), stream));
        if (s->timing) FKS_CUDA(cudaEventRecord(s->tev[0], stream));
        const int rc = launch_simulate(s->robot->host.kind, a, grid, dyn_smem, stream, l2_base, s->env->l2_window_bytes);
        if (rc != 0) return cuda_fail((cudaError_t)rc, "simulate kernel launch");
        if (s->timing) FKS_CUDA(cudaEventRecord(s->tev[1], stream));
        s->timed_kernels = s->timing ? 1 : 0;
        return FKS_OK;
    });
}

// CheckConfigCollision of n configurations d_configs[n][cfg_stride] into d_out[0 .. n), one warp per configuration
static int check_config_on_stream(fks_sim* s, const double* d_configs, size_t n, double inflation_ratio, uint8_t* d_out,
                                  cudaStream_t stream) {
    LaunchArgs a = s->plan;
    a.env = s->env->dev;
    a.sp = s->sp;
    a.robot = s->robot->d_robot;
    a.pxy = s->robot->d_pxy;
    a.pzl = s->robot->d_pzl;
    a.starts = d_configs;
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
    return serialised_launch(s, stream, [&]() -> int {
        const int rc = launch_check_config(s->robot->host.kind, a, grid, dyn_smem, stream, inflation_ratio, d_out);
        return rc != 0 ? cuda_fail((cudaError_t)rc, "check_config kernel launch") : FKS_OK;
    });
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
    rc = check_config_on_stream(s, s->d_starts, n, inflation_ratio, (uint8_t*)s->d_results, s->stream);
    if (rc != FKS_OK) return rc;
    FKS_CUDA(cudaMemcpyAsync(out, s->d_results, n, cudaMemcpyDeviceToHost, s->stream));
    FKS_CUDA(cudaStreamSynchronize(s->stream));
    return FKS_OK;
}

int fks_check_config_collision_device(fks_sim* s, const double* d_configs, size_t n, double inflation_ratio, uint8_t* d_out,
                                      void* cuda_stream) {
    if (!s) return fail(FKS_ERR_INVALID_ARGUMENT, "fks_check_config_collision_device: null simulator");
    if (n == 0) return FKS_OK;
    if (!d_configs || !d_out || std::isnan(inflation_ratio))
        return fail(FKS_ERR_INVALID_ARGUMENT, "fks_check_config_collision_device: bad argument");
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(FKS_ERR_CUDA, "fks_check_config_collision_device: cudaSetDevice failed");
    return check_config_on_stream(s, d_configs, n, inflation_ratio, d_out, (cudaStream_t)cuda_stream);
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
