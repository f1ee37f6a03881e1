// Types shared between the translation units of libfksgpu.so (not part of the C ABI).
#ifndef FKS_INTERNAL_H
#define FKS_INTERNAL_H

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only: named host ranges for Nsight Systems / ncu --nvtx, free without a tool attached

#include <cstdint>
#include <string>
#include <vector>

#include "fks_device_types.h"

namespace fks_host {
void set_last_error(const std::string& msg);

// Grid geometry chosen by BuildEnvironment (simulator_environment_builder.cpp:49-160): origin at the
// minimum corner of the obstacle bounding box minus 3.5 cells, identity rotation, ceil(size / res) cells.
struct GridGeometry {
    double origin[12];
    double inv_origin[12];
    double res;
    int64_t nx, ny, nz;
};
// Returns FKS_OK or FKS_ERR_INVALID_ARGUMENT (message set).  Used by the host and the device builder.
int compute_grid_geometry(const fks_obstacle* obstacles, size_t n_obstacles, double resolution, GridGeometry* out);

// what a sequence call asks beyond a single call's checks, before anything is allocated or copied: 1 .. 2^31 - 1 legs, their
// targets, and first_particle_id + n_legs * n computed without overflowing 64 bits (so the last id used is at most 2^64 - 2)
// -- FKS_OK or FKS_ERR_INVALID_ARGUMENT, message prefixed by `fn`
int check_sequence(const char* fn, const void* targets, size_t n, size_t n_legs, uint64_t first_particle_id);
// The host-buffer batch behind fks_forward_simulate_async / fks_forward_simulate_sequence and each device's shard of the
// multi-GPU calls: copies in, n_legs legs per particle (Philox ids first_particle_id + k * leg_id_stride + i), copies out,
// asynchronous on the simulator's stream.  Leg k's targets are read at targets + k * targets_pitch (doubles) and its
// records written at results + k * results_pitch (bytes).  Arguments are checked by the caller.
int simulate_host_async(fks_sim* s, const double* starts, const double* targets, size_t targets_pitch, size_t n, size_t n_targets,
                        size_t n_legs, uint64_t leg_id_stride, int allow_contacts, int noise_mode, const fks_noise_tape* tape,
                        uint64_t first_particle_id, void* results, size_t results_pitch);

// A workspace that calls on any stream use in turn: acquire() makes `stream` wait for the launches of the previous call that
// used it (and, when it has to grow, the host as well, since those launches may still read the old allocation); release()
// marks the end of this call's launches on `stream`.  Both return FKS_OK or an FKS_ERR_* code (message set).
struct StreamBuffer {
    unsigned char* ptr = nullptr;
    size_t cap = 0;  // bytes
    cudaEvent_t done = nullptr;
    bool pending = false;
    int acquire(size_t bytes, cudaStream_t stream);
    int release(cudaStream_t stream);
    void destroy();  // waits for the last user
};
}  // namespace fks_host

namespace {

inline int fail(int code, const std::string& msg) {
    fks_host::set_last_error(msg);
    return code;
}
inline int cuda_fail(cudaError_t err, const char* what) {
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

struct NvtxRange {  // one named range per C-ABI call and per stage inside it
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

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
    fksdev::DevRobot host;
    fksdev::DevRobot* d_robot;
    double2* d_pxy;
    fksdev::PointZL* d_pzl;
    int stride;
};

struct fks_sim {
    int device;
    const fks_env* env;
    const fks_robot* robot;
    fksdev::DevSolver sp;
    uint64_t seed;
    int32_t debug_level;
    cudaStream_t stream;
    int grid_max, num_sms;
    size_t dyn_smem;
    fksdev::KernelInfo kinfo;
    fksdev::LaunchArgs plan;  // layouts and shared-memory offsets (simulate_smem_plan)
    char* d_scratch;
    char* d_jscratch = nullptr;
    unsigned long long* d_stats;
    unsigned int* d_counter;
    // staging for the host-buffer entry point (grown on demand)
    double *d_starts, *d_targets, *d_tape;
    unsigned long long *d_tape_off, *d_dec, *d_dec_off;
    char* d_results;
    size_t cap_starts, cap_targets, cap_tape, cap_tape_off, cap_results, cap_dec, cap_dec_off;
    // workspaces of the batch consumers (fks_consumers.cu, where their layouts are)
    unsigned int* d_part = nullptr;
    size_t cap_part = 0;
    unsigned long long* d_clu = nullptr;
    size_t cap_clu = 0;
    double* d_clu_mat = nullptr;
    size_t cap_clu_mat = 0;
    unsigned long long* d_grp = nullptr;
    size_t cap_grp = 0;
    fks_host::StreamBuffer sel, near;  // fks_end_states_gather_starts, fks_nearest_configurations
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
    // for the previous one (the _device calls take the caller's stream; serialised_launch in fks_api.cu)
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

// Device environment (fks_env_create / fks_env_build_device).
struct fks_env {
    int device;
    fksdev::DevEnv dev;
    float* d_sdf;
    unsigned long long* d_keys;   // normal hash, 16-byte slots
    double* d_entries;            // 6 doubles per stored normal
    // CSR view of the normal table in ascending cell order (kept for fks_env_download)
    long long* d_cell_index;      // [n_normal_cells]
    unsigned int* d_cell_start;   // [n_normal_cells + 1]
    unsigned char* d_occupancy;   // 1 byte per cell, only for device-built environments (else null)
    long long n_normal_cells;
    size_t n_entries;
    size_t sdf_bytes;
    size_t l2_window_bytes;
    double build_ms[9];           // device builder phase timings (fks_env_build_timings)
};

// Host environment (fks_build_environment / fks_env_download).
struct fks_built_env {
    fks_env_desc desc;
    std::vector<float> sdf;
    std::vector<uint8_t> occupancy;
    std::vector<int64_t> normal_cell_index;
    std::vector<uint32_t> normal_cell_start;
    std::vector<double> normal_entries;
};

#endif
