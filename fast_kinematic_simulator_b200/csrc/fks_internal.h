// Types shared between the translation units of libfksgpu.so (not part of the C ABI).
#ifndef FKS_INTERNAL_H
#define FKS_INTERNAL_H

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
}  // namespace fks_host

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
