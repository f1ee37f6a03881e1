// Multi-GPU flavour of the batched forward simulation behind the C ABI (include/fksgpu.h, fks_multi_*): one process,
// the GPUs of one box.  SimpleParticleContactSimulator::ForwardSimulateRobots is data parallel over particles
// (simple_particle_contact_simulator.hpp:795-802), so the batch is cut into contiguous shards, one per device, with the
// environment and the robot replicated (fks_env_create / fks_robot_create / fks_sim_create per device).  Philox noise is
// keyed by the GLOBAL particle id, so the records do not depend on the number of devices.
//   * host buffers (fks_multi_forward_simulate): every device copies its shard in, simulates, and copies its records
//     straight into the caller's result array -- no collective is needed to return all N records to the caller;
//   * device-resident results (fks_multi_forward_simulate_device): every device ends with ALL N records, exchanged by one
//     ncclAllGather over NVLink.  NCCL is bound at run time (dlopen of libnccl.so.2 -- the copy the process already loaded,
//     e.g. PyTorch's, when there is one), so the library has no link-time dependency on it;
//   * statistics are summed over the devices on the host.

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "fks_internal.h"

namespace {

int mfail(int code, const std::string& msg) {
    fks_host::set_last_error(msg);
    return code;
}

// ---- NCCL through dlopen --------------------------------------------------------------------------------------------
struct Nccl {
    void* handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

Nccl& nccl() {
    static Nccl n;
    static bool tried = false;
    if (tried) return n;
    tried = true;
    n.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!n.handle) return n;
    n.CommInitAll = (decltype(n.CommInitAll))dlsym(n.handle, "ncclCommInitAll");
    n.CommDestroy = (decltype(n.CommDestroy))dlsym(n.handle, "ncclCommDestroy");
    n.AllGather = (decltype(n.AllGather))dlsym(n.handle, "ncclAllGather");
    n.GroupStart = (decltype(n.GroupStart))dlsym(n.handle, "ncclGroupStart");
    n.GroupEnd = (decltype(n.GroupEnd))dlsym(n.handle, "ncclGroupEnd");
    n.GetErrorString = (decltype(n.GetErrorString))dlsym(n.handle, "ncclGetErrorString");
    n.ok = n.CommInitAll && n.CommDestroy && n.AllGather && n.GroupStart && n.GroupEnd && n.GetErrorString;
    return n;
}

}  // namespace

struct fks_multi_sim {
    std::vector<int> devices;
    std::vector<fks_env*> envs;
    std::vector<fks_robot*> robots;
    std::vector<fks_sim*> sims;
    std::vector<ncclComm_t> comms;     // created on the first device-resident call
    std::vector<cudaStream_t> streams; // one per device for the device-resident call
    size_t rec_stride = 0;
    int cfg_stride = 0, n_dof = 0;
};

extern "C" {

void fks_multi_sim_destroy(fks_multi_sim* m) {
    if (!m) return;
    for (size_t d = 0; d < m->devices.size(); d++) {
        cudaSetDevice(m->devices[d]);
        if (d < m->comms.size() && m->comms[d]) nccl().CommDestroy(m->comms[d]);
        if (d < m->streams.size() && m->streams[d]) cudaStreamDestroy(m->streams[d]);
        if (d < m->sims.size()) fks_sim_destroy(m->sims[d]);
        if (d < m->robots.size()) fks_robot_destroy(m->robots[d]);
        if (d < m->envs.size()) fks_env_destroy(m->envs[d]);
    }
    delete m;
}

int fks_multi_sim_create(const int32_t* devices, int32_t n_devices, const fks_env_desc* env, const fks_robot_desc* robot,
                         const fks_solver_params* params, double simulation_controller_frequency, uint64_t prng_seed,
                         int32_t debug_level, fks_multi_sim** out) {
    if (!out || !env || !robot || !params || n_devices < 1 || n_devices > 64)
        return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_sim_create: bad argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return mfail(FKS_ERR_NO_DEVICE, "fks_multi_sim_create: no CUDA device");
    fks_multi_sim* m = new (std::nothrow) fks_multi_sim();
    if (!m) return mfail(FKS_ERR_OUT_OF_MEMORY, "fks_multi_sim_create: out of host memory");
    for (int d = 0; d < n_devices; d++) {
        const int dev = devices ? devices[d] : d;
        if (dev < 0 || dev >= ndev || std::find(m->devices.begin(), m->devices.end(), dev) != m->devices.end()) {
            fks_multi_sim_destroy(m);
            return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_sim_create: bad or repeated device index");
        }
        m->devices.push_back(dev);
    }
    for (int d = 0; d < n_devices; d++) {
        fks_env* e = nullptr;
        fks_robot* r = nullptr;
        fks_sim* s = nullptr;
        int rc = fks_env_create(m->devices[d], env, &e);
        if (rc == FKS_OK) m->envs.push_back(e);
        if (rc == FKS_OK) rc = fks_robot_create(m->devices[d], robot, &r);
        if (rc == FKS_OK) m->robots.push_back(r);
        if (rc == FKS_OK) rc = fks_sim_create(e, r, params, simulation_controller_frequency, prng_seed, debug_level, &s);
        if (rc == FKS_OK) m->sims.push_back(s);
        if (rc != FKS_OK) {
            fks_multi_sim_destroy(m);
            return rc;  // message set by the failing call
        }
    }
    m->rec_stride = fks_sim_result_stride(m->sims[0]);
    m->cfg_stride = fks_robot_config_stride(m->robots[0]);
    m->n_dof = robot->n_dof;
    *out = m;
    return FKS_OK;
}

int fks_multi_sim_device_count(const fks_multi_sim* m) { return m ? (int)m->devices.size() : 0; }

// contiguous shards: the first (n % G) devices take one particle more
static void shard_of(size_t n, size_t G, size_t d, size_t* lo, size_t* hi) {
    const size_t base = n / G, extra = n % G;
    *lo = d * base + std::min(d, extra);
    *hi = *lo + base + (d < extra ? 1 : 0);
}

// n_legs consecutive legs per particle (fks_multi_forward_simulate_sequence; 1 = fks_multi_forward_simulate): every shard keys
// its Philox ids by the whole batch (leg_id_stride = n) and writes its [n_legs][shard] records into the caller's [n_legs][n] array
static int multi_simulate(fks_multi_sim* m, const double* starts, const double* targets, size_t n, size_t n_targets, size_t n_legs,
                          int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id, void* results) {
    if (!m) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate: null simulator");
    if (n == 0) return FKS_OK;
    if (!starts || !targets || !results || !(n_targets == 1 || n_targets == n))
        return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate: need buffers and 1 target or one per start");
    if (noise_mode != FKS_NOISE_PHILOX && noise_mode != FKS_NOISE_INJECTED && noise_mode != FKS_NOISE_NONE)
        return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate: unknown noise mode");
    if (noise_mode == FKS_NOISE_INJECTED && (!tape || !tape->draws || !tape->offsets))
        return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate: injected noise needs a tape");
    const size_t G = m->devices.size();
    const size_t stride = (size_t)m->cfg_stride;
    int rc = FKS_OK;
    // enqueue every shard (copies and kernels are asynchronous on each simulator's stream), then wait for all of them
    std::vector<fks_noise_tape> tapes(G);
    std::vector<std::vector<uint64_t>> toff(G), doff(G);
    for (size_t d = 0; d < G && rc == FKS_OK; d++) {
        size_t lo, hi;
        shard_of(n, G, d, &lo, &hi);
        if (hi == lo) continue;
        const fks_noise_tape* t = nullptr;
        if (noise_mode == FKS_NOISE_INJECTED && tape) {
            // a shard's view of the tapes: offsets rebased to the shard's first draw / record
            toff[d].assign(tape->offsets + lo, tape->offsets + hi + 1);
            for (auto& v : toff[d]) v -= tape->offsets[lo];
            tapes[d].draws = tape->draws + tape->offsets[lo];
            tapes[d].offsets = toff[d].data();
            tapes[d].decisions = nullptr;
            tapes[d].decision_offsets = nullptr;
            if (tape->decisions && tape->decision_offsets) {
                doff[d].assign(tape->decision_offsets + lo, tape->decision_offsets + hi + 1);
                for (auto& v : doff[d]) v -= tape->decision_offsets[lo];
                const size_t rec_words = 2 + (size_t)m->n_dof;
                tapes[d].decisions = tape->decisions + tape->decision_offsets[lo] * rec_words;
                tapes[d].decision_offsets = doff[d].data();
            }
            t = &tapes[d];
        }
        rc = fks_host::simulate_host_async(m->sims[d], starts + lo * stride, n_targets == n ? targets + lo * stride : targets,
                                           n_targets * stride, hi - lo, n_targets == n ? hi - lo : 1, n_legs, n, allow_contacts, noise_mode,
                                           t, first_particle_id + lo, (char*)results + lo * m->rec_stride, n * m->rec_stride);
    }
    for (size_t d = 0; d < G; d++) {
        const int rs = fks_sim_synchronize(m->sims[d]);
        if (rc == FKS_OK) rc = rs;
    }
    return rc;
}

int fks_multi_forward_simulate(fks_multi_sim* m, const double* starts, const double* targets, size_t n, size_t n_targets,
                               int allow_contacts, int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                               void* results) {
    return multi_simulate(m, starts, targets, n, n_targets, 1, allow_contacts, noise_mode, tape, first_particle_id, results);
}

int fks_multi_forward_simulate_sequence(fks_multi_sim* m, const double* starts, const double* targets, size_t n, size_t n_targets,
                                        size_t n_legs, int allow_contacts, int noise_mode, const fks_noise_tape* tape,
                                        uint64_t first_particle_id, void* results) {
    const int rc = fks_host::check_sequence("fks_multi_forward_simulate_sequence", targets, n, n_legs, first_particle_id);
    if (rc != FKS_OK) return rc;
    return multi_simulate(m, starts, targets, n, n_targets, n_legs, allow_contacts, noise_mode, tape, first_particle_id, results);
}

int fks_multi_forward_simulate_device(fks_multi_sim* m, const double* const* d_starts, const double* const* d_targets, size_t n,
                                      size_t n_targets, int allow_contacts, uint64_t first_particle_id, void* const* d_results) {
    if (!m || !d_starts || !d_targets || !d_results) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate_device: null argument");
    if (n == 0) return FKS_OK;
    if (!(n_targets == 1 || n_targets == n)) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate_device: need 1 target or one per start");
    const size_t G = m->devices.size();
    if (n % G != 0) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_forward_simulate_device: the all-gather needs equal shards (n divisible by the device count)");
    Nccl& nc = nccl();
    if (G > 1 && !nc.ok) return mfail(FKS_ERR_UNSUPPORTED, "fks_multi_forward_simulate_device: libnccl.so.2 not found");
    if (m->streams.empty()) {
        m->streams.assign(G, nullptr);
        for (size_t d = 0; d < G; d++) {
            cudaSetDevice(m->devices[d]);
            if (cudaStreamCreateWithFlags(&m->streams[d], cudaStreamNonBlocking) != cudaSuccess)
                return mfail(FKS_ERR_CUDA, "fks_multi_forward_simulate_device: stream creation failed");
        }
        if (G > 1) {
            m->comms.assign(G, nullptr);
            const ncclResult_t r = nc.CommInitAll(m->comms.data(), (int)G, m->devices.data());
            if (r != ncclSuccess) {
                m->comms.clear();
                return mfail(FKS_ERR_CUDA, std::string("ncclCommInitAll: ") + nc.GetErrorString(r));
            }
        }
    }
    const size_t per = n / G;
    int rc = FKS_OK;
    for (size_t d = 0; d < G && rc == FKS_OK; d++) {
        cudaSetDevice(m->devices[d]);
        // device d simulates its shard straight into its slice of its own full-size result array
        rc = fks_forward_simulate_device(m->sims[d], d_starts[d], d_targets[d], per, n_targets == n ? per : 1, allow_contacts, FKS_NOISE_PHILOX,
                                         nullptr, nullptr, first_particle_id + d * per, (char*)d_results[d] + d * per * m->rec_stride,
                                         m->streams[d]);
    }
    if (rc == FKS_OK && G > 1) {
        // in-place all-gather: rank d contributes the slice it has just written
        nc.GroupStart();
        for (size_t d = 0; d < G; d++) {
            cudaSetDevice(m->devices[d]);
            const ncclResult_t r = nc.AllGather((const char*)d_results[d] + d * per * m->rec_stride, d_results[d], per * m->rec_stride, ncclChar,
                                                m->comms[d], m->streams[d]);
            if (r != ncclSuccess && rc == FKS_OK) rc = mfail(FKS_ERR_CUDA, std::string("ncclAllGather: ") + nc.GetErrorString(r));
        }
        nc.GroupEnd();
    }
    for (size_t d = 0; d < G; d++) {
        cudaSetDevice(m->devices[d]);
        const cudaError_t e = cudaStreamSynchronize(m->streams[d]);
        if (e != cudaSuccess && rc == FKS_OK) rc = mfail(FKS_ERR_CUDA, std::string("fks_multi_forward_simulate_device: ") + cudaGetErrorString(e));
    }
    return rc;
}

int fks_multi_get_statistics(fks_multi_sim* m, uint64_t* out) {
    if (!m || !out) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_get_statistics: null argument");
    std::memset(out, 0, FKS_NUM_STATS * sizeof(uint64_t));
    for (fks_sim* s : m->sims) {
        uint64_t part[FKS_NUM_STATS];
        const int rc = fks_get_statistics(s, part);
        if (rc != FKS_OK) return rc;
        for (int k = 0; k < FKS_NUM_STATS; k++) out[k] += part[k];
    }
    return FKS_OK;
}

int fks_multi_reset_statistics(fks_multi_sim* m) {
    if (!m) return mfail(FKS_ERR_INVALID_ARGUMENT, "fks_multi_reset_statistics: null argument");
    for (fks_sim* s : m->sims) {
        const int rc = fks_reset_statistics(s);
        if (rc != FKS_OK) return rc;
    }
    return FKS_OK;
}

size_t fks_multi_sim_result_stride(const fks_multi_sim* m) { return m ? m->rec_stride : 0; }

}  // extern "C"
