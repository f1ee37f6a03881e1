// sm_100a kernels of the batched particle contact simulator.
//
// One warp simulates one particle from start to finish: the controller-step loop
// (simple_particle_contact_simulator.hpp:843-919), the microstep loop and the contact resolver
// (:1546-1816).  Lanes stride over the robot's collision points; reductions over points are warp
// shuffles / votes; D-vectors (one entry per actuated axis) live one entry per lane; link transforms
// live in shared memory.  The grid is persistent: warps pull particle ids from a global counter so
// particles that spend 26 resolver iterations per microstep do not stall their neighbours.
//
// Nothing here is a dense contraction, so no tensor cores: the contended units are the FP64 pipe and
// the LSU/L2 gather path (SDF floats through the read-only path, L2-resident via an access-policy
// window).  Design points that follow from the profile (profiles/):
//   * every piece of uniform data (robot, environment metadata, solver, launch scalars, layouts) sits in
//     a shared-memory Frame at offset 0, so device functions address it with LDS + immediate offsets
//     instead of generic loads through pointers;
//   * per link, world->voxel coordinates are ONE 3x4 transform G_l = (1/res) * inverse_origin * T_l, rebuilt
//     with the forward kinematics; the per-point collision test is 9 FMAs + 3 truncations + 1 gather;
//   * "previous" and "current" kinematic state ping-pong between two buffers (no copies);
//   * actuator noise for several microsteps is drawn at once so that all lanes do Philox/Box-Muller work;
//   * the big building blocks are single __noinline__ copies (instruction-cache footprint).
//
// Reference line numbers below (spcs = simple_particle_contact_simulator.hpp, tnuva =
// tnuva_robot_models.hpp, unc = simple_uncertainty_models.hpp, pid = simple_pid_controller.hpp)
// say WHAT each function computes; the arithmetic of the un-vendored dependencies (arc_utilities,
// sdf_tools, Eigen) is written from their documented behaviour, see DESIGN.md.

#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "fks_device_types.h"
#include "fks_philox.h"

namespace fksdev {

#define FKS_FULL 0xffffffffu
#ifndef FKS_SKIP_SINGLE_ESTIMATE
#define FKS_SKIP_SINGLE_ESTIMATE 1
#endif
#ifndef FKS_MIN_BLOCKS
#define FKS_MIN_BLOCKS 1  // lock-step CTAs per SM the register allocation is planned for
#endif

extern __shared__ __align__(16) unsigned char smem_raw[];

namespace {

constexpr double kPi = 3.14159265358979323846;

// ---- shared-memory accessors -------------------------------------------------------------------
__device__ __forceinline__ const Frame& frame() { return *reinterpret_cast<const Frame*>(smem_raw); }
__device__ __forceinline__ double* wsd(int wb) { return reinterpret_cast<double*>(smem_raw + wb); }
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ void raise_flag(int wb, unsigned bits) {
    atomicOr(reinterpret_cast<unsigned*>(wsd(wb) + frame().a.wl.flags), bits);
}
__device__ __forceinline__ void add_stat(int wb, int which, unsigned long long v) {  // lane 0 only
    reinterpret_cast<unsigned long long*>(wsd(wb) + frame().a.wl.stats)[which] += v;
}
// Read-modify-write of a per-warp bookkeeping word (WarpVars, shared memory, one copy per warp, every lane holds the same
// view): all lanes read, THEN all lanes store the same new value -- under independent thread scheduling a lane that ran
// ahead could otherwise have its store read back by a lagging lane and applied twice.
template <class T>
__device__ __forceinline__ T wv_add(T* field, T inc) {
    const T v = *field + inc;
    __syncwarp();
    *field = v;
    return v;
}

// ---- bulk copies (cp.async.bulk, 1-D TMA) between a warp's shared block and global memory -------------------------------
// Lane 0 issues them with uniform operands; the bytes move in the async proxy and occupy no registers.  Addresses and sizes
// are multiples of 16 bytes (simulate_smem_plan checks the layout).  The ordering rules they rely on, from the memory
// consistency model of the PTX ISA:
//  (a) Accesses of one location through the generic proxy (the lanes' loads and stores) and through the async proxy (bulk
//      copies) are ordered only by a proxy fence.  Every lane that touched the shared data runs fence.proxy.async.shared::cta
//      (and .global for global data it wrote), then __syncwarp orders those lanes before lane 0, which issues the bulk copy.
//      A global slot last written by a bulk store of another warp is visible to lane 0's generic proxy after the barrier
//      of simulate_kernel (rule (b)); lane 0 runs fence.proxy.async.global before its bulk load reads it.
//  (b) cp.async.bulk.wait_group.read 0 returns once the sources of the issuing thread's bulk stores have been read; before
//      that nothing may write that shared memory.  cp.async.bulk.wait_group 0 returns once the writes are complete; the
//      implicit generic-async proxy fence that follows the completion of a bulk operation makes them visible to the issuer's
//      generic proxy, and a barrier then carries them to the other threads.
//  (c) A bulk load completes transactions on the warp's mbarrier.  A lane whose mbarrier.try_wait (.acquire, CTA scope)
//      observes the phase complete sees the loaded bytes, so every lane that reads them waits itself (bulk_wait_loads).
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fence_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(double* g, const double* s, int doubles) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g), "r"(smem_u32(s)), "r"(doubles * 8)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// the warp's mbarrier in the CTA's sync area
__device__ __forceinline__ unsigned warp_bar() {
    return smem_u32(smem_raw + frame().a.sync_off + kSyncBarOff) + 8u * (threadIdx.x >> 5);
}
// lane 0: arms the mbarrier for `bytes` of bulk loads; returns the token of the phase that they complete
__device__ __forceinline__ unsigned long long bulk_expect(unsigned bar, int bytes) {
    unsigned long long state;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 %0, [%1], %2;" : "=l"(state) : "r"(bar), "r"(bytes) : "memory");
    return state;
}
__device__ __forceinline__ void bulk_load(double* s, const double* g, int doubles, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s)), "l"(g), "r"(doubles * 8), "r"(bar) : "memory");
}
// (c): every lane waits for the phase lane 0 armed (its token: no parity has to be carried from one load to the next)
__device__ __forceinline__ void bulk_wait_loads(unsigned bar, unsigned long long state) {
    state = __shfl_sync(FKS_FULL, state, 0);
    unsigned done;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "l"(state) : "memory");
    } while (!done);
}
// global scratch slot of the particle context this warp has loaded (self-collision lists: written by the collision check of
// a round, read by the collect of the following solve, which another warp may run)
__device__ __forceinline__ char* context_scratch(int wb) {
    const LaunchArgs& a = frame().a;
    const int ctx = reinterpret_cast<const WarpVars*>(wsd(wb) + a.wl.vars)->ctx;
    return a.scratch + ((size_t)blockIdx.x * a.pool + ctx) * a.sl.total;
}
// global slot of this WARP for a stacked system too tall for shared memory: written and consumed inside one solve task, so it
// belongs to the warp -- 148 x 24 slots whose touched lines stay in L2, instead of one per context
__device__ __forceinline__ double* warp_jstore() {
    const LaunchArgs& a = frame().a;
    return reinterpret_cast<double*>(a.jscratch + ((size_t)blockIdx.x * a.warps_per_block + (threadIdx.x >> 5)) * a.sl.jtotal);
}

// ForwardSimulationStepTrace (spcs:1583-1617, :1703, :1714, :1778), flat: one record per assignment / push_back of the
// reference.  Only reached when the call asked for a trace (a.trace != nullptr, one particle).
__device__ __noinline__ void trace_append(unsigned kind, unsigned step, unsigned micro, unsigned iter, const double* values, int n) {
    const LaunchArgs& a = frame().a;
    const int lane = lane_id();
    unsigned idx = 0u;
    if (lane == 0) idx = atomicAdd(a.trace_count, 1u);
    idx = __shfl_sync(FKS_FULL, idx, 0);
    if (idx >= a.trace_capacity) return;
    char* rec = a.trace + (size_t)idx * (sizeof(fks_trace_header) + (size_t)a.trace_width * 8);
    if (lane == 0) {
        fks_trace_header h;
        h.kind = kind;
        h.step = step;
        h.microstep = micro;
        h.iteration = iter;
        *reinterpret_cast<fks_trace_header*>(rec) = h;
    }
    double* v = reinterpret_cast<double*>(rec + sizeof(fks_trace_header));
    for (int i = lane; i < a.trace_width; i += 32) v[i] = i < n ? values[i] : 0.0;
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FKS_FULL, v, o));
    return v;
}

// EigenHelpers::EnforceContinuousRevoluteBounds: wrap to (-pi, pi]
__device__ __forceinline__ double wrap_angle(double value) {
    if ((value <= -kPi) || (value > kPi)) {
        const double remainder = fmod(value, 2.0 * kPi);
        if (remainder <= -kPi) return remainder + (2.0 * kPi);
        if (remainder > kPi) return remainder - (2.0 * kPi);
        return remainder;
    }
    return value;
}

// (T is 16-byte aligned wherever it lives: 128-bit loads halve the shared-memory instructions and wavefronts of the point loops)
__device__ __forceinline__ void apply_T(const double* T, double x, double y, double z, double& ox, double& oy, double& oz) {
    const double2 t01 = *reinterpret_cast<const double2*>(T + 0), t23 = *reinterpret_cast<const double2*>(T + 2);
    const double2 t45 = *reinterpret_cast<const double2*>(T + 4), t67 = *reinterpret_cast<const double2*>(T + 6);
    const double2 t89 = *reinterpret_cast<const double2*>(T + 8), tab = *reinterpret_cast<const double2*>(T + 10);
    ox = t01.x * x + t01.y * y + t23.x * z + t23.y;
    oy = t45.x * x + t45.y * y + t67.x * z + t67.y;
    oz = t89.x * x + t89.y * y + tab.x * z + tab.y;
}

// Quaterniond(AngleAxisd(angle, axis)).toRotationMatrix(), translation zero
__device__ __forceinline__ void rot_axis(double angle, double ax, double ay, double az, double* R) {
    double s, w;
    sincos(0.5 * angle, &s, &w);
    const double x = s * ax, y = s * ay, z = s * az;
    const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1.0 - (tyy + tzz);
    R[1] = txy - twz;
    R[2] = txz + twy;
    R[3] = 0.0;
    R[4] = txy + twz;
    R[5] = 1.0 - (txx + tzz);
    R[6] = tyz - twx;
    R[7] = 0.0;
    R[8] = txz - twy;
    R[9] = tyz + twx;
    R[10] = 1.0 - (txx + tyy);
    R[11] = 0.0;
}

// C = A * B for rigid transforms stored row-major 3x4
__device__ __forceinline__ void iso_mul(const double* A, const double* B, double* C) {
#pragma unroll
    for (int r = 0; r < 3; r++) {
#pragma unroll
        for (int c = 0; c < 3; c++) C[4 * r + c] = A[4 * r + 0] * B[c] + A[4 * r + 1] * B[4 + c] + A[4 * r + 2] * B[8 + c];
        C[4 * r + 3] = A[4 * r + 0] * B[3] + A[4 * r + 1] * B[7] + A[4 * r + 2] * B[11] + A[4 * r + 3];
    }
}
__device__ __forceinline__ void iso_inverse(const double* A, double* C) {
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) C[4 * r + c] = A[4 * c + r];
#pragma unroll
    for (int r = 0; r < 3; r++) C[4 * r + 3] = -(C[4 * r + 0] * A[3] + C[4 * r + 1] * A[7] + C[4 * r + 2] * A[11]);
}

// EigenHelpers::ExpTwist(twist, 1.0) (call sites tnuva:360,378): twist = (v, w)
__device__ __forceinline__ void exp_twist(const double* tw, double* T) {
    const double rn = sqrt(tw[3] * tw[3] + tw[4] * tw[4] + tw[5] * tw[5]);
#pragma unroll
    for (int i = 0; i < 12; i++) T[i] = (i % 5 == 0) ? 1.0 : 0.0;
    if (rn >= 1e-100) {
        const double theta = rn * 1.0;
        const double svx = tw[0] / rn, svy = tw[1] / rn, svz = tw[2] / rn;
        const double wx = tw[3] / rn, wy = tw[4] / rn, wz = tw[5] / rn;
        double s, c;
        sincos(theta, &s, &c);
        const double c1 = 1.0 - c;
        const double K[9] = {0.0, -wz, wy, wz, 0.0, -wx, -wy, wx, 0.0};
        double K2[9], R[9];
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int cc = 0; cc < 3; cc++) K2[3 * r + cc] = K[3 * r + 0] * K[cc] + K[3 * r + 1] * K[3 + cc] + K[3 * r + 2] * K[6 + cc];
#pragma unroll
        for (int i = 0; i < 9; i++) R[i] = ((i % 4 == 0) ? 1.0 : 0.0) + (K[i] * s) + (K2[i] * c1);
        const double cxv[3] = {wy * svz - wz * svy, wz * svx - wx * svz, wx * svy - wy * svx};
        const double wv = wx * svx + wy * svy + wz * svz;
        const double wa[3] = {wx, wy, wz};
#pragma unroll
        for (int r = 0; r < 3; r++) {
            double acc = 0.0;
#pragma unroll
            for (int cc = 0; cc < 3; cc++) acc += (((r == cc) ? 1.0 : 0.0) - R[3 * r + cc]) * cxv[cc];
            T[4 * r + 3] = acc + (wa[r] * wv) * theta;
#pragma unroll
            for (int cc = 0; cc < 3; cc++) T[4 * r + cc] = R[3 * r + cc];
        }
    } else {
        T[3] = tw[0];
        T[7] = tw[1];
        T[11] = tw[2];
    }
}

__device__ __forceinline__ void safe_normal3(double& x, double& y, double& z) {
    const double n = sqrt(x * x + y * y + z * z);
    if (n > DBL_EPSILON) {
        x = x / n;
        y = y / n;
        z = z / n;
    }
}

// EigenHelpers::TwistBetweenTransforms(a, b) = unhat(log(a^-1 b)) (call site tnuva:389), closed form
__device__ __noinline__ void twist_between(const double* a, const double* b, double* twist) {
    double ai[12], Dm[12];
    iso_inverse(a, ai);
    iso_mul(ai, b, Dm);
    const double tr = Dm[0] + Dm[5] + Dm[10];
    const double axx = Dm[9] - Dm[6], axy = Dm[2] - Dm[8], axz = Dm[4] - Dm[1];
    const double s2 = sqrt(axx * axx + axy * axy + axz * axz);
    const double c = 0.5 * (tr - 1.0);
    const double theta = atan2(0.5 * s2, c);
    const double tx = Dm[3], ty = Dm[7], tz = Dm[11];
    double wx, wy, wz;
    if (theta < 1e-9) {
        wx = axx * 0.5;
        wy = axy * 0.5;
        wz = axz * 0.5;
        twist[0] = tx - (wy * tz - wz * ty) * 0.5;
        twist[1] = ty - (wz * tx - wx * tz) * 0.5;
        twist[2] = tz - (wx * ty - wy * tx) * 0.5;
        twist[3] = wx;
        twist[4] = wy;
        twist[5] = wz;
        return;
    }
    if (kPi - theta < 1e-6) {
        double xx = sqrt(fmax(0.0, 0.5 * (Dm[0] + 1.0)));
        double yy = sqrt(fmax(0.0, 0.5 * (Dm[5] + 1.0)));
        double zz = sqrt(fmax(0.0, 0.5 * (Dm[10] + 1.0)));
        if (xx >= yy && xx >= zz) {
            if (Dm[1] + Dm[4] < 0.0) yy = -yy;
            if (Dm[2] + Dm[8] < 0.0) zz = -zz;
            if (axx < 0.0) { xx = -xx; yy = -yy; zz = -zz; }
        } else if (yy >= zz) {
            if (Dm[1] + Dm[4] < 0.0) xx = -xx;
            if (Dm[6] + Dm[9] < 0.0) zz = -zz;
            if (axy < 0.0) { xx = -xx; yy = -yy; zz = -zz; }
        } else {
            if (Dm[2] + Dm[8] < 0.0) xx = -xx;
            if (Dm[6] + Dm[9] < 0.0) yy = -yy;
            if (axz < 0.0) { xx = -xx; yy = -yy; zz = -zz; }
        }
        safe_normal3(xx, yy, zz);
        wx = xx * theta;
        wy = yy * theta;
        wz = zz * theta;
    } else {
        const double f = theta / s2;
        wx = axx * f;
        wy = axy * f;
        wz = axz * f;
    }
    double st, ct;
    sincos(theta, &st, &ct);
    const double k = (1.0 - (theta * st) / (2.0 * (1.0 - ct))) / (theta * theta);
    const double wxtx = wy * tz - wz * ty, wxty = wz * tx - wx * tz, wxtz = wx * ty - wy * tx;
    const double wwx = wy * wxtz - wz * wxty, wwy = wz * wxtx - wx * wxtz, wwz = wx * wxty - wy * wxtx;
    twist[0] = tx - wxtx * 0.5 + wwx * k;
    twist[1] = ty - wxty * 0.5 + wwy * k;
    twist[2] = tz - wxtz * 0.5 + wwz * k;
    twist[3] = wx;
    twist[4] = wy;
    twist[5] = wz;
}

// robot->ComputeConfigurationDistanceTo(target) (the call at spcs:898; the robot classes are upstream, so this follows the
// oracle's restatement `Robot::distance_to`): SE2 / SE3 weigh translation and rotation angle, the linked robot takes the
// weighted joint-space norm with continuous joints wrapped.
template <int KIND>
__device__ __forceinline__ double config_distance(const DevRobot& rb, const double* cur, const double* target) {
    if (KIND == FKS_ROBOT_SE2) {
        const double dx = fabs(target[0] - cur[0]), dy = fabs(target[1] - cur[1]);
        const double dr = fabs(wrap_angle(target[2] - cur[2]));
        return (sqrt(dx * dx + dy * dy) * rb.pos_w) + (dr * rb.rot_w);
    } else if (KIND == FKS_ROBOT_SE3) {
        double c12[12], tg[12], ci[12], Dm[12];
#pragma unroll
        for (int i = 0; i < 12; i++) {
            c12[i] = cur[i];
            tg[i] = target[i];
        }
        const double dx = tg[3] - c12[3], dy = tg[7] - c12[7], dz = tg[11] - c12[11];
        iso_inverse(c12, ci);
        iso_mul(ci, tg, Dm);
        const double cs = fmin(fmax(0.5 * (Dm[0] + Dm[5] + Dm[10] - 1.0), -1.0), 1.0);
        return (sqrt(dx * dx + dy * dy + dz * dz) * rb.pos_w) + (acos(cs) * rb.rot_w);
    } else {
        double sacc = 0.0;
        for (int j = 0; j < rb.J; j++) {
            const DevJoint& jd = rb.joints[j];
            if (jd.active < 0) continue;
            double dj = target[jd.active] - cur[jd.active];
            if (jd.type == FKS_JOINT_CONTINUOUS) dj = wrap_angle(dj);
            const double wd = dj * jd.weight;
            sacc += wd * wd;
        }
        return sqrt(sacc);
    }
}

// TruncatedNormalUncertainVelocityActuator::GetControlValue (unc:70-75 noiseless, :77-90 noisy)
__device__ __forceinline__ double actuate(int wb, const DevAxis& ax, double u, bool noisy, double tn) {
    if (isnan(u) || isinf(u)) raise_flag(wb, FKS_FLAG_WOULD_ASSERT_NAN);  // assert unc:72-73
    const double vl = ax.vlim;
    const double real_u = fmin(fmax(u, -vl), vl);
    if (!noisy) return real_u;
    const double pb = ax.pnoise * fabs(real_u);
    const double mb = ax.mnoise * vl;
    const double bound = fmax(pb, mb);
    return real_u + tn * bound;
}

// ------------------------------------------------------------------------------------------------
// Kinematic state X: SetPosition (call sites spcs:875,1423-1424,1601).  Reads cfg[X] (wraps / clamps it in
// place), writes T[X].  derive != 0 additionally rebuilds what the collision checks of the CURRENT state
// read: G (world -> voxel transform per link) and the world end points of the link capsules.
// ------------------------------------------------------------------------------------------------
template <int KIND>
__device__ __noinline__ void kinematics(int wb, int X, int derive) {
    const Frame& fr = frame();
    const WarpLayout& wl = fr.a.wl;
    const DevRobot& rb = fr.rb;
    const int lane = lane_id();
    double* ws = wsd(wb);
    double* cfg = ws + wl.cfg + X * wl.S;
    double* T = ws + wl.T + X * wl.L12;
    if (KIND == FKS_ROBOT_SE2) {
        if (lane == 0) {
            const double th = wrap_angle(cfg[2]);
            cfg[2] = th;
            double R[12];
            rot_axis(th, 0.0, 0.0, 1.0, R);
            R[3] = cfg[0];
            R[7] = cfg[1];
            R[11] = 0.0;
#pragma unroll
            for (int i = 0; i < 12; i++) T[i] = R[i];
        }
        __syncwarp();
    } else if (KIND == FKS_ROBOT_SE3) {
        if (lane < 12) T[lane] = cfg[lane];
        __syncwarp();
    } else {
        double* M = ws + wl.M;
        // one joint per lane: value (wrap / clamp) and its sine / one-minus-cosine (prismatic: the value itself / 0) ...
        double* sc = ws + wl.jaxis;  // 2 J doubles; collect_corrections refills jaxis whenever it needs it
        for (int j = lane; j < rb.J; j += 32) {
            const DevJoint& jd = rb.joints[j];
            double s1 = 0.0, s2 = 0.0;
            if (jd.active >= 0) {
                double v = cfg[jd.active];
                if (jd.type == FKS_JOINT_CONTINUOUS) {
                    v = wrap_angle(v);
                } else {
                    if (v > jd.hi) v = jd.hi;
                    else if (v < jd.lo) v = jd.lo;
                }
                cfg[jd.active] = v;
                if (jd.type == FKS_JOINT_PRISMATIC) {
                    s1 = v;
                } else {
                    double c;
                    sincos(v, &s1, &c);
                    s2 = 1.0 - c;
                }
            }
            sc[2 * j] = s1;
            sc[2 * j + 1] = s2;
        }
        __syncwarp();
        // ... then all lanes build M_j = J_t + s1 (J_t K) + s2 (J_t K^2), one matrix element each (fks_robot_create)
        for (int el = lane; el < 12 * rb.J; el += 32) {
            const int j = el / 12, e = el - 12 * j;
            const DevJoint& jd = rb.joints[j];
            M[16 * j + 4 * (e & 3) + (e >> 2)] = jd.T[e] + sc[2 * j] * jd.C1[e] + sc[2 * j + 1] * jd.C2[e];  // stored by columns
        }
        // chain T_child = T_parent * M_j on lanes 0..11; lanes 12..23 run the SAME recurrence from the root
        // (1 / res) * inverse_origin * base, which yields the world->voxel transforms G_l = (1 / res) * inverse_origin * T_l
        // in the same instructions (they were a separate pass of 3 x 12 L products)
        double* G = ws + wl.G;
        if (lane < 12) T[lane] = rb.base[lane];
        else if (lane < 24 && derive) G[lane - 12] = fr.gbase[lane - 12];
        __syncwarp();
        const int e12 = lane < 12 ? lane : lane - 12;
        const int r = e12 >> 2, cc = e12 & 3;
        double* chain = lane < 12 ? T : G;
        const bool in_chain = lane < 12 || (lane < 24 && derive);
        unsigned long long parents = rb.joint_parents, children = rb.joint_children;  // one nibble per joint
        for (int j = 0; j < rb.J; j++, parents >>= 4, children >>= 4) {
            if (in_chain) {
                // row r of the parent transform and column cc of the joint matrix, two 128-bit loads each
                const double* Tp = chain + 12 * (int)(parents & 0xFull) + 4 * r;
                const double* Mc = M + 16 * j + 4 * cc;
                const double2 t01 = *reinterpret_cast<const double2*>(Tp), t23 = *reinterpret_cast<const double2*>(Tp + 2);
                const double2 m01 = *reinterpret_cast<const double2*>(Mc), m23 = *reinterpret_cast<const double2*>(Mc + 2);
                double v = t01.x * m01.x + t01.y * m01.y + t23.x * m23.x;
                if (cc == 3) v += t23.y;
                chain[12 * (int)(children & 0xFull) + e12] = v;
            }
            __syncwarp();
        }
    }
    if (derive) {
        const DevEnv& e = fr.a.env;
        double* G = ws + wl.G;
        if (KIND != FKS_ROBOT_LINKED)
        for (int el = lane; el < wl.L12; el += 32) {
            const int l = el / 12, rc = el - 12 * l, r = rc >> 2, cc = rc & 3;
            const double* Tl = T + 12 * l;
            double v = e.inv_origin[4 * r + 0] * Tl[cc] + e.inv_origin[4 * r + 1] * Tl[4 + cc] + e.inv_origin[4 * r + 2] * Tl[8 + cc];
            if (cc == 3) v += e.inv_origin[4 * r + 3];
            G[el] = v * e.inv_sdf_res;
        }
        if (KIND == FKS_ROBOT_LINKED && rb.n_pairs > 0) {
            double* caps = ws + wl.caps;
            for (int q = lane; q < 2 * rb.L; q += 32) {
                const int l = q >> 1;
                const double* cp = (q & 1) ? rb.cap_p1[l] : rb.cap_p0[l];
                double x, y, z;
                apply_T(T + 12 * l, cp[0], cp[1], cp[2], x, y, z);
                caps[3 * q] = x;
                caps[3 * q + 1] = y;
                caps[3 * q + 2] = z;
            }
        }
        __syncwarp();
    }
}

// ApplyControlInput(input[, rng]) (tnuva:152-177 SE2, :348-382 SE3, :538-596 linked): state Xout = state Xin
// advanced by u (shared vector at offset u_off); tn_off < 0 selects the noiseless overload.  Xin == Xout allowed.
template <int KIND>
__device__ __noinline__ void apply_control(int wb, int Xin, int Xout, int u_off, int tn_off, int derive) {
    const Frame& fr = frame();
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    double* ws = wsd(wb);
    const double* cin = ws + wl.cfg + Xin * wl.S;
    double* cout = ws + wl.cfg + Xout * wl.S;
    const bool noisy = tn_off >= 0;
    if (KIND == FKS_ROBOT_SE3) {
        double* qr = ws + wl.qr;  // free outside the QR solve: holds the actuated twist
        if (lane < 6) qr[lane] = actuate(wb, fr.rb.axes[lane], ws[u_off + lane], noisy, noisy ? ws[tn_off + lane] : 0.0);
        __syncwarp();
        double tw[6], E[12], A[12], Cm[12];
#pragma unroll
        for (int i = 0; i < 6; i++) tw[i] = qr[i];
        exp_twist(tw, E);
#pragma unroll
        for (int i = 0; i < 12; i++) A[i] = cin[i];
        iso_mul(A, E, Cm);
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 12; i++) cout[i] = Cm[i];
        }
        __syncwarp();
    } else {
        if (lane < fr.rb.D) cout[lane] = cin[lane] + actuate(wb, fr.rb.axes[lane], ws[u_off + lane], noisy, noisy ? ws[tn_off + lane] : 0.0);
        __syncwarp();
    }
    kinematics<KIND>(wb, Xout, derive);
}

// ------------------------------------------------------------------------------------------------
// environment queries
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sdf_cell(const DevEnv& e, int x, int y, int z) {
    return __ldg(e.sdf + ((x * e.ny + y) * e.nz + z));
}

#ifndef FKS_COLLECT_ESTIMATE
#define FKS_COLLECT_ESTIMATE estimate_distance_inl
#endif
// SignedDistanceField::EstimateDistance4d for an in-bounds point whose cell (x,y,z) holds d0f
__device__ __forceinline__ double estimate_distance_inl(double wx, double wy, double wz, int x, int y, int z, float d0f) {
    const DevEnv& e = frame().a.env;
    const double res = e.sdf_res;
    const double d0 = (double)d0f;
    const double dc = (d0 >= 0.0) ? d0 - (res * 0.5) : d0 + (res * 0.5);
    double g0, g1, g2;
    if (x > 0 && y > 0 && z > 0 && x < e.nx - 1 && y < e.ny - 1 && z < e.nz - 1) {
        g0 = (double)(sdf_cell(e, x + 1, y, z) - sdf_cell(e, x - 1, y, z)) * e.inv_twice_res;
        g1 = (double)(sdf_cell(e, x, y + 1, z) - sdf_cell(e, x, y - 1, z)) * e.inv_twice_res;
        g2 = (double)(sdf_cell(e, x, y, z + 1) - sdf_cell(e, x, y, z - 1)) * e.inv_twice_res;
    } else {
        const int lx = max(0, x - 1), hx = min(e.nx - 1, x + 1);
        const int ly = max(0, y - 1), hy = min(e.ny - 1, y + 1);
        const int lz = max(0, z - 1), hz = min(e.nz - 1, z + 1);
        const double sx = (double)(hx - lx) * res, sy = (double)(hy - ly) * res, sz = (double)(hz - lz) * res;
        g0 = g1 = g2 = 0.0;
        if (sx > 0.0) g0 = ((double)sdf_cell(e, hx, y, z) - (double)sdf_cell(e, lx, y, z)) * (1.0 / sx);
        if (sy > 0.0) g1 = ((double)sdf_cell(e, x, hy, z) - (double)sdf_cell(e, x, ly, z)) * (1.0 / sy);
        if (sz > 0.0) g2 = ((double)sdf_cell(e, x, y, hz) - (double)sdf_cell(e, x, y, lz)) * (1.0 / sz);
    }
    const double cgx = res * ((double)x + 0.5), cgy = res * ((double)y + 0.5), cgz = res * ((double)z + 0.5);
    double cx, cy, cz;
    apply_T(e.origin, cgx, cgy, cgz, cx, cy, cz);
    const double vx = wx - cx, vy = wy - cy, vz = wz - cz;
    const double gg = g0 * g0 + g1 * g1 + g2 * g2;
    double adj = 0.0;
    if (gg > 0.0) adj = (vx * g0 + vy * g1 + vz * g2) / sqrt(gg);
    return dc + adj;
}
// out-of-line copy for the rare second tier of check_env; collect_corrections inlines the body (a call there spills a
// dozen live doubles around it)
__device__ __noinline__ double estimate_distance(double wx, double wy, double wz, int x, int y, int z, float d0f) {
    return estimate_distance_inl(wx, wy, wz, x, y, z, d0f);
}

// voxel of a link-relative point through the composite transform G_l; false when out of bounds.
// VoxelGrid::LocationToGridIndex semantics: C-cast truncation of grid coordinate / cell size.
struct Voxel {
    int x, y, z;
    bool inb;
};
__device__ __forceinline__ Voxel voxel_of(const DevEnv& e, const double* Gl, double px, double py, double pz) {
    const double2 g01 = *reinterpret_cast<const double2*>(Gl + 0), g23 = *reinterpret_cast<const double2*>(Gl + 2);
    const double2 g45 = *reinterpret_cast<const double2*>(Gl + 4), g67 = *reinterpret_cast<const double2*>(Gl + 6);
    const double2 g89 = *reinterpret_cast<const double2*>(Gl + 8), gab = *reinterpret_cast<const double2*>(Gl + 10);
    const double gx = g01.x * px + g01.y * py + g23.x * pz + g23.y;
    const double gy = g45.x * px + g45.y * py + g67.x * pz + g67.y;
    const double gz = g89.x * px + g89.y * py + gab.x * pz + gab.y;
    Voxel v;
    v.x = (int)gx;
    v.y = (int)gy;
    v.z = (int)gz;
    v.inb = ((unsigned)v.x < (unsigned)e.nx) && ((unsigned)v.y < (unsigned)e.ny) && ((unsigned)v.z < (unsigned)e.nz);
    return v;
}

constexpr int kBatch = 4;       // independent SDF gathers in flight per lane

// Link-level culling.  SDF cell values are exact Euclidean distances between cell centres, hence 1-Lipschitz over
// cell centres; a point p of a link and the link's sphere centre q lie within sqrt(3)/2 res of their cells' centres,
// so  raw(cell(p)) >= raw(cell(q)) - R - sqrt(3) res.  A link whose centre cell value exceeds R + sqrt(3) res + `need`
// cannot hold a point with raw value < `need`: all of its points are skipped.  Out-of-bounds centres never cull.
__device__ __forceinline__ unsigned active_links(const DevEnv& e, const DevRobot& rb, const double* G, double need) {
    const int lane = lane_id();
    bool active = false;
    if (lane < rb.L) {
        active = true;
        const Voxel v = voxel_of(e, G + 12 * lane, rb.sph_center[lane][0], rb.sph_center[lane][1], rb.sph_center[lane][2]);
        if (v.inb) {
            const double f = (double)sdf_cell(e, v.x, v.y, v.z);
            const double reach = rb.sph_radius[lane] * (1.0 + 1e-6) + (1.7320508075688772 * (1.0 + 1e-5)) * e.sdf_res + need;
            active = !(f > reach);
        }
    }
    return __ballot_sync(FKS_FULL, active);
}
#ifndef FKS_CAND_SHARED
#define FKS_CAND_SHARED 32
#endif
constexpr int kCandShared = FKS_CAND_SHARED;  // candidate points of collect_corrections kept in shared memory (<= 32)

// second tier of the environment check (spcs:967-975) for the listed points {point index, raw cell value}: one point per
// lane, so the six extra gathers of every EstimateDistance4d are in flight together
__device__ __noinline__ bool check_env_second_tier(int wb, int X, const uint2* list, int n, double thr) {
    const Frame& fr = frame();
    const DevEnv& e = fr.a.env;
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    const double* ws = wsd(wb);
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + fr.a.P);
    bool hit = false;
    if (lane < n) {
        const uint2 rec = list[lane];
        const double2 xy = pxy[rec.x];
        const PointZL zl = pzl[rec.x];
        const Voxel v = voxel_of(e, ws + wl.G + 12 * zl.link, xy.x, xy.y, zl.z);  // same arithmetic as the first tier: same voxel
        if (!v.inb) {
            hit = true;  // an out-of-bounds value this low: EstimateDistance4d returns it too
        } else {
            double wx, wy, wz;
            apply_T(ws + wl.T + X * wl.L12 + 12 * zl.link, xy.x, xy.y, zl.z, wx, wy, wz);
            hit = estimate_distance(wx, wy, wz, v.x, v.y, v.z, __uint_as_float(rec.y)) < thr;
        }
    }
    return __any_sync(FKS_FULL, hit);
}

// CheckEnvironmentCollision (spcs:921-981) of the CURRENT state (G and T[X]); collision_threshold = 0.0 on the simulation
// path (spcs:424), inflation_ratio * resolution for CheckConfigCollision (spcs:1403).  The result is an OR over the points
// (the reference returns at the first hit, spcs:963,974): a point deep inside ends the check at once; points in the second
// tier (raw value between the two thresholds: their cell touches the surface) are only LISTED -- a link resting on a
// surface has dozens of them -- and evaluated a warp-load at a time.
__device__ __noinline__ bool check_env(int wb, int X, int use_cull, double collision_threshold) {
    const Frame& fr = frame();
    const DevEnv& e = fr.a.env;
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    double* ws = wsd(wb);
    const double* G = ws + wl.G;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + fr.a.P);
    const double res = e.sdf_res;
    const double thr = collision_threshold - (fr.a.sp.check_tolerance * res);
    const double thr_deep = thr - res;
    const float oob = e.oob;
    uint2* list = reinterpret_cast<uint2*>(ws + wl.cand);  // the candidate records of collect_corrections are not live here
    int nlist = 0;
    // points of culled links cannot collide (and an out-of-bounds value below the threshold disables culling)
    const DevRobot& rb = fr.rb;
    unsigned links = (!use_cull || !e.cull || (double)oob < thr) ? ((1u << rb.L) - 1u) : active_links(e, rb, G, thr > 0.0 ? thr : 0.0);
    // walk the runs of consecutive active links (one contiguous point range each), kBatch x 32 points -- kBatch
    // independent gathers per lane -- at a time
    // ... the DISTAL run first: the answer is a disjunction over the points, so the order is free, and a serial chain touches
    // things with its far end more often than with its base -- a colliding configuration is then settled on the first run
    bool first_run = true;
    while (links) {
        const int last = 31 - __clz(links);                     // highest active link
        const int len = __clz(~(links << (31 - last)));         // length of the run of active links that ends there
        const int first = last - len + 1;
        links &= ~(((len >= 32) ? 0xffffffffu : ((1u << len) - 1u)) << first);
        const int end = rb.link_begin[first + len];
        for (int pos = rb.link_begin[first]; pos < end; pos += 32 * kBatch) {
            float f[kBatch];
#pragma unroll
            for (int k = 0; k < kBatch; k++) {
                const int p = pos + 32 * k + lane;
                f[k] = INFINITY;  // padding lanes and (with the usual +inf oob value) out-of-bounds points: no collision
                if (p < end) {
                    const double2 xy = pxy[p];
                    const PointZL zl = pzl[p];
                    const Voxel v = voxel_of(e, G + 12 * zl.link, xy.x, xy.y, zl.z);
                    f[k] = v.inb ? sdf_cell(e, v.x, v.y, v.z) : oob;
                }
            }
            bool deep = false;
#pragma unroll
            for (int k = 0; k < kBatch; k++) deep = deep || ((double)f[k] < thr_deep);
            if (__any_sync(FKS_FULL, deep)) return true;  // deep inside (or an oob value this low, spcs:943-964)
#pragma unroll
            for (int k = 0; k < kBatch; k++) {
                const bool second = (double)f[k] < thr;
                const unsigned m = __ballot_sync(FKS_FULL, second);
                if (m == 0u) continue;
                if (nlist + __popc(m) > 32) {  // the list is full: evaluate it before it grows
                    __syncwarp();
                    if (check_env_second_tier(wb, X, list, nlist, thr)) return true;
                    nlist = 0;
                }
                if (second) list[nlist + __popc(m & ((1u << lane) - 1u))] = make_uint2((unsigned)(pos + 32 * k + lane), __float_as_uint(f[k]));
                nlist += __popc(m);
            }
        }
        if (first_run && links != 0u && nlist > 0) {  // near-surface points on the distal run: look at them before walking on
            __syncwarp();
            if (check_env_second_tier(wb, X, list, nlist, thr)) return true;
            nlist = 0;
        }
        first_run = false;
    }
    __syncwarp();
    return nlist > 0 && check_env_second_tier(wb, X, list, nlist, thr);
}

// EstimateMaxControlInputWorkspaceMotion(start_robot, end_robot) (spcs:1492-1527) between states Xa and Xb
__device__ __noinline__ double max_motion(int wb, int Xa, int Xb) {
    const Frame& fr = frame();
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    double* ws = wsd(wb);
    const double* Ta = ws + wl.T + Xa * wl.L12;
    double* Tb = ws + wl.T + Xb * wl.L12;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + fr.a.P);
    const int P = fr.a.P;
    // T_b p - T_a p = (T_b - T_a) [p; 1]: the difference of the link transforms is formed once (in place: state Xb is the
    // scratch state of the motion estimates and is not read again), which halves the work per point
    for (int el = lane; el < wl.L12; el += 32) Tb[el] = Tb[el] - Ta[el];
    __syncwarp();
    double mx = 0.0;
#pragma unroll 2
    for (int p = lane; p < P; p += 32) {
        const double2 xy = pxy[p];
        const PointZL zl = pzl[p];
        double dx, dy, dz;
        apply_T(Tb + 12 * zl.link, xy.x, xy.y, zl.z, dx, dy, dz);
        const double sq = dx * dx + dy * dy + dz * dz;
        if (sq > mx) mx = sq;
    }
    return sqrt(warp_max(mx));
}

// SurfaceNormalGrid::LookupSurfaceNormal + GetBestSurfaceNormal (spcs:186-198,235-256,111-132) for the
// in-bounds cell `li`; (dx,dy,dz) is the SafeNormal'd motion direction.
// SurfaceNormalGrid::LookupSurfaceNormal + GetBestSurfaceNormal (spcs:186-198,235-256,111-132).
// The hash probe is split from the selection so that its (dependent) loads can be issued before the
// EstimateDistance gathers of the same point and consumed after them.
__device__ __forceinline__ uint2 normal_range_probe(const DevEnv& e, long long li) {
    const unsigned long long key = (unsigned long long)li + 1ull;
    unsigned long long h = normal_hash((unsigned long long)li) & e.nh_mask;
    while (true) {
        const ulonglong2 ent = __ldg(reinterpret_cast<const ulonglong2*>(e.nh_keys) + h);  // {key, start | count << 32}
        if (ent.x == key) return make_uint2((unsigned)(ent.y & 0xFFFFFFFFull), (unsigned)(ent.y >> 32));
        if (ent.x == 0ull) return make_uint2(0u, 0u);
        h = (h + 1ull) & e.nh_mask;
    }
}
// (dx,dy,dz) is the SafeNormal'd motion direction
__device__ __forceinline__ void select_normal(int wb, const DevEnv& e, uint2 range, double dx, double dy, double dz,
                                              double& nx, double& ny, double& nz) {
    nx = ny = nz = 0.0;
    if (range.y == 0u) return;  // empty cell -> zero normal
    const double dn = sqrt(dx * dx + dy * dy + dz * dz);
    double ux = 0.0, uy = 0.0, uz = 0.0;
    if (dn > 0.0) {
        ux = dx / dn;
        uy = dy / dn;
        uz = dz / dn;
    } else {
        raise_flag(wb, FKS_FLAG_WOULD_ASSERT_NORMAL);  // assert(direction_norm > 0.0) spcs:115
    }
    double best_dot = -INFINITY;
    for (unsigned en = range.x; en < range.x + range.y; en++) {
        const double2* q = reinterpret_cast<const double2*>(e.normal_entries + 6 * (size_t)en);
        const double2 q01 = __ldg(q), q23 = __ldg(q + 1), q45 = __ldg(q + 2);
        const double dp = q01.x * ux + q01.y * uy + q23.x * uz;
        if (dp > best_dot) {  // strict: the first maximum wins (spcs:119-128)
            best_dot = dp;
            nx = q23.y;
            ny = q45.x;
            nz = q45.y;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// self collisions: CollectSelfCollisions (spcs:1183-1275) + ExtractSelfCollidingPoints (spcs:983-1171)
//
// The cell keys truncate toward zero (LocationToExtendedGridIndex, spcs:1173-1181: (int64_t)(coordinate / resolution)), so
// the cells at index 0 are TWICE as wide per axis (-res .. +res): two points share a cell only if they are within
// 2 sqrt(3) map_res of each other.  A capsule test over the DISALLOWED link pairs with that bound decides exactly when the
// hash-grid pass can be skipped (the common case).  The exact pass keeps the reference's per-cell semantics.  Returns true when at least one
// point received a correction (self_collision_map non-empty); corrections are left in the scratch slot's
// selfcorr array, per-point flags in sflag (bit 0).
// ------------------------------------------------------------------------------------------------

// squared distance between segments [p1,q1] and [p2,q2] (clamped closest points; degenerate segments allowed)
__device__ __forceinline__ double segment_distance_sq(const double* p1, const double* q1, const double* p2, const double* q2) {
    const double d1x = q1[0] - p1[0], d1y = q1[1] - p1[1], d1z = q1[2] - p1[2];
    const double d2x = q2[0] - p2[0], d2y = q2[1] - p2[1], d2z = q2[2] - p2[2];
    const double rx = p1[0] - p2[0], ry = p1[1] - p2[1], rz = p1[2] - p2[2];
    const double a = d1x * d1x + d1y * d1y + d1z * d1z;
    const double ee = d2x * d2x + d2y * d2y + d2z * d2z;
    const double f = d2x * rx + d2y * ry + d2z * rz;
    const double tiny = 1e-300;
    double s, t;
    if (a <= tiny && ee <= tiny) {
        s = t = 0.0;
    } else if (a <= tiny) {
        s = 0.0;
        t = fmin(fmax(f / ee, 0.0), 1.0);
    } else {
        const double cc = d1x * rx + d1y * ry + d1z * rz;
        if (ee <= tiny) {
            t = 0.0;
            s = fmin(fmax(-cc / a, 0.0), 1.0);
        } else {
            const double bb = d1x * d2x + d1y * d2y + d1z * d2z;
            const double denom = a * ee - bb * bb;
            s = (denom > 0.0) ? fmin(fmax((bb * f - cc * ee) / denom, 0.0), 1.0) : 0.0;
            t = (bb * s + f) / ee;
            if (t < 0.0) {
                t = 0.0;
                s = fmin(fmax(-cc / a, 0.0), 1.0);
            } else if (t > 1.0) {
                t = 1.0;
                s = fmin(fmax((bb - cc) / a, 0.0), 1.0);
            }
        }
    }
    const double cx = (p1[0] + d1x * s) - (p2[0] + d2x * t), cy = (p1[1] + d1y * s) - (p2[1] + d2y * t), cz = (p1[2] + d1z * s) - (p2[2] + d2z * t);
    return cx * cx + cy * cy + cz * cz;
}

struct SelfCtx {
    unsigned cand_pairs[kPairChunks];
    unsigned cand_links;
    unsigned long long* keys;
    unsigned char* sflag;
    double* selfcorr;
    double* selfwork;
};

// scan the points of `link` for members of the cell of point `ref`: count, first member, and the
// momentum sum (point velocities added in point order, spcs:1040-1054)
__device__ __forceinline__ void scan_link_cell(const SelfCtx& sc, const double* Tprev, const double* Tcur, int link, int ref,
                                               double time_multiplier, int& count, int& first, double& mx, double& my, double& mz) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    const int lane = lane_id();
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + fr.a.P);
    count = 0;
    first = -1;
    mx = my = mz = 0.0;
    const int begin = rb.link_begin[link], end = rb.link_begin[link + 1];
    const unsigned long long kref = sc.keys[ref];
    for (int base = begin; base < end; base += 32) {
        const int q = base + lane;
        const bool match = (q < end) && (sc.keys[q] == kref);
        double vx = 0.0, vy = 0.0, vz = 0.0;
        if (match) {
            double ax, ay, az, bx, by, bz;
            apply_T(Tcur + 12 * link, pxy[q].x, pxy[q].y, pzl[q].z, ax, ay, az);
            apply_T(Tprev + 12 * link, pxy[q].x, pxy[q].y, pzl[q].z, bx, by, bz);
            vx = (ax - bx) * time_multiplier;
            vy = (ay - by) * time_multiplier;
            vz = (az - bz) * time_multiplier;
        }
        unsigned mm = __ballot_sync(FKS_FULL, match);
        if (mm && first < 0) first = base + (__ffs(mm) - 1);
        count += __popc(mm);
        while (mm) {
            const int b = __ffs(mm) - 1;
            mm &= mm - 1u;
            mx += __shfl_sync(FKS_FULL, vx, b);
            my += __shfl_sync(FKS_FULL, vy, b);
            mz += __shfl_sync(FKS_FULL, vz, b);
        }
    }
}

// cell key of a link point: LocationToExtendedGridIndex (spcs:1173-1181) DIVIDES by the map resolution and truncates toward
// zero; the three coordinates are packed 21 bits each (cells of one robot pose never differ by 2^21)
__device__ __forceinline__ unsigned long long self_cell_key(const DevEnv& e, const double* T, double x, double y, double z) {
    double wx, wy, wz;
    apply_T(T, x, y, z, wx, wy, wz);
    const double gx = e.inv_origin[0] * wx + e.inv_origin[1] * wy + e.inv_origin[2] * wz + e.inv_origin[3];
    const double gy = e.inv_origin[4] * wx + e.inv_origin[5] * wy + e.inv_origin[6] * wz + e.inv_origin[7];
    const double gz = e.inv_origin[8] * wx + e.inv_origin[9] * wy + e.inv_origin[10] * wz + e.inv_origin[11];
    const long long kx = (long long)(gx / e.map_res), ky = (long long)(gy / e.map_res), kz = (long long)(gz / e.map_res);
    return ((unsigned long long)kx & 0x1FFFFFull) | (((unsigned long long)ky & 0x1FFFFFull) << 21) | (((unsigned long long)kz & 0x1FFFFFull) << 42);
}

// 10 bits per axis of a cell key: equal keys stay equal
__device__ __forceinline__ unsigned fold_cell_key(unsigned long long k) {
    return (unsigned)(k & 0x3FFull) | ((unsigned)((k >> 21) & 0x3FFull) << 10) | ((unsigned)((k >> 42) & 0x3FFull) << 20);
}
// Middle phase between the capsule test and the exact pass: do two links of a candidate pair have points in ONE cell at all?
// Keys in registers, compared through shuffles -- no scratch memory, a few thousand clocks -- on a 30-bit fold of the exact
// pass's key (10 bits per axis: equal keys stay equal, so a miss here is a miss there; a false hit only costs the exact pass).
// The capsule bound has to allow for cells that are two cells wide, so most of its candidates share no cell: without this
// phase 1.5 % of the arm's collision checks ran the 30 k-clock exact pass for 1 % of them to find anything, and the slowest
// warp of a lock-step round was, every third round, one of those (profiles/r2_kernel_experiments.md).
__device__ __noinline__ bool self_pairs_share_a_cell(int wb, int Xcur, unsigned cp0, unsigned cp1, unsigned cp2, unsigned cp3) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    const DevEnv& e = fr.a.env;
    const int lane = lane_id();
    const double* Tcur = wsd(wb) + fr.a.wl.T + Xcur * fr.a.wl.L12;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + fr.a.P);
    const unsigned cps[kPairChunks] = {cp0, cp1, cp2, cp3};
#pragma unroll 1
    for (int ch = 0; ch < kPairChunks; ch++) {
        unsigned m = cps[ch];
        while (m) {
            const int q = ch * 32 + (__ffs(m) - 1);
            m &= m - 1u;
            const int la = rb.pair_a[q], lb = rb.pair_b[q];
            const int a0 = rb.link_begin[la], a1 = rb.link_begin[la + 1], b0 = rb.link_begin[lb], b1 = rb.link_begin[lb + 1];
            // 64 points of link a in two registers per lane; the points of link b, 32 at a time, are passed around once
#pragma unroll 1
            for (int ab = a0; ab < a1; ab += 64) {
                unsigned ka0 = 0x80000000u, ka1 = 0x80000000u;  // no point: equal to no key of the other link
                const int pa0 = ab + lane, pa1 = ab + 32 + lane;
                if (pa0 < a1) ka0 = fold_cell_key(self_cell_key(e, Tcur + 12 * la, pxy[pa0].x, pxy[pa0].y, pzl[pa0].z));
                if (pa1 < a1) ka1 = fold_cell_key(self_cell_key(e, Tcur + 12 * la, pxy[pa1].x, pxy[pa1].y, pzl[pa1].z));
#pragma unroll 1
                for (int bb = b0; bb < b1; bb += 32) {
                    const int pb = bb + lane;
                    unsigned kb = 0xC0000000u;
                    if (pb < b1) kb = fold_cell_key(self_cell_key(e, Tcur + 12 * lb, pxy[pb].x, pxy[pb].y, pzl[pb].z));
                    const int nb = min(32, b1 - bb);
                    bool hit = false;
#pragma unroll 4
                    for (int s2 = 0; s2 < nb; s2++) {
                        const unsigned k = __shfl_sync(FKS_FULL, kb, s2);
                        hit = hit | (ka0 == k) | (ka1 == k);
                    }
                    if (__any_sync(FKS_FULL, hit)) return true;
                }
            }
        }
    }
    return false;
}

__device__ __noinline__ bool self_collisions_exact(int wb, int Xprev, int Xcur, unsigned cp0, unsigned cp1, unsigned cp2, unsigned cp3) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    const DevEnv& e = fr.a.env;
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    const int P = fr.a.P;
    const double* ws = wsd(wb);
    const double* Tprev = ws + wl.T + Xprev * wl.L12;
    const double* Tcur = ws + wl.T + Xcur * wl.L12;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + P);
    char* slot = context_scratch(wb);
    SelfCtx sc;
    sc.cand_pairs[0] = cp0;
    sc.cand_pairs[1] = cp1;
    sc.cand_pairs[2] = cp2;
    sc.cand_pairs[3] = cp3;
    sc.keys = reinterpret_cast<unsigned long long*>(slot + fr.a.sl.keys);
    sc.sflag = reinterpret_cast<unsigned char*>(slot + fr.a.sl.sflag);
    sc.selfcorr = reinterpret_cast<double*>(slot + fr.a.sl.selfcorr);
    sc.selfwork = reinterpret_cast<double*>(slot + fr.a.sl.selfwork);
    unsigned cand = 0u;  // links taking part in a candidate pair
#pragma unroll
    for (int ch = 0; ch < kPairChunks; ch++) {
        unsigned m = sc.cand_pairs[ch];
        while (m) {
            const int q = ch * 32 + (__ffs(m) - 1);
            m &= m - 1u;
            cand |= (1u << rb.pair_a[q]) | (1u << rb.pair_b[q]);
        }
    }
    sc.cand_links = cand;
    // cell keys: LocationToExtendedGridIndex (spcs:1173-1181) DIVIDES by the map resolution; the three
    // truncated coordinates are packed 21 bits each (cells of one robot pose never differ by 2^21)
    for (int p = lane; p < P; p += 32) {
        const int l = pzl[p].link;
        unsigned long long key = 0ull;
        if ((cand >> l) & 1u) {
            key = self_cell_key(e, Tcur + 12 * l, pxy[p].x, pxy[p].y, pzl[p].z);
        }
        sc.keys[p] = key;
        sc.sflag[p] = 0;
    }
    __syncwarp();
    // per candidate pair: mark the points of either link whose cell also holds a point of the other link.
    // A point is always handled by the same lane ((p - link_begin) % 32), so the flag updates need no barrier.
    bool any = false;
#pragma unroll
    for (int ch = 0; ch < kPairChunks; ch++) {
        unsigned m = sc.cand_pairs[ch];
        while (m) {
            const int q = ch * 32 + (__ffs(m) - 1);
            m &= m - 1u;
#pragma unroll
            for (int role = 0; role < 2; role++) {
                const int la = role ? rb.pair_b[q] : rb.pair_a[q];
                const int lb = role ? rb.pair_a[q] : rb.pair_b[q];
                const int a0 = rb.link_begin[la], a1 = rb.link_begin[la + 1];
                const int b0 = rb.link_begin[lb], b1 = rb.link_begin[lb + 1];
                for (int base = a0; base < a1; base += 32) {
                    const int p = base + lane;
                    const unsigned long long kp = (p < a1) ? sc.keys[p] : 0ull;
                    bool hit = false;
#pragma unroll 4
                    for (int qq = b0; qq < b1; qq++) hit = hit || (sc.keys[qq] == kp);
                    hit = hit && (p < a1);
                    if (hit) sc.sflag[p] = 1;
                    any = any || __any_sync(FKS_FULL, hit);
                }
            }
        }
    }
    __syncwarp();
    if (!any) return false;
    // leaders: the first point of its link in a colliding cell
    for (int p = lane; p < P; p += 32) {
        if (sc.sflag[p] & 1) {
            bool leader = true;
            for (int q = rb.link_begin[pzl[p].link]; q < p; q++)
                if (sc.keys[q] == sc.keys[p]) {
                    leader = false;
                    break;
                }
            if (leader) sc.sflag[p] = 3;
        }
    }
    __syncwarp();
    const double time_multiplier = 1.0 / fr.a.sp.interval;
    double* sw = sc.selfwork;
    // one (cell, link) group at a time, the whole warp working on it
    for (int base = 0; base < P; base += 32) {
        const int p = base + lane;
        unsigned leaders = __ballot_sync(FKS_FULL, (p < P) && (sc.sflag[p] == 3));
        while (leaders) {
            const int gp = base + (__ffs(leaders) - 1);
            leaders &= leaders - 1u;
            const int l = pzl[gp].link;
            int cnt_i, first_i;
            double mix, miy, miz;
            scan_link_cell(sc, Tprev, Tcur, l, gp, time_multiplier, cnt_i, first_i, mix, miy, miz);
            double aix, aiy, aiz;
            apply_T(Tprev + 12 * l, pxy[first_i].x, pxy[first_i].y, pzl[first_i].z, aix, aiy, aiz);
            const double inv_i = 1.0 / (double)cnt_i;
            const double vix = mix * inv_i, viy = miy * inv_i, viz = miz * inv_i;
            // colliding links in ascending order (std::map iteration, spcs:1000-1017)
            int m = 0;
            unsigned dis = rb.disallowed[l] & sc.cand_links;
            while (dis) {
                const int s = __ffs(dis) - 1;
                dis &= dis - 1u;
                int cnt_s, first_s;
                double msx, msy, msz;
                scan_link_cell(sc, Tprev, Tcur, s, gp, time_multiplier, cnt_s, first_s, msx, msy, msz);
                if (cnt_s == 0) continue;
                double ox, oy, oz;
                apply_T(Tprev + 12 * s, pxy[first_s].x, pxy[first_s].y, pzl[first_s].z, ox, oy, oz);
                double nx = ox - aix, ny = oy - aiy, nz = oz - aiz;
                safe_normal3(nx, ny, nz);
                const double inv_s = 1.0 / (double)cnt_s;
                const double vsx = msx * inv_s, vsy = msy * inv_s, vsz = msz * inv_s;
                const double rhs = nx * (vsx - vix) + ny * (vsy - viy) + nz * (vsz - viz);
                if (lane == 0) {
                    sw[5 * m + 0] = nx;
                    sw[5 * m + 1] = ny;
                    sw[5 * m + 2] = nz;
                    sw[5 * m + 3] = rhs;
                    sw[5 * m + 4] = rb.link_mass[s];
                }
                m++;
            }
            double* out = sw + 5 * kMaxSelfPartners;  // per-point correction (3)
            __syncwarp();
            if (lane == 0) {
                // A = N^T C^T M^-1 C N (spcs:1135), inverse by partial-pivot Gauss elimination, lambda = A^-1 r
                double* Mx = out + 4;                                          // m x 2m augmented
                double* Ainv = Mx + kMaxSelfPartners * 2 * kMaxSelfPartners;  // m x m
                const double mass_i = rb.link_mass[l];
                const int n = m;
                for (int a = 0; a < n; a++)
                    for (int b = 0; b < n; b++) {
                        double v = (sw[5 * a] * sw[5 * b] + sw[5 * a + 1] * sw[5 * b + 1] + sw[5 * a + 2] * sw[5 * b + 2]) / mass_i;
                        if (a == b) v += (sw[5 * a] * sw[5 * a] + sw[5 * a + 1] * sw[5 * a + 1] + sw[5 * a + 2] * sw[5 * a + 2]) / sw[5 * a + 4];
                        Mx[a * 2 * n + b] = v;
                        Mx[a * 2 * n + n + b] = (a == b) ? 1.0 : 0.0;
                    }
                for (int k = 0; k < n; k++) {
                    int piv = k;
                    double best = fabs(Mx[k * 2 * n + k]);
                    for (int r = k + 1; r < n; r++)
                        if (fabs(Mx[r * 2 * n + k]) > best) {
                            best = fabs(Mx[r * 2 * n + k]);
                            piv = r;
                        }
                    if (piv != k)
                        for (int cc = 0; cc < 2 * n; cc++) {
                            const double t = Mx[k * 2 * n + cc];
                            Mx[k * 2 * n + cc] = Mx[piv * 2 * n + cc];
                            Mx[piv * 2 * n + cc] = t;
                        }
                    const double pv = Mx[k * 2 * n + k];
                    for (int r = k + 1; r < n; r++) {
                        const double f = Mx[r * 2 * n + k] / pv;
                        for (int cc = k; cc < 2 * n; cc++) Mx[r * 2 * n + cc] -= f * Mx[k * 2 * n + cc];
                    }
                }
                for (int cc = 0; cc < n; cc++)
                    for (int r = n - 1; r >= 0; r--) {
                        double s = Mx[r * 2 * n + n + cc];
                        for (int j = r + 1; j < n; j++) s -= Mx[r * 2 * n + j] * Ainv[j * n + cc];
                        Ainv[r * n + cc] = s / Mx[r * 2 * n + r];
                    }
                double cx = 0.0, cy = 0.0, cz = 0.0;
                for (int a = 0; a < n; a++) {
                    double lam = 0.0;
                    for (int b = 0; b < n; b++) lam += Ainv[a * n + b] * sw[5 * b + 3];
                    cx = cx + sw[5 * a] * lam;
                    cy = cy + sw[5 * a + 1] * lam;
                    cz = cz + sw[5 * a + 2] * lam;
                }
                const double im = 1.0 / mass_i;
                cx = cx * im;
                cy = cy * im;
                cz = cz * im;
                out[0] = cx * inv_i;
                out[1] = cy * inv_i;
                out[2] = cz * inv_i;
            }
            __syncwarp();
            const double ppx = out[0], ppy = out[1], ppz = out[2];
            if (isnan(ppx) || isnan(ppy) || isnan(ppz)) raise_flag(wb, FKS_FLAG_WOULD_ASSERT_NAN);  // asserts spcs:1151-1153
            const unsigned long long kgp = sc.keys[gp];
            for (int q = rb.link_begin[l] + lane; q < rb.link_begin[l + 1]; q += 32)
                if (sc.keys[q] == kgp) {
                    sc.selfcorr[3 * q] = ppx;
                    sc.selfcorr[3 * q + 1] = ppy;
                    sc.selfcorr[3 * q + 2] = ppz;
                }
            __syncwarp();
        }
    }
    return true;
}

// broad phase over the disallowed link pairs, on the capsule end points kinematics() left in shared memory
__device__ __forceinline__ bool collect_self(int wb, int Xprev, int Xcur) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    if (rb.n_pairs == 0) return false;  // one link, or every pair allowed (spcs:1186-1197)
    const int lane = lane_id();
    const double* caps = wsd(wb) + fr.a.wl.caps;
    const double diag = 2.0 * 1.7320508075688772 * fr.a.env.map_res * (1.0 + 1e-6) + 1e-9;  // cells at index 0 are two cells wide
    unsigned cp[kPairChunks] = {0u, 0u, 0u, 0u};
    bool anyc = false;
    const int nch = (rb.n_pairs + 31) >> 5;
    for (int ch = 0; ch < nch; ch++) {
        const int q = ch * 32 + lane;
        bool hit = false;
        if (q < rb.n_pairs) {
            const int a = rb.pair_a[q], b = rb.pair_b[q];
            // midpoints first: the segments are at least |m_a - m_b| - half lengths apart (triangle inequality), so far-apart
            // links never reach the segment-segment distance -- for an arm away from itself that is every pair, every check
            const double* ca = caps + 6 * a;
            const double* cb = caps + 6 * b;
            const double mx = 0.5 * ((ca[0] + ca[3]) - (cb[0] + cb[3])), my = 0.5 * ((ca[1] + ca[4]) - (cb[1] + cb[4])),
                         mz = 0.5 * ((ca[2] + ca[5]) - (cb[2] + cb[5]));
            hit = mx * mx + my * my + mz * mz <= fr.pair_reach_sq[q];
        }
        if (__any_sync(FKS_FULL, hit)) {
            if (hit) {
                const int a = rb.pair_a[q], b = rb.pair_b[q];
                const double d2 = segment_distance_sq(caps + 6 * a, caps + 6 * a + 3, caps + 6 * b, caps + 6 * b + 3);
                const double reach = rb.cap_radius[a] + rb.cap_radius[b] + diag;
                hit = d2 <= reach * reach;
                // Only the cells at index 0 of an axis are two cells wide (they span -res .. +res of the grid coordinate): beyond
                // the ordinary cell diagonal the two links can share a cell only if BOTH reach that slab on the same axis.
                const double narrow = rb.cap_radius[a] + rb.cap_radius[b] + 0.5 * diag;
                if (hit && d2 > narrow * narrow) {
                    const DevEnv& e = fr.a.env;
                    bool both = false;
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        bool reaches[2];
#pragma unroll
                        for (int side = 0; side < 2; side++) {
                            const double* c = caps + 6 * (side ? b : a);
                            const double g0 = e.inv_origin[4 * k] * c[0] + e.inv_origin[4 * k + 1] * c[1] + e.inv_origin[4 * k + 2] * c[2] + e.inv_origin[4 * k + 3];
                            const double g1 = e.inv_origin[4 * k] * c[3] + e.inv_origin[4 * k + 1] * c[4] + e.inv_origin[4 * k + 2] * c[5] + e.inv_origin[4 * k + 3];
                            const double nearest = (g0 < 0.0) != (g1 < 0.0) ? 0.0 : fmin(fabs(g0), fabs(g1));
                            reaches[side] = nearest - rb.cap_radius[side ? b : a] <= e.map_res * (1.0 + 1e-6) + 1e-9;
                        }
                        both = both || (reaches[0] && reaches[1]);
                    }
                    hit = both;
                }
            }
        }
        const unsigned m = __ballot_sync(FKS_FULL, hit);
        if (ch == 0) cp[0] = m;
        else if (ch == 1) cp[1] = m;
        else if (ch == 2) cp[2] = m;
        else cp[3] = m;
        anyc = anyc || (m != 0u);
    }
    if (!anyc) return false;
    if (!self_pairs_share_a_cell(wb, Xcur, cp[0], cp[1], cp[2], cp[3])) return false;
    return self_collisions_exact(wb, Xprev, Xcur, cp[0], cp[1], cp[2], cp[3]);
}

// CheckCollision (spcs:1418-1436): bit 0 = in collision, bit 1 = self-collision map non-empty
#ifdef FKS_PHASE_TIMERS
__device__ unsigned long long g_dbg[64];  // developer counters: [0..15] histogram of check_env clocks (bins of 2048), [16..31] of collect_self, 32.. sums
#endif
template <int KIND>
__device__ __forceinline__ unsigned check_collision(int wb, int Xprev, int Xcur, int use_cull) {
#ifdef FKS_PHASE_TIMERS
    const long long t0 = clock64();
#endif
    const bool envc = check_env(wb, Xcur, use_cull, 0.0);
#ifdef FKS_PHASE_TIMERS
    const long long t1 = clock64();
#endif
    const bool has_self = (KIND == FKS_ROBOT_LINKED) ? collect_self(wb, Xprev, Xcur) : false;
#ifdef FKS_PHASE_TIMERS
    if (lane_id() == 0) {
        const long long t2 = clock64();
        atomicAdd(&g_dbg[min((int)((t1 - t0) >> 11), 15)], 1ull);
        atomicAdd(&g_dbg[16 + min((int)((t2 - t1) >> 11), 15)], 1ull);
        atomicAdd(&g_dbg[32], (unsigned long long)(t1 - t0));
        atomicAdd(&g_dbg[33], (unsigned long long)(t2 - t1));
        atomicAdd(&g_dbg[34 + (envc ? 1 : 0)], 1ull);
        atomicAdd(&g_dbg[36 + (envc ? 1 : 0)], (unsigned long long)(t1 - t0));
        atomicAdd(&g_dbg[38 + (has_self ? 1 : 0)], 1ull);
    }
#endif
    return ((envc || has_self) ? 1u : 0u) | (has_self ? 2u : 0u);
}

// A collected system that outgrew the small shared-memory store (its rows < cap_s are there, the others in the warp's global
// store): where it is factored.  In the larger shared-memory store (what a solve may overwrite once the corrections are
// collected: world->voxel transforms, joint axes / origins, candidate list -- all rebuilt before they are read again) when
// it fits, else in place in the global store, where every load of the in-place update is an L2 round trip.  Either way the
// small store's rows first complete the global copy (the two shared stores overlap with different leading dimensions).
// Every column moves as one bulk copy: leading dimensions are even, so columns start on 16 bytes.  Called at the end of
// collect_corrections rather than from the main loop, which has no registers to spare.
__device__ __forceinline__ void move_tall_system(int wb, int rows, int cols) {
    const Frame& fr = frame();
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    double* As = wsd(wb) + wl.jsm;
    double* Ag = warp_jstore();
    const int lds = wl.jsm_ld, cap_s = (wl.jsm_ld / 3) * 3, ldg = fr.a.sl.ldj, ldb = wl.jsm_big_ld;
    // of an odd row count the lanes copy the last row: rounding the copies up would overwrite row cap_s of the global
    // columns, which the collect wrote
    const int nb = cap_s & ~1;
    if (nb < cap_s && lane <= cols) Ag[(size_t)lane * ldg + nb] = As[lane * lds + nb];
    fence_async_shared();  // (a): the collect's rows in both stores, and the row above
    fence_async_global();
    __syncwarp();
    if (lane == 0) {
        for (int c = 0; c <= cols; c++) bulk_store(Ag + (size_t)c * ldg, As + c * lds, nb);
        bulk_commit();
        bulk_wait_all();  // (b): complete, the global copy is read next
    }
    __syncwarp();
    if (rows > ldb) return;
    // an odd row count is rounded up by one row, which stays inside the column (ldb is even, ldg a multiple of 4, rows <= both)
    const int n = (rows + 1) & ~1;
    const unsigned bar = warp_bar();
    unsigned long long state = 0ull;
    if (lane == 0) {
        fence_async_global();  // (a): the bulk stores above are visible to lane 0's generic proxy (b), the loads read them
        state = bulk_expect(bar, (cols + 1) * n * 8);
        for (int c = 0; c <= cols; c++) bulk_load(As + c * ldb, Ag + (size_t)c * ldg, n, bar);
    }
    bulk_wait_loads(bar, state);
}

// ------------------------------------------------------------------------------------------------
// CollectPointCorrectionsAndJacobians (spcs:1818-1939): fills the stacked Jacobian (column major,
// column D holds the corrections), rows in link-major point-minor order: the first rows into the warp's
// shared-memory store (leading dimension wl.jsm_ld), the rows beyond its capacity into the global scratch slot
// (leading dimension sl.ldj, same row indices).  Returns the number of rows; place_system() decides where it is solved.
//
// Two passes.  Pass 1 is the cheap voxel test of check_env over all points, kBatch gathers in flight per
// lane: EstimateDistance4d = f -/+ res/2 + (|.| <= sqrt(3)/2 res) cannot be negative when the raw cell value
// f >= 2 res, so only "near" points (and points holding a self-collision correction) survive, compacted in
// point order into the scratch slot's key array.  Pass 2 runs the expensive part -- 6 more gathers, the
// normal lookup, the Jacobian row -- on the survivors only.
// ------------------------------------------------------------------------------------------------
template <int KIND>
__device__ __noinline__ int collect_corrections(int wb, int Xprev, int Xcur, bool has_self) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    const DevEnv& e = fr.a.env;
    const WarpLayout& wl = fr.a.wl;
    const int lane = lane_id();
    const int P = fr.a.P, D = rb.D;
    double* ws = wsd(wb);
    const double* Tprev = ws + wl.T + Xprev * wl.L12;
    const double* Tcur = ws + wl.T + Xcur * wl.L12;
    const double* G = ws + wl.G;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + P);
    const char* cslot = context_scratch(wb);
    double* Ag = warp_jstore();
    const unsigned char* sflag = reinterpret_cast<const unsigned char*>(cslot + fr.a.sl.sflag);
    const double* selfcorr = reinterpret_cast<const double*>(cslot + fr.a.sl.selfcorr);
    // candidate list: {point index | bit 31 = needs the environment estimate, raw cell value}; the first kCandShared
    // live in shared memory, the rest behind the Jacobian columns of the global store
    uint2* cand_s = reinterpret_cast<uint2*>(ws + wl.cand);
    uint2* cand_g = reinterpret_cast<uint2*>(Ag + (size_t)(D + 1) * fr.a.sl.ldj);
    double* jaxis = ws + wl.jaxis;
    double* jorig = ws + wl.jorig;
    if (KIND == FKS_ROBOT_LINKED) {
        // world axis / origin of every joint (frame = child link transform)
        for (int j = lane; j < rb.J; j += 32) {
            const DevJoint& jd = rb.joints[j];
            const double* Tj = Tcur + 12 * jd.child;
            jaxis[3 * j + 0] = Tj[0] * jd.axis[0] + Tj[1] * jd.axis[1] + Tj[2] * jd.axis[2];
            jaxis[3 * j + 1] = Tj[4] * jd.axis[0] + Tj[5] * jd.axis[1] + Tj[6] * jd.axis[2];
            jaxis[3 * j + 2] = Tj[8] * jd.axis[0] + Tj[9] * jd.axis[1] + Tj[10] * jd.axis[2];
            jorig[3 * j + 0] = Tj[3];
            jorig[3 * j + 1] = Tj[7];
            jorig[3 * j + 2] = Tj[11];
        }
    }
    const double res = e.sdf_res;
    const float near = (float)(2.0 * res);
    // ---- pass 1 -----------------------------------------------------------------------------------
    int ncand = 0;
    unsigned links = (fr.a.cull_mode != 1 || !e.cull || has_self) ? ((1u << rb.L) - 1u) : active_links(e, rb, G, 2.0 * res);
    while (links) {  // ascending: the rows of the stacked system are in (link, point) order (spcs:1893-1929)
        const int first = __ffs(links) - 1;
        const int len = __ffs(~(links >> first)) - 1;
        links &= ~(((len >= 32) ? 0xffffffffu : ((1u << len) - 1u)) << first);
        const int end = rb.link_begin[first + len];
        for (int pos = rb.link_begin[first]; pos < end; pos += 32 * kBatch) {
            float f[kBatch];
#pragma unroll
            for (int k = 0; k < kBatch; k++) {
                const int p = pos + 32 * k + lane;
                f[k] = INFINITY;
                if (p < end) {
                    const double2 xy = pxy[p];
                    const PointZL zl = pzl[p];
                    const Voxel v = voxel_of(e, G + 12 * zl.link, xy.x, xy.y, zl.z);
                    if (v.inb) f[k] = sdf_cell(e, v.x, v.y, v.z);
                }
            }
#pragma unroll
            for (int k = 0; k < kBatch; k++) {
                const int p = pos + 32 * k + lane;
                const bool is_near = f[k] < near;  // out of bounds / padding: +inf
                const bool keep = (p < end) && (is_near || (has_self && (sflag[p] & 1)));
                const unsigned mask = __ballot_sync(FKS_FULL, keep);
                if (keep) {
                    const int ci = ncand + __popc(mask & ((1u << lane) - 1u));
                    const uint2 rec = make_uint2((unsigned)p | (is_near ? 0x80000000u : 0u), __float_as_uint(f[k]));
                    if (ci < kCandShared) cand_s[ci] = rec;
                    else cand_g[ci] = rec;
                }
                ncand += __popc(mask);
            }
        }
    }
    __syncwarp();
    // Optimistic placement: rows go to the shared-memory store while they fit it (cap_s rows, a multiple of 3, so a point's
    // three rows never straddle) and to the global store beyond; most candidates turn out not to penetrate, so most systems
    // end up entirely in shared memory.  A system that outgrew the small store is moved at the end (move_tall_system).
    double* As = ws + wl.jsm;
    const int lds = wl.jsm_ld, cap_s = (wl.jsm_ld / 3) * 3, ldg = fr.a.sl.ldj;
    // ---- pass 2 -----------------------------------------------------------------------------------
    int npts = 0;
    for (int base = 0; base < ncand; base += 32) {
        const int ci = base + lane;
        bool have = false;
        double cx = 0.0, cy = 0.0, cz = 0.0;
        double wx = 0.0, wy = 0.0, wz = 0.0, lx = 0.0, ly = 0.0, lz = 0.0;
        int l = 0;
        if (ci < ncand) {
            const uint2 rec2 = (ci < kCandShared) ? cand_s[ci] : cand_g[ci];
            const unsigned rec = rec2.x;
            const int p = (int)(rec & 0x7FFFFFFFu);
            const double2 xy = pxy[p];
            const PointZL zl = pzl[p];
            l = zl.link;
            lx = xy.x;
            ly = xy.y;
            lz = zl.z;
            apply_T(Tcur + 12 * l, lx, ly, lz, wx, wy, wz);
            if (has_self && (sflag[p] & 1)) {
                have = true;
                cx = cx + selfcorr[3 * p];
                cy = cy + selfcorr[3 * p + 1];
                cz = cz + selfcorr[3 * p + 2];
            }
            if (rec >> 31) {
                const Voxel v = voxel_of(e, G + 12 * l, lx, ly, lz);  // same arithmetic as pass 1: same voxel
                const int vxx = v.x, vyy = v.y, vzz = v.z;
                const float f = __uint_as_float(rec2.y);
                const long long li = ((long long)vxx * e.ny + vyy) * e.nz + vzz;
                const uint2 nrange = (f < 0.5f * near) ? normal_range_probe(e, li) : make_uint2(0u, 0u);  // issued early
                const double est = FKS_COLLECT_ESTIMATE(wx, wy, wz, vxx, vyy, vzz, f);
                if (est < 0.0) {  // resolution_distance_threshold_ = 0.0 (spcs:425,1874)
                    double qx, qy, qz;
                    apply_T(Tprev + 12 * l, lx, ly, lz, qx, qy, qz);
                    double dx = wx - qx, dy = wy - qy, dz = wz - qz;
                    safe_normal3(dx, dy, dz);
                    double nx, ny, nz;
                    // est < 0 needs f < res/2 + sqrt(3)/2 res < 2 res: the probe above covered every such point
                    const uint2 nr = (f < 0.5f * near) ? nrange : normal_range_probe(e, li);
                    select_normal(wb, e, nr, dx, dy, dz, nx, ny, nz);
                    safe_normal3(nx, ny, nz);
                    const double pen = fabs(0.0 - est);
                    cx = cx + nx * pen;
                    cy = cy + ny * pen;
                    cz = cz + nz * pen;
                    have = true;
                }
            }
        }
        const unsigned mask = __ballot_sync(FKS_FULL, have);
        if (have) {
            const int row0 = 3 * (npts + __popc(mask & ((1u << lane) - 1u)));
            const bool small = row0 < cap_s;
            double* A = small ? As : Ag;
            const int ld = small ? lds : ldg;
            double* b = A + (size_t)D * ld + row0;
            b[0] = cx;
            b[1] = cy;
            b[2] = cz;
            // ComputeLinkPointTranslationJacobian (3 x D)
            if (KIND == FKS_ROBOT_SE2) {
                const double rx = wx - Tcur[3], ry = wy - Tcur[7];
                double* a0 = A + row0;
                a0[0] = 1.0; a0[1] = 0.0; a0[2] = 0.0;
                double* a1 = A + ld + row0;
                a1[0] = 0.0; a1[1] = 1.0; a1[2] = 0.0;
                double* a2 = A + 2 * ld + row0;  // z x (p_world - (x, y, 0))
                a2[0] = 0.0 - ry;
                a2[1] = rx;
                a2[2] = 0.0;
            } else if (KIND == FKS_ROBOT_SE3) {
#pragma unroll
                for (int r = 0; r < 3; r++) {
                    const double t0 = Tcur[4 * r + 0], t1 = Tcur[4 * r + 1], t2 = Tcur[4 * r + 2];
                    A[0 * ld + row0 + r] = t0;
                    A[1 * ld + row0 + r] = t1;
                    A[2 * ld + row0 + r] = t2;
                    A[3 * ld + row0 + r] = t1 * (-lz) + t2 * ly;
                    A[4 * ld + row0 + r] = t0 * lz + t2 * (-lx);
                    A[5 * ld + row0 + r] = t0 * (-ly) + t1 * lx;
                }
            } else {
                const unsigned anc = rb.link_ancestors[l];
                for (int a = 0; a < D; a++) {
                    const int j = rb.active_joint[a];
                    double jx = 0.0, jy = 0.0, jz = 0.0;
                    if ((anc >> j) & 1u) {
                        const double ax = jaxis[3 * j], ay = jaxis[3 * j + 1], az = jaxis[3 * j + 2];
                        if (rb.joints[j].type == FKS_JOINT_PRISMATIC) {
                            jx = ax; jy = ay; jz = az;
                        } else {
                            const double rx = wx - jorig[3 * j], ry = wy - jorig[3 * j + 1], rz = wz - jorig[3 * j + 2];
                            jx = ay * rz - az * ry;
                            jy = az * rx - ax * rz;
                            jz = ax * ry - ay * rx;
                        }
                    }
                    double* col = A + (size_t)a * ld + row0;
                    col[0] = jx;
                    col[1] = jy;
                    col[2] = jz;
                }
            }
        }
        npts += __popc(mask);
    }
    __syncwarp();
    if (3 * npts > cap_s) move_tall_system(wb, 3 * npts, D);
    return 3 * npts;
}

// ------------------------------------------------------------------------------------------------
// ComputeResolverCorrectionStepStackedJacobian (spcs:1990-1998): x = J.colPivHouseholderQr().solve(c).
//
// Eigen 3.3's ColPivHouseholderQR::compute + solve restated OPERATION FOR OPERATION (SURVEY A.3; the oracle's
// colpiv_qr_solve is the same restatement): LAPACK-style downdated column norms, pivot = first largest updated norm, rank
// cut |pivot|^2 < (eps max|col|)^2 / rows (rows - k), makeHouseholderInPlace from the tail's squared norm, reflectors
// applied as  tmp = essential . bottom + top;  top -= tau tmp;  bottom -= (tau essential) tmp,  basic solution.
//
// Why verbatim.  With a single distal link of the arm in contact the stacked Jacobian has rank <= 6 in 7 unknowns: the
// last pivot is pure round-off and Eigen cuts or keeps it by the last bit; when it is kept the solve divides by it and the
// "correction" saturates every joint, which usually fails the resolve.  How OFTEN that happens decides the failure rate of
// the whole workload, and it moves between 6 % and 11 % with the summation order, the association of the reflector update
// or FMA contraction (profiles/r2_qr_keep_rate.md).  So every product and sum here rounds once (__dmul_rn / __dadd_rn: the
// reference is x86-64 code without FMA) and every reduction over rows uses the oracle's order -- Eigen's SSE2 reduction:
// four interleaved partial sums, partial sum i over the rows congruent to i modulo 4 in ascending order, result
// (p0 + p2) + (p1 + p3).  On identical input this solver returns the oracle's bits (tests/test_gpu_qr_solver.py).
//
// Mapping: FOUR lanes per column, lane 4 g + i owns the rows = i (mod 4) of column g (+ 8 per extra slot when there are
// more than 8 columns; column `cols` is the right-hand side), so a partial sum is a private sequential loop and a reduction
// ends with two exchanges inside the quad.  A lane only ever touches its own rows of its own columns, except for the pivot
// column's essential part, which every lane reads (a broadcast).  The squared norms Eigen computes in separate passes (the
// tail of the next pivot column, the recomputed norm of a downdate) are accumulated while the column is updated -- same
// values, same order, no extra pass.  ~450 instructions in one loop nest: the register-resident warp-cooperative QR it
// replaces was 2 500 per copy and instruction-cache bound.
//
// A = (cols + 1) columns of leading dimension ld (shared memory when the system is small, the warp's global scratch slot
// otherwise: generic addressing).  Result in the shared vector at x_off.
//
// Parity mode (decision tape, fksgpu.h): the pivot order and the rank are taken from the tape, the solver's own are
// still computed and a difference raises FKS_FLAG_DECISION_OVERRIDDEN; a record flagged OVERRIDE_SOLUTION replaces the
// solve altogether.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
// (p0 + p2) + (p1 + p3) over the four lanes of a quad; every lane of the quad gets the same bits (+ is commutative)
__device__ __forceinline__ double quad_sum(unsigned mask, double p) {
    p = add_rn(p, __shfl_xor_sync(mask, p, 2));
    return add_rn(p, __shfl_xor_sync(mask, p, 1));
}

// the solver's row loops stay rolled: 30 KB less code for the warps of a SOLVE cycle to fetch, 2-5 % faster on the contact
// workloads than nvcc's default unrolling (profiles/r2_kernel_experiments.md)
#define FKS_QR_INNER_LOOP _Pragma("unroll 1")
// ... but the loads of FKS_QR_BATCH rows go out together: a system in the global store pays an L2 round trip per load
// otherwise (solve from the global store 126 k -> 82 k clocks at 4; 2 measured as fast as 4 and 8 end to end, with less code); the sums stay in row order
#ifndef FKS_QR_BATCH
#define FKS_QR_BATCH 2
#endif
template <int SLOTS>  // columns per quad: 1 for up to 8 columns (every robot of the reference), 2 for up to 16
__device__ __noinline__ void colpiv_qr_lanes(int wb, double* A, int ld, int rows, int cols, int x_off) {
    const Frame& fr = frame();
    const int lane = lane_id();
    double* ws = wsd(wb);
    WarpVars* wv = reinterpret_cast<WarpVars*>(ws + fr.a.wl.vars);
    double* x = ws + x_off;
    const int g = lane >> 2, i = lane & 3;
    const unsigned quad = 0xFu << (lane & ~3);
    // ---- decision tape (parity mode only) ----------------------------------------------------------------------
    bool forced = false;
    int f_rank = 0;
    unsigned long long f_order = 0ull;
    if (fr.a.dec_tape != nullptr) {
        const unsigned long long dp = wv->dec_pos;
        bool desync = true, replaced = false;
        if (dp < wv->dec_end) {
            const unsigned long long* rec = fr.a.dec_tape + dp * (unsigned long long)(2 + cols);
            const unsigned long long w0 = rec[0];
            if ((int)((w0 >> 16) & 0xFFFFFFFFull) == rows) {
                desync = false;
                forced = true;
                f_rank = (int)(w0 & 0xFFull);
                f_order = rec[1];
                if (w0 & (unsigned long long)FKS_DECISION_OVERRIDE_SOLUTION) {
                    replaced = true;
                    if (lane < cols) x[lane] = __longlong_as_double((long long)rec[2 + lane]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) {
            wv->dec_pos = dp + 1ull;
            if (desync) raise_flag(wb, FKS_FLAG_DECISION_DESYNC);
            if (replaced) raise_flag(wb, FKS_FLAG_DECISION_OVERRIDDEN);
        }
        __syncwarp();
        if (replaced) return;
    }
    const int size = rows < cols ? rows : cols;
    // per column slot of this quad: colNormsUpdated / colNormsDirect, the position in Eigen's permuted order, and this
    // lane's partial of sum_{r > k} a_r^2 for the coming step (= the tail's squared norm should the column be the pivot)
    double nu[SLOTS], nd[SLOTS], tailp[SLOTS];
    int pos[SLOTS];
    double max_norm = 0.0;
    int own_rank = size, nonzero_pivots = size;
    unsigned long long order = 0ull;  // 4 bits per position: the column sitting there
    bool differed = false, near_cut = false;
#pragma unroll
    for (int sl = 0; sl < SLOTS; sl++) {
        const int c = g + 8 * sl;
        nu[sl] = nd[sl] = tailp[sl] = 0.0;
        pos[sl] = c;
        if (c < cols) {  // uniform inside the quad
            const double* mine = A + (size_t)c * ld;
            double pf = 0.0, pt = 0.0;
            FKS_QR_INNER_LOOP
            for (int r = i; r < rows; r += 4) {
                const double a = mine[r];
                const double sq = mul_rn(a, a);
                pf = add_rn(pf, sq);
                if (r >= 1) pt = add_rn(pt, sq);
            }
            nd[sl] = nu[sl] = sqrt(quad_sum(quad, pf));
            tailp[sl] = pt;
            max_norm = fmax(max_norm, nu[sl]);
        }
    }
    max_norm = warp_max(max_norm);
    const double me = mul_rn(max_norm, DBL_EPSILON);
    const double threshold_helper = div_rn(mul_rn(me, me), (double)rows);
    const double norm_downdate_threshold = 1.4901161193847656e-08;  // sqrt(epsilon)
#pragma unroll 1
    for (int k = 0; k < size; k++) {
        // biggest updated norm among the positions k .. cols-1, the first position wins (Eigen's maxCoeff scan)
        double bv = -1.0;
        int bp = 0x7fffffff, bc = 0;
#pragma unroll
        for (int sl = 0; sl < SLOTS; sl++) {
            const int c = g + 8 * sl;
            if (c < cols && pos[sl] >= k && (nu[sl] > bv || (nu[sl] == bv && pos[sl] < bp))) {
                bv = nu[sl];
                bp = pos[sl];
                bc = c;
            }
        }
#pragma unroll
        for (int o = 16; o >= 4; o >>= 1) {
            const double ov = __shfl_xor_sync(FKS_FULL, bv, o);
            const int op = __shfl_xor_sync(FKS_FULL, bp, o), oc = __shfl_xor_sync(FKS_FULL, bc, o);
            if (ov > bv || (ov == bv && op < bp)) {
                bv = ov;
                bp = op;
                bc = oc;
            }
        }
        int p = bc;
        if (forced) {
            const int fp = (int)((f_order >> (4 * k)) & 0xFull);
            // position and norm of the tape's pivot column, from its quad
            double fnu = nu[0];
            int fpos = pos[0];
            if (SLOTS > 1 && (fp >> 3) == 1) {
                fnu = nu[SLOTS - 1];
                fpos = pos[SLOTS - 1];
            }
            fnu = __shfl_sync(FKS_FULL, fnu, 4 * (fp & 7));
            fpos = __shfl_sync(FKS_FULL, fpos, 4 * (fp & 7));
            if (fp < cols && fpos >= k) {
                if (fp != p) differed = true;
                p = fp;
                bp = fpos;
                bv = fnu;
            } else {
                differed = true;  // a record that does not fit this system: keep the solver's own pivot
            }
        }
        const double big_sq = mul_rn(bv, bv);
        const double cut = mul_rn(threshold_helper, (double)(rows - k));
        if (own_rank == size && big_sq < cut) own_rank = k;
        if (max_norm > 0.0 && big_sq > 0.0 && big_sq < cut * 1e6) near_cut = true;
        nonzero_pivots = forced ? (f_rank < size ? f_rank : size) : own_rank;
        // Eigen carries the factorisation on after the cut ("to make sure that the initial matrix is properly reproduced"), but
        // its solve reads the first nonzero_pivots reflectors and the leading nonzero_pivots x nonzero_pivots triangle only,
        // and nonzero_pivots never changes once set: nothing computed from here on reaches the solution.
        if (k >= nonzero_pivots) {
            if (forced && own_rank != nonzero_pivots) differed = true;
            own_rank = nonzero_pivots;
            break;
        }
        // the column that sat at position k takes the pivot's old position (m_qr.col(k).swap(m_qr.col(biggest)))
        double tail_sq = 0.0;
#pragma unroll
        for (int sl = 0; sl < SLOTS; sl++) {
            const int c = g + 8 * sl;
            if (c < cols && pos[sl] == k) pos[sl] = bp;
            if (c == p) {
                pos[sl] = k;
                tail_sq = tailp[sl];
            }
        }
        order |= (unsigned long long)p << (4 * k);
        double* piv = A + (size_t)p * ld;
        // makeHouseholderInPlace on col(k).tail(rows - k): the tail's squared norm was accumulated with the last update
        tail_sq = __shfl_sync(FKS_FULL, quad_sum(FKS_FULL, tail_sq), 4 * (p & 7));
        const double c0 = piv[k];
        double tau, beta;
        if (tail_sq <= DBL_MIN) {
            tau = 0.0;
            beta = c0;
            FKS_QR_INNER_LOOP
            for (int r = k + 1 + lane; r < rows; r += 32) piv[r] = 0.0;
        } else {
            beta = sqrt(add_rn(mul_rn(c0, c0), tail_sq));
            if (c0 >= 0.0) beta = -beta;
            const double denom = sub_rn(c0, beta);
            FKS_QR_INNER_LOOP
            for (int r = k + 1 + lane; r < rows; r += 32) piv[r] = div_rn(piv[r], denom);  // element-wise: any lane may do it
            tau = div_rn(sub_rn(beta, c0), beta);
        }
        __syncwarp();  // c0 has been read by everyone, the essential part is visible to everyone
        if (lane == 0) piv[k] = beta;
        // applyHouseholderOnTheLeft to the remaining columns; to the right-hand side only below the rank cut (Eigen's solve
        // applies the first nonzero_pivots reflectors to c).  The loop that updates a column also accumulates the squared
        // norms of its rows > k (a downdate may need it) and > k + 1 (the next tail).
        // In the LAST step the remaining columns end up at positions >= size, which the solve never reads: only the
        // right-hand side is reflected.
        const bool last_row = rows - k == 1;
        const bool last_step = k == size - 1;
        const int r0 = k + 1 + ((i - (k + 1)) & 3);  // first row > k that is = i (mod 4)
#pragma unroll
        for (int sl = 0; sl < SLOTS; sl++) {
            const int c = g + 8 * sl;
            const bool is_col = c < cols;
            if (!((is_col && pos[sl] > k && !last_step) || (c == cols && nonzero_pivots > k))) continue;  // uniform inside the quad
            double* mine = A + (size_t)c * ld;
            double ak = mine[k];
            double tmp = 0.0;
            const bool reflect = !last_row && tau != 0.0;
            if (reflect) {
                double pd = 0.0;
                int r = r0;
                FKS_QR_INNER_LOOP
                for (; r + 4 * (FKS_QR_BATCH - 1) < rows; r += 4 * FKS_QR_BATCH) {
                    double av[FKS_QR_BATCH], bv2[FKS_QR_BATCH];
#pragma unroll
                    for (int u = 0; u < FKS_QR_BATCH; u++) {
                        av[u] = piv[r + 4 * u];
                        bv2[u] = mine[r + 4 * u];
                    }
#pragma unroll
                    for (int u = 0; u < FKS_QR_BATCH; u++) pd = add_rn(pd, mul_rn(av[u], bv2[u]));
                }
                FKS_QR_INNER_LOOP
                for (; r < rows; r += 4) pd = add_rn(pd, mul_rn(piv[r], mine[r]));
                tmp = add_rn(quad_sum(quad, pd), ak);
                ak = sub_rn(ak, mul_rn(tau, tmp));
            } else if (last_row) {
                ak = mul_rn(ak, sub_rn(1.0, tau));
            }
            __syncwarp(quad);  // every lane of the quad has read the old mine[k]
            if (i == 0) mine[k] = ak;
            double p1 = 0.0, p2 = 0.0;
            int r = r0;
            FKS_QR_INNER_LOOP
            for (; r + 4 * (FKS_QR_BATCH - 1) < rows; r += 4 * FKS_QR_BATCH) {
                double v[FKS_QR_BATCH];
#pragma unroll
                for (int u = 0; u < FKS_QR_BATCH; u++) v[u] = mine[r + 4 * u];
                if (reflect) {
                    double av[FKS_QR_BATCH];
#pragma unroll
                    for (int u = 0; u < FKS_QR_BATCH; u++) av[u] = piv[r + 4 * u];
#pragma unroll
                    for (int u = 0; u < FKS_QR_BATCH; u++) {
                        v[u] = sub_rn(v[u], mul_rn(mul_rn(tau, av[u]), tmp));
                        mine[r + 4 * u] = v[u];
                    }
                }
#pragma unroll
                for (int u = 0; u < FKS_QR_BATCH; u++) {
                    const double sq = mul_rn(v[u], v[u]);
                    p1 = add_rn(p1, sq);
                    if (u > 0 || r >= k + 2) p2 = add_rn(p2, sq);  // r + 4 >= k + 2 always (r >= k + 1)
                }
            }
            FKS_QR_INNER_LOOP
            for (; r < rows; r += 4) {
                double v = mine[r];
                if (reflect) {
                    v = sub_rn(v, mul_rn(mul_rn(tau, piv[r]), tmp));
                    mine[r] = v;
                }
                const double sq = mul_rn(v, v);
                p1 = add_rn(p1, sq);
                if (r >= k + 2) p2 = add_rn(p2, sq);
            }
            tailp[sl] = p2;
            const double direct = quad_sum(quad, p1);
            if (is_col && nu[sl] != 0.0) {  // LAPACK-style norm downdate
                double temp = div_rn(fabs(ak), nu[sl]);
                temp = mul_rn(add_rn(1.0, temp), sub_rn(1.0, temp));
                temp = temp < 0.0 ? 0.0 : temp;
                const double ratio = div_rn(nu[sl], nd[sl]);
                const double temp2 = mul_rn(temp, mul_rn(ratio, ratio));
                if (temp2 <= norm_downdate_threshold) {
                    nd[sl] = sqrt(direct);
                    nu[sl] = nd[sl];
                } else {
                    nu[sl] = mul_rn(nu[sl], sqrt(temp));
                }
            }
        }
        __syncwarp();
    }
    if (lane == 0) {
        if (near_cut) raise_flag(wb, FKS_FLAG_NEAR_RANK_CUT);
        if (forced && (differed || own_rank != nonzero_pivots)) raise_flag(wb, FKS_FLAG_DECISION_OVERRIDDEN);
    }
    // solve: back substitution on the leading nonzero_pivots x nonzero_pivots triangle, the other unknowns zero.  Lane j holds
    // position j: its column, c_j, then x_j.  Row ii: the products R(ii, j) x_j are formed by their lanes, lane ii subtracts them
    // in ascending j (Eigen's triangular solve, the oracle's order) and divides by the diagonal.
    if (lane < cols) x[lane] = 0.0;
    __syncwarp();
    {
        const double* rhs = A + (size_t)cols * ld;
        const bool mine_pos = lane < nonzero_pivots;
        const int my_col = (int)((order >> (4 * (mine_pos ? lane : 0))) & 0xFull);
        const double* colp = A + (size_t)my_col * ld;
        double xj = mine_pos ? rhs[lane] : 0.0;  // c_j until row j is solved
#pragma unroll 1
        for (int ii = nonzero_pivots - 1; ii >= 0; ii--) {
            const double prod = (mine_pos && lane > ii) ? mul_rn(colp[ii], xj) : 0.0;
            double sacc = xj;  // meaningful in lane ii
            FKS_QR_INNER_LOOP
            for (int j = ii + 1; j < nonzero_pivots; j++) sacc = sub_rn(sacc, __shfl_sync(FKS_FULL, prod, j));
            if (lane == ii) xj = div_rn(sacc, colp[ii]);
        }
        if (mine_pos) x[my_col] = xj;
    }
    __syncwarp();
}
// the solver for `cols` unknowns (+ the right-hand side): one column per quad when they fit 8 quads
__device__ __forceinline__ void colpiv_qr_solve(int wb, double* A, int ld, int rows, int cols, int x_off) {
    if (cols + 1 <= 8) colpiv_qr_lanes<1>(wb, A, ld, rows, cols, x_off);
    else colpiv_qr_lanes<2>(wb, A, ld, rows, cols, x_off);
}

// actuator noise of the next `count` microsteps, one truncated-normal draw per axis in axis order (SURVEY A.6); `pid` is the
// Philox particle id relative to first_id (leg * leg_id_stride + particle in a sequence call)
__device__ __noinline__ void fill_noise(int wb, unsigned long long pid, unsigned step, unsigned micro0, int count,
                                        unsigned long long tape_pos, unsigned long long tape_end) {
    const Frame& fr = frame();
    const int lane = lane_id();
    const int D = fr.rb.D;
    double* tn = wsd(wb) + fr.a.wl.tn;
    const int m = lane / D, dof = lane - m * D;
    if (m < count) {
        double v = 0.0;
        if (fr.a.noise_mode == FKS_NOISE_INJECTED) {
            const unsigned long long pos = tape_pos + (unsigned long long)(m * D + dof);
            if (pos < tape_end) v = fr.a.tape[pos];  // read-ahead past the end is checked where the draw is consumed
        } else if (fr.a.noise_mode == FKS_NOISE_PHILOX) {
            v = fks_philox_truncated_normal(fr.a.seed, fr.a.first_id + pid, step, micro0 + (unsigned)m, (uint32_t)dof, fr.rb.axes[dof].sigma);
        }
        tn[m * fr.a.wl.S + dof] = v;
    }
    __syncwarp();
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// The kernel: a persistent grid, ONE CTA of up to kWarpsPerBlock (24) warps per SM; a warp works on one particle at a time.
//
// The nested loops of the reference (controller step -> microstep -> resolver iteration) are flattened into a per-PARTICLE
// state machine with two kinds of phases:
//
//     ROUND   A  advance a kinematic state      apply_control / kinematics
//             B  measure it                     max_motion  or  check_collision
//             T  bookkeeping, next operation    scalar code, noise draws, particle fetch / result record
//     SOLVE   C  collect corrections            -- only for a particle whose last check found a collision --
//             D  stacked-Jacobian QR solve
//             E  motion estimate of the raw correction
//
// LOCK STEP.  All warps of the CTA run the SAME phase at the same time (a CTA barrier per cycle).  The profile of a
// free-running version showed 60 % of the issue slots lost to instruction fetch (a few hundred KB of SASS walked by the
// warps at unrelated places against a 32 KB instruction cache), and every relaxation tried since -- private rounds, late
// joiners, independent lock-step groups -- cost 5-40 % (profiles/r2_kernel_experiments.md).
//
// CONTEXT POOL.  Lock step alone wastes warps: in the contact regime a third of the rounds ends in a collision, and a warp
// tied to its particle then waits for the others' rounds while they wait for its solve.  So warps are NOT tied to
// particles: the CTA keeps `pool` (two per warp) particle CONTEXTS in flight -- configurations, link transforms,
// control vectors, noise batch, bookkeeping: ~3.5 KB for the arm, in global memory (L2) unless a warp has them loaded --
// and every cycle
//     1. takes the census: how many contexts need a ROUND, how many a SOLVE;
//     2. picks the phase: SOLVE as soon as a full batch (one per warp) is waiting or nothing else can run, else ROUND;
//     3. every warp keeps its loaded context when that needs the chosen phase, else swaps it for one that does (store
//        3.5 KB, load 3.5 KB), admitting a fresh particle when a ROUND has no taker;
//     4. the phase runs once, and the census is updated.
// Solve phases are full batches, round phases are full batches, and the only idle warps are those of the last cycles.
// ------------------------------------------------------------------------------------------------
// Lock-step rounds a ROUND cycle runs while no context of the CTA is waiting for a solve (pure free flight: 3 extra).
#ifndef FKS_FREE_ROUNDS
#define FKS_FREE_ROUNDS 3
#endif
// ... and while some are (a warp whose particle collides sits out the rest of the cycle): one for the linked robots, two for
// the rigid bodies, whose rounds are short (measured: SE(2) 43.7 -> 41.9 ms, SE(3) 61.5 -> 61.2, arm_table 119.5 -> 120.8 with two)
#ifndef FKS_CONTACT_ROUNDS
#define FKS_CONTACT_ROUNDS(KIND) ((KIND) == FKS_ROBOT_LINKED ? 1 : 2)
#endif
// waiting contexts that make the CTA switch to a SOLVE cycle, as a fraction (numerator / 8) of its warps
#ifndef FKS_SOLVE_BATCH_EIGHTHS
#define FKS_SOLVE_BATCH_EIGHTHS 8
#endif
namespace {
enum { OP_NONE = 0, OP_KIN = 1, OP_APPLY = 2 };
enum { M_NONE = 0, M_MOTION = 1, M_CHECK = 2 };
enum {
    AF_FETCH = 0,       // no particle: fetch the next one
    AF_INIT,            // initial kinematics done -> begin the first controller step
    AF_EST_RU,          // motion of the whole controller step is known -> number of microsteps
    AF_EST_DU,          // motion of one microstep is known -> start the microstep loop
    AF_MICRO_CHECK,     // a noisy microstep was applied and checked
    AF_EST_RAW,         // motion of the raw correction step is known -> scale and apply it
    AF_RESOLVE_CHECK,   // a correction step was applied and checked
    AF_FAIL_KIN,        // previous configuration restored after a failed resolve
    AF_STOP_KIN,        // previous configuration restored after a collision with allow_contacts == false
    AF_NOCONTACT_KIN,   // step-start configuration restored -> the particle ends
    AF_DONE             // no particles left
};
enum { NEED_EMPTY = 0, NEED_ROUND = 1, NEED_SOLVE = 2, NEED_DEAD = 3 };  // what a context of the pool waits for
// WarpVars::leg of a sequence call: set when a leg has ended and the next one is due (AF_FETCH then continues the particle
// instead of claiming a new one).  A flag rather than an `after` state of its own: an extra case of the state machine's switch
// changes the single-call kernel's code even where it is never taken.
constexpr unsigned kLegPending = 0x80000000u;

// A context's three ranges (fks_device_types.h) between the warp's shared block and slots of the global context store, where
// they lie back to back: parks the context in the block into the slot of context park_ctx, then loads context load_ctx
// (-1: none).
// Lane 0 issues three bulk copies per direction; the lanes wait for the load only.  The park's writes are waited for at the
// end of the cycle (simulate_kernel): the next cycle's __syncthreads is where another warp may start to load that slot.
// (A per-lane copy kept the loads in registers: batches of loads in flight made the whole kernel slower through spills of
// the main loop, profiles/r2_kernel_experiments.md; the bulk copy holds nothing.)
__device__ __forceinline__ void context_swap(double* ws, int park_ctx, int load_ctx, const WarpLayout& wl) {
    const LaunchArgs& a = frame().a;
    char* store = a.ctx_store + (size_t)blockIdx.x * a.pool * a.ctx_stride;  // the CTA's slots
    double* park = reinterpret_cast<double*>(store + (size_t)park_ctx * a.ctx_stride);
    const double* load = reinterpret_cast<const double*>(store + (size_t)load_ctx * a.ctx_stride);
    const int n0 = wl.T + 2 * wl.L12 - wl.cfg, n1 = wl.L12, n2 = (wl.save2_end - wl.target + 1) & ~1;
    const unsigned bar = warp_bar();
    fence_async_shared();  // (a): every lane wrote the block (WarpVars included)
    __syncwarp();
    unsigned long long state = 0ull;
    if (lane_id() == 0) {
        if (park_ctx >= 0) {
            bulk_store(park, ws + wl.cfg, n0);
            bulk_store(park + n0, ws + wl.G, n1);
            bulk_store(park + n0 + n1, ws + wl.target, n2);
            bulk_commit();
            bulk_wait_read();  // (b): the load and a fresh context's set-up overwrite what the park reads
        }
        if (load_ctx >= 0) {
            fence_async_global();  // (a): the slot was last written by a park of some warp
            state = bulk_expect(bar, (n0 + n1 + n2) * 8);
            bulk_load(ws + wl.cfg, load, n0, bar);
            bulk_load(ws + wl.G, load + n0, n1, bar);
            bulk_load(ws + wl.target, load + n0 + n1, n2, bar);
        }
    }
    __syncwarp();  // (b) for the other lanes
    if (load_ctx >= 0) bulk_wait_loads(bar, state);
}
}  // namespace

// TRACE = true is the single-particle instantiation that records the step trace (fks_forward_simulate_traced); the batch
// kernel carries none of it.  SEQ = true is the instantiation of sequence calls (n_legs > 1, fks_forward_simulate_sequence):
// every particle runs n_legs legs; the single-call kernel has no leg logic at all (leg is 0 there).
template <int KIND, bool TRACE = false, bool SEQ = false>
__global__ void __launch_bounds__(kThreadsPerBlock, FKS_MIN_BLOCKS) simulate_kernel(const __grid_constant__ LaunchArgs args) {
    // ---- stage parameters, robot and points into shared memory, once per CTA ---------------------
    {
        Frame* f = reinterpret_cast<Frame*>(smem_raw);
        const unsigned* src = reinterpret_cast<const unsigned*>(&args);
        unsigned* dst = reinterpret_cast<unsigned*>(&f->a);
        for (int i = threadIdx.x; i < (int)(sizeof(LaunchArgs) / 4); i += blockDim.x) dst[i] = src[i];
        const unsigned* rsrc = reinterpret_cast<const unsigned*>(args.robot);
        unsigned* rdst = reinterpret_cast<unsigned*>(&f->rb);
        for (int i = threadIdx.x; i < (int)(sizeof(DevRobot) / 4); i += blockDim.x) rdst[i] = rsrc[i];
        double2* pxy = reinterpret_cast<double2*>(smem_raw + args.pts_off);
        PointZL* pzl = reinterpret_cast<PointZL*>(pxy + args.P);
        for (int i = threadIdx.x; i < args.P; i += blockDim.x) {
            pxy[i] = args.pxy[i];
            pzl[i] = args.pzl[i];
        }
        if (threadIdx.x < 12) {  // root of the world->voxel chain of the linked robot (kinematics)
            const int r = threadIdx.x >> 2, c = threadIdx.x & 3;
            const double* io = args.env.inv_origin;
            const double* bs = args.robot->base;
            double v = io[4 * r + 0] * bs[c] + io[4 * r + 1] * bs[4 + c] + io[4 * r + 2] * bs[8 + c];
            if (c == 3) v += io[4 * r + 3];
            f->gbase[threadIdx.x] = v * args.env.inv_sdf_res;
        }
        for (int q = threadIdx.x; q < args.robot->n_pairs; q += blockDim.x) {  // midpoint pre-test of the self-collision broad phase
            const DevRobot* r = args.robot;
            const int la = r->pair_a[q], lb = r->pair_b[q];
            double ha = 0.0, hb = 0.0;
            for (int k = 0; k < 3; k++) {
                const double da = r->cap_p1[la][k] - r->cap_p0[la][k], db = r->cap_p1[lb][k] - r->cap_p0[lb][k];
                ha += da * da;
                hb += db * db;
            }
            const double diag = 2.0 * 1.7320508075688772 * args.env.map_res * (1.0 + 1e-6) + 1e-9;
            const double reach = (0.5 * sqrt(ha) + 0.5 * sqrt(hb) + r->cap_radius[la] + r->cap_radius[lb] + diag) * (1.0 + 1e-9);
            f->pair_reach_sq[q] = reach * reach;
        }
    }
    __syncthreads();
    const Frame& fr = frame();
    const LaunchArgs& a = fr.a;
    const DevRobot& rb = fr.rb;
    const WarpLayout& wl = a.wl;
    const DevSolver& sp = a.sp;
    const int lane = lane_id();
    const int warp = (int)(threadIdx.x >> 5);
    const int wb = a.warps_off + warp * wl.total * 8;
    double* ws = wsd(wb);
    const int D = rb.D, S = wl.S, stride = a.cfg_stride;
    if (lane < FKS_NUM_STATS) reinterpret_cast<unsigned long long*>(ws + wl.stats)[lane] = 0ull;
    __syncwarp();
    const double target_microstep_distance = a.env.map_res * 0.125;
    const double allowed_microstep_distance = a.env.map_res * 1.0;
    WarpVars* wv = reinterpret_cast<WarpVars*>(ws + wl.vars);
    double* pid_state = ws + wl.vars + kWarpVarsDoubles;  // [0..S) integral, [S..2S) last error: lane i owns axis i

    // ---- the CTA's context pool: scheduling state in shared memory behind the warp blocks ------------------------------
    const int n_warps = a.warps_per_block, pool = a.pool;
    unsigned char* need = smem_raw + a.sync_off + 16;                     // [pool] NEED_*
    signed char* holds = reinterpret_cast<signed char*>(need + kMaxPool); // [warps] the context in the warp's block, -1: none
    volatile unsigned* exhausted = reinterpret_cast<volatile unsigned*>(smem_raw + a.sync_off);  // no particles left to admit
    for (int c = threadIdx.x; c < kMaxPool; c += blockDim.x) {
        need[c] = c < n_warps ? NEED_ROUND : (c < pool ? NEED_EMPTY : NEED_DEAD);  // context w starts out in warp w, about to fetch
        holds[c] = c < n_warps ? (signed char)c : (signed char)-1;
    }
    if (threadIdx.x == 0) *exhausted = 0u;
    if (lane == 0) {
        wv->after = AF_FETCH;
        wv->op = OP_NONE;
        wv->measure = M_NONE;
        wv->want_solve = 0;
        wv->cc = 0u;
        wv->cur = wv->prev = 0;
        wv->m_result = 0.0;
        wv->ctx = warp;
        if (SEQ) wv->leg = 0u;
        // the warp's mbarrier of its bulk loads (context_swap, move_tall_system): one arrival per phase, lane 0's
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(warp_bar()) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

#ifdef FKS_PHASE_TIMERS
    long long tacc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    long long tqr[4] = {0, 0, 0, 0};
    long long textra[4] = {0, 0, 0, 0};  // cycles, sum of solver warps over the solve cycles, solve cycles, estimate clocks
    long long t0 = clock64(), t1;
#define FKS_TICK(i) { t1 = clock64(); tacc[i] += t1 - t0; t0 = t1; }
    long long tcyc[4] = {0, 0, 0, 0};  // warp 0: clocks of round cycles, their number, clocks of solve cycles, their number
    long long tc_start = clock64();
    int last_kind = -1;
    __shared__ unsigned cyc_max[8];     // per cycle: longest A, B, T, swap, collect, solve, estimate of any warp
    long long tmax[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (threadIdx.x < 8) cyc_max[threadIdx.x] = 0u;
#define FKS_MAXTICK(i, since) { if (lane == 0) { const unsigned dt_ = (unsigned)(clock64() - (since)); atomicMax(&cyc_max[i], dt_); if ((i) == 0 || (i) == 2 || (i) == 3) atomicAdd(&g_dbg[((i) == 0 ? 40 : ((i) == 2 ? 48 : 56)) + min((int)(dt_ >> 11), 7)], 1ull); } }
#else
#define FKS_TICK(i)
#define FKS_MAXTICK(i, since)
#endif
    for (;;) {
        __syncthreads();  // the census of the previous cycle is complete (and what it parked is in global memory)
#ifdef FKS_PHASE_TIMERS
        {
            const long long now = clock64();
            if (last_kind >= 0) {
                tcyc[2 * last_kind] += now - tc_start;
                tcyc[2 * last_kind + 1] += 1;
            }
            tc_start = now;
            for (int i = 0; i < 8; i++) tmax[i] += cyc_max[i];
        }
        __syncthreads();
        if (threadIdx.x < 8) cyc_max[threadIdx.x] = 0u;
        __syncthreads();
        const long long tm_swap = clock64();
#endif
        FKS_TICK(5)
        // ---- 1. census: every warp reads the same snapshot and derives the same plan, so one barrier per cycle is enough ----
        const int n_lo = need[lane], n_hi = need[32 + lane];  // lane c / c + 32 looks at context c / c + 32 (NEED_DEAD beyond the pool)
        const int h = lane < n_warps ? (int)holds[lane] : -1; // lane w looks at warp w
        const int ns = __popc(__ballot_sync(FKS_FULL, n_lo == NEED_SOLVE)) + __popc(__ballot_sync(FKS_FULL, n_hi == NEED_SOLVE));
        const int nr = __popc(__ballot_sync(FKS_FULL, n_lo == NEED_ROUND)) + __popc(__ballot_sync(FKS_FULL, n_hi == NEED_ROUND));
        const unsigned e_lo = __ballot_sync(FKS_FULL, n_lo == NEED_EMPTY), e_hi = __ballot_sync(FKS_FULL, n_hi == NEED_EMPTY);
        const bool can_admit = (e_lo | e_hi) != 0u && *exhausted == 0u;
        if (ns + nr == 0 && !can_admit) break;  // every particle of this CTA has ended and there is none left to fetch
        // ---- 2. phase: a batch of solves as soon as it is big enough, or when the rounds run out of takers; else a round -----
        const int round_supply = nr + (can_admit ? __popc(e_lo) + __popc(e_hi) : 0);
        int want = NEED_ROUND;
        if (ns > 0 && 8 * ns >= FKS_SOLVE_BATCH_EIGHTHS * n_warps) want = NEED_SOLVE;
        else if (2 * round_supply < n_warps && ns > round_supply) want = NEED_SOLVE;
        else if (round_supply == 0) want = NEED_SOLVE;
        const bool solve_phase = want != NEED_ROUND;
#ifdef FKS_PHASE_TIMERS
        last_kind = solve_phase ? 1 : 0;
#endif
        // ---- 3. contexts: a warp keeps the one in its block when that wants this phase; the others share out, in warp
        //         order, the waiting contexts nobody holds, then (ROUND only) the empty ones, which admit fresh particles ----
        const bool keeps = h >= 0 && need[h] == want;                       // does warp `lane` keep its context?
        const unsigned keep_mask = __ballot_sync(FKS_FULL, keeps);
        const unsigned held_lo = __reduce_or_sync(FKS_FULL, (h >= 0 && h < 32) ? (1u << h) : 0u);
        const unsigned held_hi = __reduce_or_sync(FKS_FULL, (h >= 32) ? (1u << (h - 32)) : 0u);
        const unsigned r_lo = __ballot_sync(FKS_FULL, n_lo == want) & ~held_lo, r_hi = __ballot_sync(FKS_FULL, n_hi == want) & ~held_hi;
        const int my = (int)holds[warp];
        const bool keep = (keep_mask >> warp) & 1u;
        bool active = keep;
        int got = -1;
        bool fresh = false;
        if (!keep) {
            const int rank = __popc(~keep_mask & ((1u << warp) - 1u));      // my place among the warps that look for work
            const int n_r_lo = __popc(r_lo), n_ready = n_r_lo + __popc(r_hi);
            if (rank < n_ready) {
                got = rank < n_r_lo ? (int)__fns(r_lo, 0, rank + 1) : 32 + (int)__fns(r_hi, 0, rank - n_r_lo + 1);
            } else if (!solve_phase && can_admit) {
                const int k = rank - n_ready, n_e_lo = __popc(e_lo);
                if (k < n_e_lo + __popc(e_hi)) {
                    got = k < n_e_lo ? (int)__fns(e_lo, 0, k + 1) : 32 + (int)__fns(e_hi, 0, k - n_e_lo + 1);
                    fresh = true;
                }
            }
            if (got >= 0) {
                // the context in the block (if any) is not needed in this phase: it waits in the global store; the assigned
                // one comes in unless it is fresh
                context_swap(ws, my, fresh ? -1 : got, wl);
                if (fresh) {
                    // a fresh context: its first round fetches a particle
                    if (lane == 0) {
                        wv->after = AF_FETCH;
                        wv->op = OP_NONE;
                        wv->measure = M_NONE;
                        wv->want_solve = 0;
                        wv->cc = 0u;
                        wv->cur = wv->prev = 0;
                        wv->m_result = 0.0;
                        wv->ctx = got;
                        if (SEQ) wv->leg = 0u;
                    }
                    __syncwarp();
                }
                active = true;
            }
        }
        const int ctx = keep ? my : got;  // the context this warp runs in this cycle (when active)
        FKS_MAXTICK(3, tm_swap)
        FKS_TICK(1)
        // ---- 4. the phase ----------------------------------------------------------------------------------------------
        if (active) {
        int after = wv->after, op = wv->op, op_in = wv->op_in, op_out = wv->op_out, op_u = wv->op_u, op_tn = wv->op_tn,
            op_derive = wv->op_derive, measure = wv->measure, cur = wv->cur, prev = wv->prev;
        bool want_solve = wv->want_solve != 0;
        unsigned cc = wv->cc;
        double m_result = wv->m_result;
        __syncwarp();
        if (!solve_phase) {
        // pure free flight (no context of the CTA waits for a solve): several rounds per cycle, a barrier every fourth round only
        const int n_rounds = (ns == 0) ? 1 + FKS_FREE_ROUNDS : FKS_CONTACT_ROUNDS(KIND);
        for (int round = 0; round < n_rounds && !want_solve && after != AF_DONE; round++) {
        // =========================== phase A: advance a kinematic state ===============================
#ifdef FKS_PHASE_TIMERS
        const long long tmA = clock64();
#endif
        if (op == OP_KIN) kinematics<KIND>(wb, op_out, op_derive);
        else if (op == OP_APPLY) apply_control<KIND>(wb, op_in, op_out, op_u, op_tn, op_derive);
        FKS_MAXTICK(0, tmA)
        FKS_TICK(0)
        // =========================== phase B: measure =================================================
#ifdef FKS_PHASE_TIMERS
        const long long tmB = clock64();
#endif
        if (measure == M_MOTION) m_result = max_motion(wb, op_in, op_out);  // spcs:1492-1527
        else if (measure == M_CHECK) cc = check_collision<KIND>(wb, prev, cur, a.cull_mode == 2 ? ((cc & 1u) ? 0 : 1) : a.cull_mode);  // spcs:1418-1436
        FKS_MAXTICK(1, tmB)
        FKS_TICK(2)
#ifdef FKS_PHASE_TIMERS
        const long long tmT = clock64();
#endif
        // =========================== phase T: transitions =============================================
        if (!want_solve) {
        op = OP_NONE;
        measure = M_NONE;
        // Each pass of this loop handles one event; it ends as soon as the next operation is known.
        // `ev` is a small program counter: 0 = dispatch on `after`, 1 = begin controller step,
        // 2 = begin microstep, 3 = end of controller step, 4 = end of particle.
        int ev = 0;
        while (op == OP_NONE && !want_solve && after != AF_DONE) {
            __syncwarp();  // the WarpVars updates below are read-modify-writes done by every lane with the same value
            if (ev == 0) {
                switch (after) {
                    case AF_FETCH: {
                        // ForwardSimulateRobot (spcs:824-829): clone + ResetPosition(start).  The start of a fresh particle is
                        // its entry of `starts`; a later leg of a sequence call starts where the previous leg left the
                        // particle, as the next call of a chain of single calls would, and its tape positions run on.
                        const bool next_leg = SEQ && (wv->leg & kLegPending) != 0u;
                        const unsigned leg = next_leg ? wv->leg & ~kLegPending : 0u;
                        const double* start = ws + wl.cfg + cur * S;
                        if (!next_leg) {
                            unsigned long long next_id = 0ull;
                            if (lane == 0) next_id = (unsigned long long)atomicAdd(a.counter, 1u);
                            next_id = __shfl_sync(FKS_FULL, next_id, 0);
                            wv->pid = next_id;  // every lane stores the same value
                            if (next_id >= a.n_particles) {
                                after = AF_DONE;
                                break;
                            }
                            start = a.starts + (size_t)wv->pid * stride;
                        }
                        cur = 0;
                        const double* tgt = a.targets + (a.n_targets == a.n_particles ? (size_t)wv->pid * stride : 0);
                        if (SEQ) tgt += (size_t)leg * a.n_targets * stride;  // targets are leg-major
                        if (lane < stride) {
                            ws[wl.cfg + lane] = start[lane];
                            ws[wl.target + lane] = tgt[lane];
                        }
                        if (lane == 0) *reinterpret_cast<unsigned*>(ws + wl.flags) = 0u;
                        __syncwarp();
                        if (SEQ) wv->leg = leg;  // every lane has read the pending flag above
                        if (lane < S) {  // pid:98-102 zeroed
                            pid_state[lane] = 0.0;
                            pid_state[S + lane] = 0.0;
                        }
                        if (!next_leg) {
                            wv->tape_pos = wv->tape_end = 0ull;
                            if (a.noise_mode == FKS_NOISE_INJECTED) {
                                wv->tape_pos = a.tape_off[wv->pid];
                                wv->tape_end = a.tape_off[wv->pid + 1];
                            }
                            wv->dec_pos = wv->dec_end = 0ull;
                            if (a.dec_tape != nullptr) {
                                wv->dec_pos = a.dec_off[wv->pid];
                                wv->dec_end = a.dec_off[wv->pid + 1];
                            }
                        }
                        wv->collided = wv->any_resolve_failed = false;
                        wv->flags = wv->n_micro_total = wv->n_iter_total = wv->n_steps = 0u;
                        wv->step = 0u;
                        op = OP_KIN;
                        op_out = cur;
                        op_derive = 1;
                        after = AF_INIT;
                        break;
                    }
                    case AF_INIT:
                        ev = 1;
                        break;
                    case AF_EST_RU: {  // spcs:1559-1568
                        const double ratio = m_result / target_microstep_distance;
                        wv->number_microsteps = (unsigned)ceil(ratio);
                        if (wv->number_microsteps < 1u) wv->number_microsteps = 1u;
                        if (lane < D) ws[wl.du + lane] = ws[wl.ru + lane] / (double)wv->number_microsteps;
                        __syncwarp();
                        if (FKS_SKIP_SINGLE_ESTIMATE && wv->number_microsteps == 1u) {
                            // control_input_step == real_control_input bit for bit (x / 1.0): its motion estimate
                            // (spcs:1569) is the one just computed
                            after = AF_EST_DU;
                            break;
                        }
                        op = OP_APPLY; op_in = cur; op_out = 2; op_u = wl.du; op_tn = -1; op_derive = 0;
                        measure = M_MOTION;
                        after = AF_EST_DU;
                        break;
                    }
                    case AF_EST_DU:  // spcs:1569-1575
                        if (m_result > allowed_microstep_distance) wv->flags |= FKS_FLAG_WOULD_ASSERT_MICROSTEP;
                        if (TRACE) {  // spcs:1583-1588
                            trace_append(FKS_TRACE_CONTROL_INPUT, wv->step, 0u, 0u, ws + wl.ru, D);
                            trace_append(FKS_TRACE_CONTROL_INPUT_STEP, wv->step, 0u, 0u, ws + wl.du, D);
                        }
                        wv->step_collided = wv->step_failed = wv->step_stopped = false;
                        wv->micro = 0u;
                        ev = 2;
                        break;
                    case AF_MICRO_CHECK: {  // spcs:1608-1625
                        const bool in_collision = (cc & 1u) != 0u;
                        if (in_collision) wv->step_collided = true;
                        if (TRACE) {
                            trace_append(FKS_TRACE_POST_ACTION, wv->step, wv->micro, 0u, ws + wl.cfg + cur * S, stride);  // spcs:1615-1618
                            if (in_collision && !a.allow_contacts)
                                trace_append(FKS_TRACE_RETURNED_PREVIOUS, wv->step, wv->micro, 0u, ws + wl.cfg + prev * S, stride);  // spcs:1778
                        }
                        if (in_collision && a.allow_contacts) {
                            wv->resolver_iterations = 0u;
                            wv->scaling = sp.initial_step;
                            want_solve = true;
                        } else if (in_collision) {  // spcs:1769-1786
                            if (lane == 0) add_stat(wb, FKS_STAT_SUCCESSFUL_RESOLVES, 1ull);
                            cur = prev;
                            wv->step_stopped = true;
                            op = OP_KIN; op_out = cur; op_derive = 1;
                            after = AF_STOP_KIN;
                        } else {
                            ev = (wv_add(&wv->micro, 1u) < wv->number_microsteps) ? 2 : 3;
                        }
                        break;
                    }
                    case AF_EST_RAW: {  // spcs:1681-1689
                        const double step_fraction = fmax(m_result / allowed_microstep_distance, 1.0);
                        if (lane < D) ws[wl.stepv + lane] = (ws[wl.raw + lane] / step_fraction) * fabs(wv->scaling);
                        __syncwarp();
                        op = OP_APPLY; op_in = cur; op_out = cur; op_u = wl.stepv; op_tn = -1; op_derive = 1;
                        measure = M_CHECK;
                        after = AF_RESOLVE_CHECK;
                        break;
                    }
                    case AF_RESOLVE_CHECK: {  // spcs:1694-1761
                        const bool in_collision = (cc & 1u) != 0u;
                        wv_add(&wv->resolver_iterations, 1u);
                        wv_add(&wv->n_iter_total, 1u);
                        __syncwarp();
                        if (TRACE) {
                            __syncwarp();
                            trace_append(FKS_TRACE_RESOLUTION_STEP, wv->step, wv->micro, wv->resolver_iterations, ws + wl.cfg + cur * S, stride);  // spcs:1703
                            if (wv->resolver_iterations > sp.max_iters)
                                trace_append(FKS_TRACE_RETURNED_PREVIOUS, wv->step, wv->micro, wv->resolver_iterations, ws + wl.cfg + prev * S, stride);  // spcs:1714
                        }
                        if (wv->resolver_iterations > sp.max_iters) {  // spcs:1705-1746
                            if (lane == 0) {
                                add_stat(wb, FKS_STAT_UNSUCCESSFUL_RESOLVES, 1ull);
                                add_stat(wb, (cc & 2u) ? FKS_STAT_UNSUCCESSFUL_SELF_COLLISION_RESOLVES : FKS_STAT_UNSUCCESSFUL_ENV_COLLISION_RESOLVES, 1ull);
                            }
                            cur = prev;  // return previous_configuration
                            wv->step_collided = true;
                            wv->step_failed = true;
                            op = OP_KIN; op_out = cur; op_derive = 1;
                            after = AF_FAIL_KIN;
                            break;
                        }
                        if ((wv->resolver_iterations % sp.decay_iters) == 0u) {  // spcs:1747-1761
                            double sc = wv->scaling;
                            if (sc >= 0.0) {
                                sc = sc * sp.decay_rate;
                                if (sc < sp.min_scaling) sc = -sp.min_scaling;
                            } else {
                                sc = -sp.min_scaling;
                            }
                            __syncwarp();
                            wv->scaling = sc;
                        }
                        if (in_collision) {
                            want_solve = true;
                        } else {
                            ev = (wv_add(&wv->micro, 1u) < wv->number_microsteps) ? 2 : 3;
                        }
                        break;
                    }
                    case AF_FAIL_KIN:
                    case AF_STOP_KIN:
                        ev = 3;
                        break;
                    case AF_NOCONTACT_KIN:
                        ev = 4;
                        break;
                    default:
                        break;
                }
            } else if (ev == 1) {
                // ---- begin controller step: GenerateControlAction (tnuva:179-198, :384-412, :598-614) --------
                ev = 0;
                wv_add(&wv->n_steps, 1u);
                double* cfg = ws + wl.cfg + cur * S;
                if (!a.allow_contacts) {  // a colliding wv->step is discarded as a whole: keep the wv->step's start (spcs:904-909)
                    if (lane < stride) ws[wl.scfg + lane] = cfg[lane];
                    __syncwarp();
                }
                if (KIND == FKS_ROBOT_SE3) {
                    if (lane == 0) {
                        double c12[12], tg[12], tw[6];
#pragma unroll
                        for (int i = 0; i < 12; i++) {
                            c12[i] = cfg[i];
                            tg[i] = ws[wl.target + i];
                        }
                        twist_between(c12, tg, tw);
#pragma unroll
                        for (int i = 0; i < 6; i++) ws[wl.stepv + i] = tw[i];
                    }
                    __syncwarp();
                }
                if (lane < D) {
                    double err;
                    if (KIND == FKS_ROBOT_SE2) {
                        err = ws[wl.target + lane] - cfg[lane];
                        if (lane == 2) err = wrap_angle(err);
                    } else if (KIND == FKS_ROBOT_SE3) {
                        err = ws[wl.stepv + lane];
                    } else {
                        err = ws[wl.target + lane] - cfg[lane];
                        if (rb.joints[rb.active_joint[lane]].type == FKS_JOINT_CONTINUOUS) err = wrap_angle(err);
                    }
                    // SimplePIDController::ComputeFeedbackTerm (wv->pid:122-135)
                    const DevAxis& ax = rb.axes[lane];
                    const double dt = sp.interval;
                    const double timestep_error_integral = ((err * 0.5) + (pid_state[S + lane] * 0.5)) * dt;
                    const double new_error_integral = pid_state[lane] + timestep_error_integral;
                    pid_state[lane] = fmax(-ax.iclamp, fmin(ax.iclamp, new_error_integral));
                    const double error_derivative = (err - pid_state[S + lane]) / dt;
                    pid_state[S + lane] = err;
                    const double term = (err * ax.kp) + (pid_state[lane] * ax.ki) + (error_derivative * ax.kd);
                    const double action = actuate(wb, ax, term, false, 0.0);
                    ws[wl.act + lane] = action;
                    ws[wl.ru + lane] = action * sp.interval;  // real_control_input (spcs:1549)
                }
                __syncwarp();
                // ResolveForwardSimulation (spcs:1546-1816) starts with the motion estimate of the whole wv->step
                op = OP_APPLY; op_in = cur; op_out = 2; op_u = wl.ru; op_tn = -1; op_derive = 0;
                measure = M_MOTION;
                after = AF_EST_RU;
            } else if (ev == 2) {
                // ---- begin microstep (spcs:1590-1608) ---------------------------------------------------------
                ev = 0;
                wv_add(&wv->n_micro_total, 1u);
                const int nb = wl.noise_batch;
                const int slot = (int)(wv->micro % (unsigned)nb);
                if (slot == 0) {
                    const unsigned left = wv->number_microsteps - wv->micro;
                    const unsigned long long noise_id = SEQ ? wv->pid + (unsigned long long)wv->leg * a.leg_id_stride : wv->pid;
                    fill_noise(wb, noise_id, wv->step, wv->micro, left < (unsigned)nb ? (int)left : nb, wv->tape_pos, wv->tape_end);
                }
                if (a.noise_mode == FKS_NOISE_INJECTED && wv->tape_pos + (unsigned long long)D > wv->tape_end) wv->flags |= FKS_FLAG_TAPE_EXHAUSTED;
                wv_add(&wv->tape_pos, (unsigned long long)D);
                // previous_configuration (spcs:1597) is the old current state; the new one is built in the other buffer
                prev = cur;
                cur ^= 1;
                op = OP_APPLY; op_in = prev; op_out = cur; op_u = wl.du; op_tn = wl.tn + slot * S; op_derive = 1;  // spcs:1599-1601
                measure = M_CHECK;
                after = AF_MICRO_CHECK;
            } else if (ev == 3) {
                // ---- end of controller step (spcs:1797-1815, then back in ForwardSimulateMutableRobot :873-909) ----
                ev = 0;
                if (!wv->step_failed && !wv->step_stopped && lane == 0) {
                    add_stat(wb, FKS_STAT_SUCCESSFUL_RESOLVES, 1ull);
                    add_stat(wb, wv->step_collided ? FKS_STAT_COLLISION_RESOLVES : FKS_STAT_FREE_RESOLVES, 1ull);
                }
                bool ends = false;
                if (a.allow_contacts || !wv->step_collided) {
                    if (wv->step_collided) wv->collided = true;
                    if (wv->step_failed) {
                        wv->flags |= FKS_FLAG_RESOLVE_FAILED;
                        if (sp.failed_ends_motion) {
                            wv->flags |= FKS_FLAG_ENDED_BY_FAILURE;
                            ends = true;
                        }
                        wv->any_resolve_failed = true;
                    } else if (wv->any_resolve_failed) {
                        if (lane == 0) add_stat(wb, FKS_STAT_RECOVERED_UNSUCCESSFUL_RESOLVES, 1ull);
                    }
                    if (!ends && sp.shortcut_distance > 0.0) {  // ComputeConfigurationDistanceTo (spcs:898); never < 0
                        const double dist = config_distance<KIND>(rb, ws + wl.cfg + cur * S, ws + wl.target);
                        if (dist < sp.shortcut_distance) {
                            wv->flags |= FKS_FLAG_ENDED_BY_SHORTCUT;
                            ends = true;
                        }
                    }
                    const unsigned next_step = wv_add(&wv->step, 1u);
                    if (!ends && next_step < sp.n_steps) ev = 1;
                    else ev = 4;
                } else {
                    // robot->SetPosition(resolved_configuration) is skipped: the particle stays where the wv->step began
                    if (lane < stride) ws[wl.cfg + cur * S + lane] = ws[wl.scfg + lane];
                    __syncwarp();
                    wv->flags |= FKS_FLAG_ENDED_BY_NOCONTACT;
                    op = OP_KIN; op_out = cur; op_derive = 1;
                    after = AF_NOCONTACT_KIN;
                }
            } else {
                // ---- end of particle (of its leg): result record = cfg_stride doubles + fks_result_tail, leg-major --------
                ev = 0;
                if (wv->collided) wv->flags |= FKS_FLAG_DID_CONTACT;
                __syncwarp();
                wv->flags |= *reinterpret_cast<const unsigned*>(ws + wl.flags);
                char* rec = a.results + (size_t)wv->pid * a.rec_stride;
                if (SEQ) rec += (size_t)wv->leg * a.n_particles * a.rec_stride;  // records are leg-major
                if (lane < stride) reinterpret_cast<double*>(rec)[lane] = ws[wl.cfg + cur * S + lane];
                if (lane == 0) {
                    unsigned* tail = reinterpret_cast<unsigned*>(rec + (size_t)stride * 8);
                    tail[0] = wv->flags;
                    tail[1] = wv->n_micro_total;
                    tail[2] = wv->n_iter_total;
                    tail[3] = wv->n_steps;
                    add_stat(wb, FKS_STAT_TOTAL_MICROSTEPS, wv->n_micro_total);
                    add_stat(wb, FKS_STAT_TOTAL_RESOLVER_ITERATIONS, wv->n_iter_total);
                }
                __syncwarp();
                after = AF_FETCH;
                if (SEQ && wv->leg + 1u < (unsigned)a.n_legs) wv_add(&wv->leg, 1u | kLegPending);  // the next fetch continues it
            }
        }
        }  // end of phase T
        FKS_MAXTICK(2, tmT)
        FKS_TICK(4)
        }  // rounds
        } else {
        // =========================== SOLVE: phase C, collect corrections (spcs:1627) ====================
            int rows = 0;
#ifdef FKS_PHASE_TIMERS
            const long long tc0 = clock64();
            textra[1] += 1;
#endif
            rows = collect_corrections<KIND>(wb, prev, cur, (cc & 2u) != 0u);
            if (lane == 0) add_stat(wb, FKS_STAT_TOTAL_CORRECTED_POINTS, (unsigned long long)(rows / 3));
            // where collect_corrections left the system: the small store, the bigger one, or the warp's global slot
            double* jstore = ws + wl.jsm;
            int jld = wl.jsm_ld;
            if (rows > (wl.jsm_ld / 3) * 3) {
                jld = wl.jsm_big_ld;
                if (rows > jld) {
                    jstore = warp_jstore();
                    jld = a.sl.ldj;
                }
            }
#ifdef FKS_PHASE_TIMERS
            tacc[10] += clock64() - tc0;
            tacc[11] += 1;
#endif
            FKS_MAXTICK(4, tc0)
            FKS_TICK(6)
            {
            // ======================= phase D: stacked-Jacobian solve (spcs:1629,1990-1998) ==============
#ifdef FKS_PHASE_TIMERS
            const long long tq0 = clock64();
#endif
            if (rows == 0) {
                // Eigen would return an empty vector and ApplyControlInput would assert; documented device
                // behaviour: zero correction step
                wv->flags |= FKS_FLAG_EMPTY_JACOBIAN;
                if (lane < D) ws[wl.raw + lane] = 0.0;
                __syncwarp();
            } else {
                colpiv_qr_solve(wb, jstore, jld, rows, D, wl.raw);
                __syncwarp();
            }
#ifdef FKS_PHASE_TIMERS
            if (jstore == ws + wl.jsm) { tqr[0] += clock64() - tq0; tqr[1] += 1; } else { tqr[2] += clock64() - tq0; tqr[3] += 1; }
            FKS_MAXTICK(5, tq0)
            const long long te0 = clock64();
#endif
            // ======================= phase E: motion estimate of the raw correction (spcs:1630) =========
            apply_control<KIND>(wb, cur, 2, wl.raw, -1, 0);
            m_result = max_motion(wb, cur, 2);
#ifdef FKS_PHASE_TIMERS
            textra[3] += clock64() - te0;
#endif
            FKS_MAXTICK(6, te0)
            {  // spcs:1681-1689
                const double step_fraction = fmax(m_result / allowed_microstep_distance, 1.0);
                if (lane < D) ws[wl.stepv + lane] = (ws[wl.raw + lane] / step_fraction) * fabs(wv->scaling);
                __syncwarp();
            }
            op = OP_APPLY; op_in = cur; op_out = cur; op_u = wl.stepv; op_tn = -1; op_derive = 1;
            measure = M_CHECK;
            after = AF_RESOLVE_CHECK;
            want_solve = false;
            }
            FKS_TICK(8)
        }
        // the context's control state goes back to its block, its need into the census
        __syncwarp();
        if (lane == 0) {
            wv->after = after; wv->op = op; wv->op_in = op_in; wv->op_out = op_out; wv->op_u = op_u; wv->op_tn = op_tn;
            wv->op_derive = op_derive; wv->measure = measure; wv->cur = cur; wv->prev = prev;
            wv->want_solve = want_solve ? 1 : 0;
            wv->cc = cc;
            wv->m_result = m_result;
            // (written here, not when the context was taken over: other warps may still be reading the census)
            holds[warp] = (signed char)ctx;
            need[ctx] = want_solve ? NEED_SOLVE : (after == AF_DONE ? NEED_DEAD : NEED_ROUND);
            if (after == AF_DONE) *exhausted = 1u;
            // (b) of the bulk copies: a park of this cycle is complete before the next __syncthreads, after which any warp
            // may load that slot (only a warp that runs a context parks one; none is outstanding when the CTA exits)
            bulk_wait_all();
        }
        __syncwarp();
        }  // active
#ifdef FKS_PHASE_TIMERS
        textra[0] += 1;
        if (solve_phase) textra[2] += 1;
#endif
        FKS_TICK(9)
    }
#ifdef FKS_PHASE_TIMERS
    if (lane == 0)
    {
        for (int i = 0; i < 12; i++) atomicAdd(a.stats + 16 + i, (unsigned long long)tacc[i]);
        for (int i = 0; i < 4; i++) atomicAdd(a.stats + 28 + i, (unsigned long long)tqr[i]);
        for (int i = 0; i < 4; i++) atomicAdd(a.stats + 32 + i, (unsigned long long)textra[i]);
        if (warp == 0) {
            for (int i = 0; i < 4; i++) atomicAdd(a.stats + 36 + i, (unsigned long long)tcyc[i]);
            for (int i = 0; i < 8; i++) atomicAdd(a.stats + 40 + i, (unsigned long long)tmax[i]);
        }
    }
#endif
    __syncwarp();
    if (lane < FKS_NUM_STATS) {
        const unsigned long long v = reinterpret_cast<const unsigned long long*>(ws + wl.stats)[lane];
        if (v) atomicAdd(a.stats + lane, v);
    }
}

// ------------------------------------------------------------------------------------------------
// CheckConfigCollision (spcs:1398-1416), the planner-side static query, batched: one warp per configuration.
//   environment: CheckEnvironmentCollision with threshold inflation_ratio * map resolution (spcs:1403,1405)
//   self:        CheckSelfCollisions (spcs:1324-1396): two points of links whose pair is not allowed share a cell of
//                edge (inflation_ratio + 1) * map resolution (spcs:1404) -- same capsule broad phase, same cell keys
// ------------------------------------------------------------------------------------------------
namespace {
__device__ __noinline__ bool self_collision_bool(int wb, int X, double check_resolution) {
    const Frame& fr = frame();
    const DevRobot& rb = fr.rb;
    const DevEnv& e = fr.a.env;
    const WarpLayout& wl = fr.a.wl;
    if (rb.n_pairs == 0) return false;  // spcs:1327-1338
    const int lane = lane_id();
    const int P = fr.a.P;
    const double* ws = wsd(wb);
    const double* T = ws + wl.T + X * wl.L12;
    const double* caps = ws + wl.caps;
    const double2* pxy = reinterpret_cast<const double2*>(smem_raw + fr.a.pts_off);
    const PointZL* pzl = reinterpret_cast<const PointZL*>(pxy + P);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(context_scratch(wb) + fr.a.sl.keys);
    const double diag = 2.0 * 1.7320508075688772 * check_resolution * (1.0 + 1e-6) + 1e-9;  // cells at index 0 are two cells wide
    bool found = false;
    bool keys_ready = false;
    const int nch = (rb.n_pairs + 31) >> 5;
    for (int ch = 0; ch < nch && !found; ch++) {
        const int q = ch * 32 + lane;
        bool hit = false;
        if (q < rb.n_pairs) {
            const int a = rb.pair_a[q], b = rb.pair_b[q];
            const double d2 = segment_distance_sq(caps + 6 * a, caps + 6 * a + 3, caps + 6 * b, caps + 6 * b + 3);
            const double reach = rb.cap_radius[a] + rb.cap_radius[b] + diag;
            hit = d2 <= reach * reach;
        }
        unsigned m = __ballot_sync(FKS_FULL, hit);
        if (m && !keys_ready) {
            // cell keys of every point at the check resolution (LocationToExtendedGridIndex, spcs:1173-1181,1360)
            for (int p = lane; p < P; p += 32) {
                double wx, wy, wz;
                apply_T(T + 12 * pzl[p].link, pxy[p].x, pxy[p].y, pzl[p].z, wx, wy, wz);
                const double gx = e.inv_origin[0] * wx + e.inv_origin[1] * wy + e.inv_origin[2] * wz + e.inv_origin[3];
                const double gy = e.inv_origin[4] * wx + e.inv_origin[5] * wy + e.inv_origin[6] * wz + e.inv_origin[7];
                const double gz = e.inv_origin[8] * wx + e.inv_origin[9] * wy + e.inv_origin[10] * wz + e.inv_origin[11];
                const long long kx = (long long)(gx / check_resolution), ky = (long long)(gy / check_resolution), kz = (long long)(gz / check_resolution);
                keys[p] = ((unsigned long long)kx & 0x1FFFFFull) | (((unsigned long long)ky & 0x1FFFFFull) << 21) |
                          (((unsigned long long)kz & 0x1FFFFFull) << 42);
            }
            __syncwarp();
            keys_ready = true;
        }
        while (m && !found) {
            const int qq = ch * 32 + (__ffs(m) - 1);
            m &= m - 1u;
            const int la = rb.pair_a[qq], lb = rb.pair_b[qq];
            const int b0 = rb.link_begin[lb], b1 = rb.link_begin[lb + 1];
            for (int base = rb.link_begin[la]; base < rb.link_begin[la + 1] && !found; base += 32) {
                const int p = base + lane;
                const bool valid = p < rb.link_begin[la + 1];
                const unsigned long long kp = valid ? keys[p] : 0ull;
                bool h = false;
                for (int j = b0; j < b1; j++) h = h || (keys[j] == kp);
                found = __any_sync(FKS_FULL, h && valid);
            }
        }
    }
    return found;
}
}  // namespace

template <int KIND>
__global__ void __launch_bounds__(kThreadsPerBlock, FKS_MIN_BLOCKS) check_config_kernel(const __grid_constant__ LaunchArgs args, double inflation_ratio,
                                                                                       unsigned char* out) {
    {
        Frame* f = reinterpret_cast<Frame*>(smem_raw);
        const unsigned* src = reinterpret_cast<const unsigned*>(&args);
        unsigned* dst = reinterpret_cast<unsigned*>(&f->a);
        for (int i = threadIdx.x; i < (int)(sizeof(LaunchArgs) / 4); i += blockDim.x) dst[i] = src[i];
        const unsigned* rsrc = reinterpret_cast<const unsigned*>(args.robot);
        unsigned* rdst = reinterpret_cast<unsigned*>(&f->rb);
        for (int i = threadIdx.x; i < (int)(sizeof(DevRobot) / 4); i += blockDim.x) rdst[i] = rsrc[i];
        double2* pxy = reinterpret_cast<double2*>(smem_raw + args.pts_off);
        PointZL* pzl = reinterpret_cast<PointZL*>(pxy + args.P);
        for (int i = threadIdx.x; i < args.P; i += blockDim.x) {
            pxy[i] = args.pxy[i];
            pzl[i] = args.pzl[i];
        }
        if (threadIdx.x < 12) {  // root of the world->voxel chain of the linked robot (kinematics)
            const int r = threadIdx.x >> 2, c = threadIdx.x & 3;
            const double* io = args.env.inv_origin;
            const double* bs = args.robot->base;
            double v = io[4 * r + 0] * bs[c] + io[4 * r + 1] * bs[4 + c] + io[4 * r + 2] * bs[8 + c];
            if (c == 3) v += io[4 * r + 3];
            f->gbase[threadIdx.x] = v * args.env.inv_sdf_res;
        }
        for (int q = threadIdx.x; q < args.robot->n_pairs; q += blockDim.x) {  // midpoint pre-test of the self-collision broad phase
            const DevRobot* r = args.robot;
            const int la = r->pair_a[q], lb = r->pair_b[q];
            double ha = 0.0, hb = 0.0;
            for (int k = 0; k < 3; k++) {
                const double da = r->cap_p1[la][k] - r->cap_p0[la][k], db = r->cap_p1[lb][k] - r->cap_p0[lb][k];
                ha += da * da;
                hb += db * db;
            }
            const double diag = 2.0 * 1.7320508075688772 * args.env.map_res * (1.0 + 1e-6) + 1e-9;
            const double reach = (0.5 * sqrt(ha) + 0.5 * sqrt(hb) + r->cap_radius[la] + r->cap_radius[lb] + diag) * (1.0 + 1e-9);
            f->pair_reach_sq[q] = reach * reach;
        }
    }
    __syncthreads();
    const Frame& fr = frame();
    const LaunchArgs& a = fr.a;
    const int lane = lane_id();
    const int wb = a.warps_off + (threadIdx.x >> 5) * a.wl.total * 8;
    double* ws = wsd(wb);
    if (lane == 0) reinterpret_cast<WarpVars*>(ws + a.wl.vars)->ctx = (int)(threadIdx.x >> 5);  // scratch slot of this warp
    __syncwarp();
    const double map_res = a.env.map_res;
    const unsigned long long warps_total = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < a.n_particles; i += warps_total) {
        if (lane < a.cfg_stride) ws[a.wl.cfg + lane] = a.starts[(size_t)i * a.cfg_stride + lane];
        __syncwarp();
        kinematics<KIND>(wb, 0, 1);  // current_robot->SetPosition(config) (spcs:1401)
        const bool envc = check_env(wb, 0, 1, inflation_ratio * map_res);
        const bool selfc = (KIND == FKS_ROBOT_LINKED) ? self_collision_bool(wb, 0, (inflation_ratio + 1.0) * map_res) : false;
        if (lane == 0) out[i] = (envc || selfc) ? 1 : 0;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// Test entry (fks_debug_qr_solve): the contact solver of the simulate kernel on caller-provided stacked systems, one
// warp per system.  `work` holds, per system, (cols + 1) columns of rows[i] doubles (column major, the right-hand side
// last) starting at offsets[i]; they are factored in place.  The solutions go to x_out (cols doubles per system), the
// FKS_FLAG_* bits the solver raised to flags_out.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) qr_solve_kernel(double* work, const unsigned long long* offsets, const int* rows, int cols, int n,
                                                       double* x_out, unsigned* flags_out) {
    Frame* f = reinterpret_cast<Frame*>(smem_raw);
    {
        unsigned* dst = reinterpret_cast<unsigned*>(f);
        for (int i = threadIdx.x; i < (int)(sizeof(Frame) / 4); i += blockDim.x) dst[i] = 0u;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        f->a.wl = make_warp_layout(1, 0, cols, cols);
        f->a.warps_off = (int)((sizeof(Frame) + 15) & ~(size_t)15);
    }
    __syncthreads();
    const Frame& fr = frame();
    const int lane = lane_id();
    const int wb = fr.a.warps_off + (threadIdx.x >> 5) * fr.a.wl.total * 8;
    double* ws = wsd(wb);
    const int warps_total = gridDim.x * (blockDim.x >> 5);
    for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps_total) {
        if (lane == 0) *reinterpret_cast<unsigned*>(ws + fr.a.wl.flags) = 0u;
        __syncwarp();
        colpiv_qr_solve(wb, work + offsets[i], rows[i], rows[i], cols, fr.a.wl.raw);
        if (lane < cols) x_out[(size_t)i * cols + lane] = ws[fr.a.wl.raw + lane];
        if (lane == 0) flags_out[i] = *reinterpret_cast<const unsigned*>(ws + fr.a.wl.flags);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// roofline micro-benchmarks (SURVEY 8d): FP64 FMA throughput and random 4-byte gather rate
// ------------------------------------------------------------------------------------------------
__global__ void fp64_peak_kernel(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0, a6 = a0 + 6.0, a7 = a0 + 7.0;
    const double m = 1.0000001, b = 1e-9;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
        a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) out[0] = s;
}

__global__ void gather_kernel(const float* __restrict__ data, unsigned long long n_mask, float* out, int iters) {
    unsigned long long x = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull + 12345ull;
    float acc = 0.f;
    for (int i = 0; i < iters; i++) {
        // 4 independent gathers per iteration (xorshift addresses)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            x ^= x << 13;
            x ^= x >> 7;
            x ^= x << 17;
            acc += __ldg(data + (x & n_mask));
        }
    }
    if (acc == 123.456f) out[0] = acc;
}

// ------------------------------------------------------------------------------------------------
// host-side launch helpers
// ------------------------------------------------------------------------------------------------
size_t simulate_smem_plan(LaunchArgs* args, int L, int J, int D, int P, int stride, int warps_per_block, size_t smem_limit) {
    args->sl = make_scratch_layout(D, P);
    args->P = P;
    args->warps_per_block = warps_per_block;
    const size_t pts_off = (sizeof(Frame) + 15) & ~(size_t)15;
    const size_t warps_off = pts_off + (size_t)P * (sizeof(double2) + sizeof(PointZL));
    // shared-memory Jacobian store: whatever the CTA leaves free goes to it, up to every point of the robot (3 P rows)
    const WarpLayout w0 = make_warp_layout(L, J, D, stride, 0);
    const size_t base = warps_off + (size_t)warps_per_block * w0.total * 8 + kSyncBytes;
    int extra = 0;
    if (smem_limit > base) {
        const long long spare = (long long)((smem_limit - base) / (size_t)warps_per_block / 8);
        int want_ld = 3 * P < 255 ? 3 * P : 255;
        want_ld |= 1;
        const long long want = (long long)(D + 1) * want_ld - (long long)(12 * L + 16 * J + 6 * L);
        long long e = want < spare ? want : spare;
        if (e < 0) e = 0;
        extra = (int)(e & ~1ll);
        // (the layout pads for alignment: step back until the CTA fits again)
        while (extra > 0 && warps_off + (size_t)warps_per_block * make_warp_layout(L, J, D, stride, extra).total * 8 + kSyncBytes > smem_limit) extra -= 2;
    }
    args->wl = make_warp_layout(L, J, D, stride, extra);
    args->pts_off = (int)pts_off;
    args->warps_off = (int)warps_off;
    size_t off = warps_off + (size_t)warps_per_block * args->wl.total * 8;
    args->sync_off = (int)off;  // CTA-level scheduling state (context pool)
    off += kSyncBytes;
    // Bulk copies (context_swap, move_tall_system) move whole 16-byte units between 16-byte boundaries: every
    // warp block, range start and length, and store column they move has to sit on an even double.  0: it does not
    const WarpLayout& w = args->wl;
    const int ranges[] = {w.total, w.cfg, w.T + 2 * w.L12 - w.cfg, w.G, w.L12, w.target, w.jsm, w.jsm_ld, w.jsm_big_ld,
                          args->sl.ldj};
    bool aligned = warps_off % 16 == 0 && (w.save2_end + 1) / 2 * 2 <= w.total;
    for (int v : ranges) aligned = aligned && v % 2 == 0;
    return aligned ? off : 0;
}

template <int KIND>
static const void* kernel_ptr_of(bool trace, bool seq) {
    if (trace) return (const void*)simulate_kernel<KIND, true>;
    return seq ? (const void*)simulate_kernel<KIND, false, true> : (const void*)simulate_kernel<KIND>;
}
static const void* kernel_ptr(int kind, bool trace = false, bool seq = false) {
    switch (kind) {
        case FKS_ROBOT_SE2: return kernel_ptr_of<FKS_ROBOT_SE2>(trace, seq);
        case FKS_ROBOT_SE3: return kernel_ptr_of<FKS_ROBOT_SE3>(trace, seq);
        case FKS_ROBOT_LINKED: return kernel_ptr_of<FKS_ROBOT_LINKED>(trace, seq);
    }
    return nullptr;
}

// (the third range rounded up to whole 16-byte units as context_swap moves it; slots on 128-byte boundaries)
size_t context_bytes(const WarpLayout& wl) {
    const size_t bytes = (size_t)((wl.T + 2 * wl.L12 - wl.cfg) + wl.L12 + ((wl.save2_end - wl.target + 1) & ~1)) * 8;
    return (bytes + 127) & ~(size_t)127;
}

int simulate_kernel_info(int kind, size_t dyn_smem, int warps_per_block, KernelInfo* out) {
    const void* fn = kernel_ptr(kind);
    if (!fn) return (int)cudaErrorInvalidValue;
    cudaError_t err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem);
    if (err != cudaSuccess) return (int)err;
    cudaFuncAttributes fa;
    err = cudaFuncGetAttributes(&fa, fn);
    if (err != cudaSuccess) return (int)err;
    int nb = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, 32 * warps_per_block, dyn_smem);
    if (err != cudaSuccess) return (int)err;
    out->regs = fa.numRegs;
    out->static_smem = (int)fa.sharedSizeBytes;
    out->local_bytes = (int)fa.localSizeBytes;
    out->max_blocks_per_sm = nb;
    out->dyn_smem = dyn_smem;
    return 0;
}

int launch_simulate(int kind, const LaunchArgs& args, int grid, size_t dyn_smem, void* stream,
                    const void* l2_window_base, size_t l2_window_bytes) {
    const int block_threads = 32 * args.warps_per_block;
    const void* fn = kernel_ptr(kind, args.trace != nullptr, args.n_legs > 1);
    if (!fn) return (int)cudaErrorInvalidValue;
    {
        // the attribute is per function and per device, and simulators of the same robot kind share the function: set it for
        // THIS launch (a second simulator with a smaller robot must not lower the limit under a live one)
        const cudaError_t err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem);
        if (err != cudaSuccess) return (int)err;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block_threads);
    cfg.dynamicSmemBytes = dyn_smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    int nattr = 0;
    if (l2_window_base && l2_window_bytes) {
        attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(l2_window_base);
        attr[0].val.accessPolicyWindow.num_bytes = l2_window_bytes;
        attr[0].val.accessPolicyWindow.hitRatio = 1.0f;
        attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        nattr = 1;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
    void* params[1] = {const_cast<LaunchArgs*>(&args)};
    return (int)cudaLaunchKernelExC(&cfg, fn, params);
}

int launch_check_config(int kind, const LaunchArgs& args, int grid, size_t dyn_smem, void* stream, double inflation_ratio, unsigned char* out) {
    const int threads = 32 * args.warps_per_block;
    cudaError_t err;
    switch (kind) {
        case FKS_ROBOT_SE2:
            if ((err = cudaFuncSetAttribute(check_config_kernel<FKS_ROBOT_SE2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem)) != cudaSuccess) return (int)err;
            check_config_kernel<FKS_ROBOT_SE2><<<grid, threads, dyn_smem, (cudaStream_t)stream>>>(args, inflation_ratio, out);
            break;
        case FKS_ROBOT_SE3:
            if ((err = cudaFuncSetAttribute(check_config_kernel<FKS_ROBOT_SE3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem)) != cudaSuccess) return (int)err;
            check_config_kernel<FKS_ROBOT_SE3><<<grid, threads, dyn_smem, (cudaStream_t)stream>>>(args, inflation_ratio, out);
            break;
        case FKS_ROBOT_LINKED:
            if ((err = cudaFuncSetAttribute(check_config_kernel<FKS_ROBOT_LINKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem)) != cudaSuccess) return (int)err;
            check_config_kernel<FKS_ROBOT_LINKED><<<grid, threads, dyn_smem, (cudaStream_t)stream>>>(args, inflation_ratio, out);
            break;
        default:
            return (int)cudaErrorInvalidValue;
    }
    return (int)cudaGetLastError();
}

int launch_qr_solve(double* work, const unsigned long long* offsets, const int* rows, int cols, int n, double* x_out, unsigned* flags_out,
                    void* stream) {
    const int warps = 4;
    const WarpLayout wl = make_warp_layout(1, 0, cols, cols);
    const size_t smem = ((sizeof(Frame) + 15) & ~(size_t)15) + (size_t)warps * wl.total * 8;
    cudaError_t err = cudaFuncSetAttribute(qr_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return (int)err;
    const int grid = (n + warps - 1) / warps < 4096 ? (n + warps - 1) / warps : 4096;
    qr_solve_kernel<<<grid, 32 * warps, smem, (cudaStream_t)stream>>>(work, offsets, rows, cols, n, x_out, flags_out);
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// SURVEY 8(f)-3: the first consumer of a batch, on the device.  The planner (uncertainty_planning_core.cpp:97-99) splits the
// returned particles by did_contact and groups them by configuration distance; with these two kernels the end-state records
// stay in HBM between ForwardSimulateRobots and that step.  Records are cfg_stride doubles + fks_result_tail.
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
    __shared__ double from[kMaxDof < 12 ? 12 : kMaxDof];
    const unsigned a = blockIdx.y, b = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t ia = subset ? subset[a] : a;
    if ((int)threadIdx.x < cfg_stride) from[threadIdx.x] = reinterpret_cast<const double*>(results + ia * rec_stride)[threadIdx.x];
    __syncthreads();
    if (b >= m) return;
    const size_t ib = subset ? subset[b] : b;
    out[(size_t)a * m + b] = config_distance<KIND>(*robot, from, reinterpret_cast<const double*>(results + ib * rec_stride));
}

int launch_partition(const char* results, size_t rec_stride, int cfg_stride, size_t n, unsigned* block_counts, unsigned long long* totals,
                     unsigned* order, void* stream) {
    const unsigned n_blocks = (unsigned)((n + kPartitionBlock - 1) / kPartitionBlock);
    cudaStream_t st = (cudaStream_t)stream;
    partition_count_kernel<<<n_blocks, kPartitionBlock, 0, st>>>(results, rec_stride, cfg_stride, n, block_counts);
    partition_scan_kernel<<<1, kPartitionBlock, 0, st>>>(block_counts, n_blocks, n, totals);
    partition_scatter_kernel<<<n_blocks, kPartitionBlock, 0, st>>>(results, rec_stride, cfg_stride, n, block_counts, totals, order);
    return (int)cudaGetLastError();
}
int launch_pairwise_distance(int kind, const DevRobot* robot, const char* results, size_t rec_stride, int cfg_stride, const unsigned* subset,
                             unsigned m, double* out, void* stream) {
    const dim3 grid((m + 255) / 256, m);
    cudaStream_t st = (cudaStream_t)stream;
    switch (kind) {
        case FKS_ROBOT_SE2: pairwise_distance_kernel<FKS_ROBOT_SE2><<<grid, 256, 0, st>>>(robot, results, rec_stride, cfg_stride, subset, m, out); break;
        case FKS_ROBOT_SE3: pairwise_distance_kernel<FKS_ROBOT_SE3><<<grid, 256, 0, st>>>(robot, results, rec_stride, cfg_stride, subset, m, out); break;
        case FKS_ROBOT_LINKED: pairwise_distance_kernel<FKS_ROBOT_LINKED><<<grid, 256, 0, st>>>(robot, results, rec_stride, cfg_stride, subset, m, out); break;
        default: return (int)cudaErrorInvalidValue;
    }
    return (int)cudaGetLastError();
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
// ---------------------------------------------------------------------------------------------
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

__device__ __forceinline__ bool cluster_key_less(double d, unsigned i, double e, unsigned j) { return d < e || (d == e && i < j); }

// (d, i) of the warp's smallest key, in every lane
__device__ __forceinline__ void cluster_warp_min(double& d, unsigned& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(FKS_FULL, d, o);
        const unsigned oi = __shfl_xor_sync(FKS_FULL, i, o);
        if (cluster_key_less(od, oi, d, i)) {
            d = od;
            i = oi;
        }
    }
}

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
    cluster_warp_min(bd, bj);
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
        cluster_warp_min(bd, bi);
        if (lane == 0) {
            sh.wd[warp] = bd;
            sh.wi[warp] = bi;
        }
        __syncthreads();
        if (warp == 0) {
            bd = lane < n_warps ? sh.wd[lane] : INFINITY;
            bi = lane < n_warps ? sh.wi[lane] : n;
            cluster_warp_min(bd, bi);
            if (lane == 0) {
                sh.go = bd < INFINITY && bd <= a.threshold;
                sh.a = bi;
                sh.b = sh.go ? st.nn[bi] : 0u;
                sh.n_list = 0;
            }
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
                    if (cluster_key_less(d, ca, st.nnd[i], j)) {
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

size_t cluster_small_smem(unsigned n_cap) { return (size_t)n_cap * n_cap * 8 + cluster_state_bytes(n_cap); }

template <typename Kernel>
static int cluster_launch(Kernel k, const ClusterArgs& a, int block, size_t smem, int max_grid, void* stream) {
    if (a.n_segs == 0) return 0;
    cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return (int)err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, block, smem);
    if (err != cudaSuccess) return (int)err;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long grid = (long long)(per_sm > 0 ? per_sm : 1) * sms;
    if (grid > (long long)a.n_segs) grid = a.n_segs;
    if (max_grid > 0 && grid > max_grid) grid = max_grid;
    k<<<(unsigned)grid, block, smem, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
}

int launch_cluster(int kind, const ClusterLaunch& c, void* stream) {
    ClusterArgs a;
    a.robot = c.robot;
    a.results = c.results;
    a.rec_stride = c.rec_stride;
    a.cfg_stride = c.cfg_stride;
    a.complete = c.complete;
    a.separate_contact = c.separate_contact;
    a.threshold = c.threshold;
    a.order = c.order;
    a.offsets = c.offsets;
    a.labels = c.labels;
    a.counts = c.counts;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    ClusterArgs sm = a, lg = a;
    sm.segs = c.small_segs;
    sm.n_segs = c.n_small;
    sm.n_cap = c.small_cap;
    sm.work = nullptr;
    lg.segs = c.large_segs;
    lg.n_segs = c.n_large;
    lg.n_cap = c.large_cap;
    lg.work = c.work;
    const size_t small_smem = cluster_small_smem(c.small_cap), large_smem = cluster_state_bytes(c.large_cap);
    switch (kind) {
        case FKS_ROBOT_SE2:
            if ((rc = cluster_launch(cluster_small_kernel<FKS_ROBOT_SE2>, sm, kClusterSmallBlock, small_smem, 0, stream)) != 0) return rc;
            if ((rc = cluster_launch(cluster_large_kernel<FKS_ROBOT_SE2>, lg, kClusterLargeBlock, large_smem, c.large_slots, stream)) != 0) return rc;
            break;
        case FKS_ROBOT_SE3:
            if ((rc = cluster_launch(cluster_small_kernel<FKS_ROBOT_SE3>, sm, kClusterSmallBlock, small_smem, 0, stream)) != 0) return rc;
            if ((rc = cluster_launch(cluster_large_kernel<FKS_ROBOT_SE3>, lg, kClusterLargeBlock, large_smem, c.large_slots, stream)) != 0) return rc;
            break;
        case FKS_ROBOT_LINKED:
            if ((rc = cluster_launch(cluster_small_kernel<FKS_ROBOT_LINKED>, sm, kClusterSmallBlock, small_smem, 0, stream)) != 0) return rc;
            if ((rc = cluster_launch(cluster_large_kernel<FKS_ROBOT_LINKED>, lg, kClusterLargeBlock, large_smem, c.large_slots, stream)) != 0) return rc;
            break;
        default: return (int)cudaErrorInvalidValue;
    }
    // base of every segment's ids: partition's exclusive scan, in place over the counts (totals[1] = all clusters)
    partition_scan_kernel<<<1, kPartitionBlock, 0, st>>>(c.counts, c.n_segments, 0, c.totals);
    const unsigned relabel_grid = c.n_segments < 65535u ? c.n_segments : 65535u;
    cluster_relabel_kernel<<<relabel_grid, 256, 0, st>>>(c.offsets, c.n_segments, c.counts, c.labels);
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// fks_end_states_groups: the clusters of a labelled position range as particle groups.  Members: a stable counting sort by
// label -- count, the partition's one-block scan, a scatter in arrival order, then each group sorted by position in shared
// memory, so the result does not depend on the order of the scatter's atomics.  Representative: the member with the smallest
// (r, position), r(p) = max over the other members q of d(min(p,q), max(p,q)), d = the pairwise kernel's entry (same
// inlined config_distance, same operands), NaN as +inf.  Every pair is evaluated in both rows, so a row's maximum is a plain
// warp reduction; max over non-NaN values and the (r, position) argmin are exact in any order, so every result is.
// ---------------------------------------------------------------------------------------------
constexpr int kGroupBlock = 256;
constexpr unsigned kGroupWarps = kGroupBlock / 32;
constexpr unsigned kGroupRowsPerTask = 32;  // rows of a large cluster per task of the row pass

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
        double d = config_distance<KIND>(*g.robot, j > i ? rec_i : rec_j, j > i ? rec_j : rec_i);
        if (isnan(d)) d = INFINITY;
        if (d > r) r = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(FKS_FULL, r, o);
        if (x > r) r = x;
    }
    return k == 1 ? 0.0 : r;
}

// the CTA's smallest (d, i) over its warps' (lane-uniform) candidates, in thread 0
__device__ __forceinline__ void group_block_min(double& d, unsigned& i, double* wd, unsigned* wi) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        wd[warp] = d;
        wi[warp] = i;
    }
    __syncthreads();
    if (warp == 0) {
        d = lane < kGroupWarps ? wd[lane] : INFINITY;
        i = lane < kGroupWarps ? wi[lane] : 0xffffffffu;
        cluster_warp_min(d, i);
    }
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
            if (cluster_key_less(r, i, bd, bi)) {
                bd = r;
                bi = i;
            }
        }
        group_block_min(bd, bi, wd, wi);
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
            if (cluster_key_less(r, i, bd, bi)) {
                bd = r;
                bi = i;
            }
        }
        cluster_warp_min(bd, bi);
        group_block_min(bd, bi, wd, wi);
        if (threadIdx.x == 0) {
            g.reps[c] = g.members[begin + bi];
            g.radius[c] = bd;
        }
        __syncthreads();
    }
}

template <typename Kernel>
static unsigned groups_resident_ctas(Kernel k) {
    int per_sm = 0, dev = 0, sms = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kGroupBlock, 0);
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (unsigned)((per_sm > 0 ? per_sm : 1) * (sms > 0 ? sms : 1));
}

template <int KIND>
static void groups_search(const GroupsLaunch& g, cudaStream_t st) {
    // the host does not know how many groups are large: the row and argmin passes run a full grid and read the list
    const unsigned resident = groups_resident_ctas(groups_sort_small_kernel<KIND>);
    const unsigned rows_grid = groups_resident_ctas(groups_large_rows_kernel<KIND>);
    groups_sort_small_kernel<KIND><<<g.n_clusters < resident ? g.n_clusters : resident, kGroupBlock, 0, st>>>(g);
    groups_large_rows_kernel<KIND><<<rows_grid, kGroupBlock, 0, st>>>(g);
    groups_large_argmin_kernel<<<rows_grid, kGroupBlock, 0, st>>>(g);
}

int launch_groups(int kind, const GroupsLaunch& g, void* stream) {
    if (g.m == 0 || g.n_clusters == 0) return (int)cudaErrorInvalidValue;
    void (*search)(const GroupsLaunch&, cudaStream_t);
    switch (kind) {
        case FKS_ROBOT_SE2: search = groups_search<FKS_ROBOT_SE2>; break;
        case FKS_ROBOT_SE3: search = groups_search<FKS_ROBOT_SE3>; break;
        case FKS_ROBOT_LINKED: search = groups_search<FKS_ROBOT_LINKED>; break;
        default: return (int)cudaErrorInvalidValue;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t blocks = ((size_t)g.m + kGroupBlock - 1) / kGroupBlock;
    const unsigned grid = blocks < 65535 ? (unsigned)blocks : 65535u;
    groups_count_kernel<<<grid, kGroupBlock, 0, st>>>(g.labels, g.m, g.n_clusters, g.offsets, g.state);
    partition_scan_kernel<<<1, kPartitionBlock, 0, st>>>(g.offsets, g.n_clusters, g.m, g.totals);
    groups_scatter_kernel<<<grid, kGroupBlock, 0, st>>>(g.labels, g.m, g.n_clusters, g.offsets, g.totals, g.cursor, g.members);
    search(g, st);
    return (int)cudaGetLastError();
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

int launch_gather_starts(const char* results, size_t rec_stride, int cfg_stride, const unsigned* offsets, const unsigned* members,
                         const unsigned* selected, unsigned n_selected, unsigned per_group, const double* group_targets, double* starts,
                         double* targets, void* stream) {
    const size_t n_values = (size_t)n_selected * per_group * (size_t)cfg_stride;
    const size_t grid = (n_values + 255) / 256 < 65535 ? (n_values + 255) / 256 : 65535;
    gather_starts_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(results, rec_stride, cfg_stride, offsets, members, selected, per_group,
                                                                            n_values, group_targets, starts, targets);
    return (int)cudaGetLastError();
}

#ifdef FKS_PHASE_TIMERS
__global__ void dbg_copy_kernel(unsigned long long* out) {
    if (threadIdx.x < 64) {
        out[threadIdx.x] = g_dbg[threadIdx.x];
        g_dbg[threadIdx.x] = 0ull;
    }
}
#endif
int launch_dbg_copy(unsigned long long* out, void* stream) {
#ifdef FKS_PHASE_TIMERS
    dbg_copy_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(out);
#else
    (void)out;
    (void)stream;
#endif
    return (int)cudaGetLastError();
}
int launch_fp64_peak(double* out, int grid, int iters, void* stream) {
    fp64_peak_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, iters);
    return (int)cudaGetLastError();
}
int launch_gather(const float* data, unsigned long long n_mask, float* out, int grid, int iters, void* stream) {
    gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(data, n_mask, out, iters);
    return (int)cudaGetLastError();
}

}  // namespace fksdev
