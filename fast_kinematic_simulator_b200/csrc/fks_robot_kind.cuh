// Code that depends on the robot kind (FKS_ROBOT_SE2 / SE3 / LINKED) and is shared by the translation units: the
// configuration distance, which the simulate kernel's shortcut test and every batch consumer (fks_consumers.cu) compute
// from this one definition, and the host dispatch from a run-time kind to a kernel instance.
#ifndef FKS_ROBOT_KIND_CUH
#define FKS_ROBOT_KIND_CUH

#include <cuda_runtime.h>
#include <math.h>

#include <type_traits>

#include "fks_device_types.h"

namespace fksdev {

#define FKS_FULL 0xffffffffu

constexpr double kPi = 3.14159265358979323846;

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

// f(std::integral_constant<int, KIND>{}) for the robot's kind, whose result it returns; cudaErrorInvalidValue for any other
// kind.  A launcher's generic lambda names the kernel instance as kernel<decltype(K)::value>.
template <typename F>
int for_kind(int kind, F&& f) {
    switch (kind) {
        case FKS_ROBOT_SE2: return f(std::integral_constant<int, FKS_ROBOT_SE2>{});
        case FKS_ROBOT_SE3: return f(std::integral_constant<int, FKS_ROBOT_SE3>{});
        case FKS_ROBOT_LINKED: return f(std::integral_constant<int, FKS_ROBOT_LINKED>{});
        default: return (int)cudaErrorInvalidValue;
    }
}

}  // namespace fksdev

#endif
