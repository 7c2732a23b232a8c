// Langevin (NVT) integration of the device MD loop: BAOAB (Leimkuhler-Matthews) as two fused element-wise passes around
// the force evaluation -- B-A-O-A before it, the closing B (plus per-atom kinetic energies) after it.
//
// Noise is a pure function of (replica seed, replica-local atom index, step): Philox4x32-10 from the header-only
// <curand_philox4x32_x.h> (no libcurand link) keyed on the seed, with the step counter read from device memory.  A
// captured replay therefore draws fresh noise without any host argument changing, a restart at step k reproduces the
// trajectory, and a replica's noise does not depend on which other replicas share its batch.
#include <curand_philox4x32_x.h>

#include "hn_common.cuh"

namespace {

// exact fp32 uniform in [2^-24, 1 - 2^-24]: an odd 24-bit integer times 2^-24
__device__ __forceinline__ float md_uniform(unsigned int r) { return (float)((r >> 9) * 2u + 1u) * 0x1p-24f; }

__global__ void md_langevin_baoa_kernel(float *__restrict__ pos, float *__restrict__ vel, const float *__restrict__ force,
                                        const float *__restrict__ inv_mass, const int *__restrict__ replica,
                                        const int *__restrict__ replica_ptr, const float *__restrict__ kT,
                                        const unsigned long long *__restrict__ seed, const unsigned long long *__restrict__ step,
                                        float c1, float c2, float half_dt, int n_atoms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int g = __ldg(replica + i);
    const unsigned int j = (unsigned int)(i - __ldg(replica_ptr + g));
    const unsigned long long s = __ldg(seed + g), n = __ldg(step);
    const uint4 r = curand_Philox4x32_10(make_uint4(j, (unsigned int)n, (unsigned int)(n >> 32), 0u),
                                         make_uint2((unsigned int)s, (unsigned int)(s >> 32)));
    const float u0 = md_uniform(r.x), u1 = md_uniform(r.y), u2 = md_uniform(r.z), u3 = md_uniform(r.w);
    const float rad01 = sqrtf(-2.0f * logf(u0)), rad23 = sqrtf(-2.0f * logf(u2));
    float s1, co1, s3, co3;
    sincospif(2.0f * u1, &s1, &co1);
    sincospif(2.0f * u3, &s3, &co3);
    const float xi[3] = {rad01 * co1, rad01 * s1, rad23 * co3};

    const float im = __ldg(inv_mass + i);
    const float sigma = c2 * sqrtf(__ldg(kT + g) * im);
    const size_t b = 3 * (size_t)i;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = vel[b + k], x = pos[b + k];
        v += half_dt * __ldg(force + b + k) * im;     // B
        x += half_dt * v;                              // A
        v = c1 * v + sigma * xi[k];                    // O
        x += half_dt * v;                              // A
        vel[b + k] = v;
        pos[b + k] = x;
    }
}

__global__ void md_kick_kernel(float *__restrict__ vel, const float *__restrict__ force, const float *__restrict__ inv_mass,
                               float half_dt, int n_atoms, float *__restrict__ kinetic, unsigned long long *__restrict__ step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *step += 1ull;      // read by the next step's B-A-O-A, which is stream-ordered after this kernel
    if (i >= n_atoms) return;
    const float im = __ldg(inv_mass + i);
    const size_t b = 3 * (size_t)i;
    float v2 = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float v = vel[b + k] + half_dt * __ldg(force + b + k) * im;
        vel[b + k] = v;
        v2 += v * v;
    }
    if (kinetic != nullptr) kinetic[i] = 0.5f * v2 / im;
}

}  // namespace

extern "C" int hn_md_langevin_baoa(float *pos, float *vel, const float *force, const float *inv_mass, const int32_t *replica,
                                   const int32_t *replica_ptr, int32_t n_replicas, const float *kT, const int64_t *seed,
                                   const int64_t *step, float c1, float c2, float dt, int64_t n_atoms, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_md_langevin_baoa", "n_atoms must be in [0, 2^31)");
    HN_REQUIRE(n_replicas >= 1, "hn_md_langevin_baoa", "n_replicas must be >= 1");
    HN_REQUIRE(dt > 0.f, "hn_md_langevin_baoa", "dt must be > 0");
    HN_REQUIRE(c1 >= 0.f && c1 <= 1.f, "hn_md_langevin_baoa", "c1 must be in [0, 1]");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(pos && vel && force && inv_mass && replica && replica_ptr && kT && seed && step, "hn_md_langevin_baoa",
               "null pointer");
    md_langevin_baoa_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        pos, vel, force, inv_mass, replica, replica_ptr, kT, (const unsigned long long *)seed, (const unsigned long long *)step,
        c1, c2, 0.5f * dt, (int)n_atoms);
    return hn::check_launch("hn_md_langevin_baoa");
}

extern "C" int hn_md_kick(float *vel, const float *force, const float *inv_mass, float half_dt, int64_t n_atoms, float *kinetic,
                          int64_t *step, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_md_kick", "n_atoms must be in [0, 2^31)");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(vel && force && inv_mass && step, "hn_md_kick", "null pointer");
    md_kick_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        vel, force, inv_mass, half_dt, (int)n_atoms, kinetic, (unsigned long long *)step);
    return hn::check_launch("hn_md_kick");
}

// ---------------------------------------------------------------------------------------------------------------------
// Constant pressure: isotropic stochastic cell rescaling (Bernetti & Bussi, JCP 153, 114107 (2020)) after the closing
// kick.  One thread per replica computes the strain increment in float64 and scales its cell; a per-atom pass then
// applies the same factor to positions (x mu) and velocities (/ mu).  The barostat noise is Philox keyed on the replica
// seed like the Langevin noise, with counter word 3 = 1 so the two streams never share a draw.
// ---------------------------------------------------------------------------------------------------------------------
namespace {

__global__ void md_scr_barostat_kernel(float *__restrict__ cell, const float *__restrict__ kinetic,
                                       const float *__restrict__ virial, const float *__restrict__ P0,
                                       const float *__restrict__ kT, const float *__restrict__ beta,
                                       const unsigned long long *__restrict__ seed, const unsigned long long *__restrict__ step,
                                       double dt_over_tau, int n_replicas, float *__restrict__ mu, float *__restrict__ pressure) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_replicas) return;
    float *c = cell + 9 * (size_t)g;
    double h[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) h[k] = (double)c[k];
    const double V = fabs(h[0] * (h[4] * h[8] - h[5] * h[7]) - h[1] * (h[3] * h[8] - h[5] * h[6]) +
                          h[2] * (h[3] * h[7] - h[4] * h[6]));
    const float *w = virial + 9 * (size_t)g;
    const double P = (2.0 * (double)__ldg(kinetic + g) + (double)__ldg(w) + (double)__ldg(w + 4) + (double)__ldg(w + 8)) / (3.0 * V);

    const unsigned long long s = __ldg(seed + g), n = __ldg(step);
    const uint4 r = curand_Philox4x32_10(make_uint4(0u, (unsigned int)n, (unsigned int)(n >> 32), 1u),
                                         make_uint2((unsigned int)s, (unsigned int)(s >> 32)));
    const double xi = sqrt(-2.0 * log((double)md_uniform(r.x))) * cospi(2.0 * (double)md_uniform(r.y));

    const double b = (double)__ldg(beta + g) * dt_over_tau;                    // beta_T dt / tau_p
    const double de = -b * ((double)__ldg(P0 + g) - P) + sqrt(2.0 * (double)__ldg(kT + g) * b / V) * xi;
    const float m = (float)exp(de / 3.0);
#pragma unroll
    for (int k = 0; k < 9; ++k) c[k] = m * c[k];
    mu[g] = m;
    pressure[g] = (float)P;
}

__global__ void md_affine_scale_kernel(float *__restrict__ pos, float *__restrict__ vel, const int *__restrict__ replica,
                                       const float *__restrict__ mu, int n_atoms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const float m = __ldg(mu + __ldg(replica + i));
    const size_t b = 3 * (size_t)i;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        pos[b + k] = m * pos[b + k];
        vel[b + k] = vel[b + k] / m;
    }
}

}  // namespace

extern "C" int hn_md_scr_barostat(float *cell, const float *kinetic, const float *virial, const float *P0, const float *kT,
                                  const float *beta, const int64_t *seed, const int64_t *step, int32_t n_replicas, float dt,
                                  float tau_p, float *mu, float *pressure, void *stream) {
    HN_REQUIRE(n_replicas >= 0, "hn_md_scr_barostat", "n_replicas must be >= 0");
    HN_REQUIRE(dt > 0.f, "hn_md_scr_barostat", "dt must be > 0");
    HN_REQUIRE(tau_p > 0.f, "hn_md_scr_barostat", "tau_p must be > 0");
    if (n_replicas == 0) return 0;
    HN_REQUIRE(cell && kinetic && virial && P0 && kT && beta && seed && step && mu && pressure, "hn_md_scr_barostat",
               "null pointer");
    md_scr_barostat_kernel<<<(unsigned)((n_replicas + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        cell, kinetic, virial, P0, kT, beta, (const unsigned long long *)seed, (const unsigned long long *)step,
        (double)dt / (double)tau_p, (int)n_replicas, mu, pressure);
    return hn::check_launch("hn_md_scr_barostat");
}

extern "C" int hn_md_affine_scale(float *pos, float *vel, const int32_t *replica, const float *mu, int64_t n_atoms, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_md_affine_scale", "n_atoms must be in [0, 2^31)");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(pos && vel && replica && mu, "hn_md_affine_scale", "null pointer");
    md_affine_scale_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pos, vel, replica, mu,
                                                                                              (int)n_atoms);
    return hn::check_launch("hn_md_affine_scale");
}
