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

// ---------------------------------------------------------------------------------------------------------------------
// Constant pressure with the cell shape free: triclinic stochastic cell rescaling of a lower-triangular cell (a along x,
// b in the xy plane, positive diagonal).  Per replica the strain increment delta is lower-triangular, mu = expm(delta),
// and h <- h mu, x <- x mu, v <- v mu^-T hold the scaled coordinates s = x h^-1 and momenta pi = p h^T fixed.  The drift
// carries (b kT / 3V) diag(2, 0, -2): the noise-induced drift of dh = h dXi, the gradient of the measure 1/(h11 h22^2) of
// triangular cells and the E[delta^2]/2 of the exponential step together (DESIGN.md, "Triclinic constant pressure").
// The noise is Philox keyed on the replica seed with counter word 3 = 2, disjoint from the Langevin (0) and isotropic (1)
// streams.
// ---------------------------------------------------------------------------------------------------------------------
namespace {

// divided difference exp[a, b] = (e^a - e^b) / (a - b), exact limit e^b at a == b (expm1 keeps it accurate when close)
__device__ __forceinline__ double exp_dd1(double a, double b) {
    const double x = a - b;
    return x == 0.0 ? exp(b) : exp(b) * (expm1(x) / x);
}

// second divided difference exp[a, b, c] (symmetric in its arguments).  Spread above 1e-3: the recursion over the widest
// pair (relative error ~ 1e-16 / spread); below: the series e^m sum_k h_k(a-m, b-m, c-m) / (k+2)! about the mean m,
// where h_k is the complete homogeneous symmetric polynomial (terms past k = 5 are below 1e-17)
__device__ __forceinline__ double exp_dd2(double a, double b, double c) {
    // order so that (a, c) is the widest pair
    if (fabs(a - b) > fabs(a - c) && fabs(a - b) >= fabs(b - c)) { const double t = b; b = c; c = t; }
    else if (fabs(b - c) > fabs(a - c)) { const double t = b; b = a; a = t; }
    if (fabs(a - c) > 1e-3) return (exp_dd1(a, b) - exp_dd1(b, c)) / (a - c);
    const double m = (a + b + c) / 3.0, u[3] = {a - m, b - m, c - m};
    double h[6] = {1.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int v = 0; v < 3; ++v)
#pragma unroll
        for (int k = 1; k < 6; ++k) h[k] += u[v] * h[k - 1];
    const double inv_fact[6] = {1.0 / 2, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040};
    double s = 0.0;
#pragma unroll
    for (int k = 5; k >= 0; --k) s += h[k] * inv_fact[k];
    return exp(m) * s;
}

// expm of the lower-triangular d = (00, 10, 11, 20, 21, 22) into e (same packing), Parlett's closed form
__device__ __forceinline__ void expm_lower3(const double d[6], double e[6]) {
    e[0] = exp(d[0]);
    e[2] = exp(d[2]);
    e[5] = exp(d[5]);
    e[1] = d[1] * exp_dd1(d[2], d[0]);
    e[4] = d[4] * exp_dd1(d[5], d[2]);
    e[3] = d[3] * exp_dd1(d[5], d[0]) + d[4] * d[1] * exp_dd2(d[5], d[2], d[0]);
}

__global__ void md_kinetic_tensor_kernel(const float *__restrict__ vel, const float *__restrict__ inv_mass, int n_atoms,
                                         float *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const float im = __ldg(inv_mass + i);
    const float v0 = __ldg(vel + 3 * (size_t)i), v1 = __ldg(vel + 3 * (size_t)i + 1), v2 = __ldg(vel + 3 * (size_t)i + 2);
    float *o = out + 6 * (size_t)i;
    o[0] = v0 * v0 / im;
    o[1] = v1 * v0 / im;
    o[2] = v1 * v1 / im;
    o[3] = v2 * v0 / im;
    o[4] = v2 * v1 / im;
    o[5] = v2 * v2 / im;
}

__global__ void md_scr_barostat_tri_kernel(float *__restrict__ cell, const float *__restrict__ kin6,
                                           const float *__restrict__ virial, const float *__restrict__ P0,
                                           const float *__restrict__ kT, const float *__restrict__ beta,
                                           const unsigned long long *__restrict__ seed,
                                           const unsigned long long *__restrict__ step, double dt_over_tau, int n_replicas,
                                           float *__restrict__ mu, float *__restrict__ mu_inv_t, float *__restrict__ pressure) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_replicas) return;
    constexpr int I[6] = {0, 1, 1, 2, 2, 2}, J[6] = {0, 0, 1, 0, 1, 2};       // packed lower triangle (00, 10, 11, 20, 21, 22)
    float *c = cell + 9 * (size_t)g;
    double h[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) h[q] = (double)c[3 * I[q] + J[q]];
    const double V = h[0] * h[2] * h[5];
    const float *w = virial + 9 * (size_t)g;
    double P[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) P[q] = ((double)__ldg(kin6 + 6 * (size_t)g + q) + (double)__ldg(w + 3 * I[q] + J[q])) / V;

    const unsigned long long s = __ldg(seed + g), n = __ldg(step);
    double xi[8];
#pragma unroll
    for (unsigned int k = 0; k < 2; ++k) {
        const uint4 r = curand_Philox4x32_10(make_uint4(k, (unsigned int)n, (unsigned int)(n >> 32), 2u),
                                             make_uint2((unsigned int)s, (unsigned int)(s >> 32)));
        const double rad01 = sqrt(-2.0 * log((double)md_uniform(r.x))), rad23 = sqrt(-2.0 * log((double)md_uniform(r.z)));
        double s1, c1, s3, c3;
        sincospi(2.0 * (double)md_uniform(r.y), &s1, &c1);
        sincospi(2.0 * (double)md_uniform(r.w), &s3, &c3);
        xi[4 * k] = rad01 * c1;
        xi[4 * k + 1] = rad01 * s1;
        xi[4 * k + 2] = rad23 * c3;
        xi[4 * k + 3] = rad23 * s3;
    }

    const double b = (double)__ldg(beta + g) * dt_over_tau;                    // beta_T dt / tau_p
    const double p0 = (double)__ldg(P0 + g), bkT3V = b * (double)__ldg(kT + g) / (3.0 * V);
    const double sig = sqrt(2.0 * bkT3V);
    double d[6], e[6], ei[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) d[q] = (b / 3.0) * (I[q] == J[q] ? P[q] - p0 : P[q]) + sig * xi[q];
    d[0] += 2.0 * bkT3V;
    d[5] -= 2.0 * bkT3V;
    expm_lower3(d, e);
#pragma unroll
    for (int q = 0; q < 6; ++q) d[q] = -d[q];
    expm_lower3(d, ei);                                                          // mu^-1 = expm(-delta)

    // h mu (lower-triangular product); the upper triangle is written as exact zeros
    const double hm[6] = {h[0] * e[0], h[1] * e[0] + h[2] * e[1], h[2] * e[2], h[3] * e[0] + h[4] * e[1] + h[5] * e[3],
                          h[4] * e[2] + h[5] * e[4], h[5] * e[5]};
    float *m = mu + 9 * (size_t)g, *mi = mu_inv_t + 9 * (size_t)g, *p = pressure + 9 * (size_t)g;
#pragma unroll
    for (int k = 0; k < 9; ++k) { c[k] = 0.f; m[k] = 0.f; mi[k] = 0.f; }
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        c[3 * I[q] + J[q]] = (float)hm[q];
        m[3 * I[q] + J[q]] = (float)e[q];
        mi[3 * J[q] + I[q]] = (float)ei[q];                                      // transposed: upper-triangular
        p[3 * I[q] + J[q]] = p[3 * J[q] + I[q]] = (float)P[q];
    }
}

__global__ void md_affine_deform_kernel(float *__restrict__ pos, float *__restrict__ vel, const int *__restrict__ replica,
                                        const float *__restrict__ mu, const float *__restrict__ mu_inv_t, int n_atoms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const size_t gg = 9 * (size_t)__ldg(replica + i), b = 3 * (size_t)i;
    float m[9], mt[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) { m[k] = __ldg(mu + gg + k); mt[k] = __ldg(mu_inv_t + gg + k); }
    const float x[3] = {pos[b], pos[b + 1], pos[b + 2]}, v[3] = {vel[b], vel[b + 1], vel[b + 2]};
#pragma unroll
    for (int j = 0; j < 3; ++j) {                                                // row vectors: x_j = sum_k x_k mu_kj
        pos[b + j] = fmaf(x[2], m[6 + j], fmaf(x[1], m[3 + j], x[0] * m[j]));
        vel[b + j] = fmaf(v[2], mt[6 + j], fmaf(v[1], mt[3 + j], v[0] * mt[j]));
    }
}

}  // namespace

extern "C" int hn_md_kinetic_tensor(const float *vel, const float *inv_mass, int64_t n_atoms, float *out, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_md_kinetic_tensor", "n_atoms must be in [0, 2^31)");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(vel && inv_mass && out, "hn_md_kinetic_tensor", "null pointer");
    md_kinetic_tensor_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vel, inv_mass, (int)n_atoms,
                                                                                                   out);
    return hn::check_launch("hn_md_kinetic_tensor");
}

extern "C" int hn_md_scr_barostat_tri(float *cell, const float *kin6, const float *virial, const float *P0, const float *kT,
                                      const float *beta, const int64_t *seed, const int64_t *step, int32_t n_replicas, float dt,
                                      float tau_p, float *mu, float *mu_inv_t, float *pressure, void *stream) {
    HN_REQUIRE(n_replicas >= 0, "hn_md_scr_barostat_tri", "n_replicas must be >= 0");
    HN_REQUIRE(dt > 0.f, "hn_md_scr_barostat_tri", "dt must be > 0");
    HN_REQUIRE(tau_p > 0.f, "hn_md_scr_barostat_tri", "tau_p must be > 0");
    if (n_replicas == 0) return 0;
    HN_REQUIRE(cell && kin6 && virial && P0 && kT && beta && seed && step && mu && mu_inv_t && pressure,
               "hn_md_scr_barostat_tri", "null pointer");
    md_scr_barostat_tri_kernel<<<(unsigned)((n_replicas + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        cell, kin6, virial, P0, kT, beta, (const unsigned long long *)seed, (const unsigned long long *)step,
        (double)dt / (double)tau_p, (int)n_replicas, mu, mu_inv_t, pressure);
    return hn::check_launch("hn_md_scr_barostat_tri");
}

extern "C" int hn_md_affine_deform(float *pos, float *vel, const int32_t *replica, const float *mu, const float *mu_inv_t,
                                   int64_t n_atoms, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_md_affine_deform", "n_atoms must be in [0, 2^31)");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(pos && vel && replica && mu && mu_inv_t, "hn_md_affine_deform", "null pointer");
    md_affine_deform_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pos, vel, replica, mu,
                                                                                               mu_inv_t, (int)n_atoms);
    return hn::check_launch("hn_md_affine_deform");
}
