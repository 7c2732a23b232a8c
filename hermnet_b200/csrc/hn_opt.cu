// Structure relaxation of the device loop: FIRE (Bitzek et al., PRL 97, 170201 (2006)) with ASE's rules and defaults,
// per replica, over the generalized coordinates of ASE's UnitCellFilter (atom rows r' = x A^-1 and, when the cell is
// relaxed, three cell rows c_f A^T with A = h0^-1 h).  Three launches around each force evaluation:
//   reduce  per atom:    F'_i = f_i A^T and the per-replica sums F'.v, |F'|^2, |v|^2, max |F'_i|^2 (fixed order, float64)
//   step    per replica: the cell rows, the convergence test and FIRE's mixing / dt / alpha logic in float64, with the
//                        max_step cap in closed form from the three sums (no second pass over the atoms)
//   update  per atom:    v = c_v v + c_f F',  r' += s dt v,  x = r' A
#include "hn_common.cuh"
#include "hn_reduce.cuh"

namespace {

constexpr int OPT_N_MIN = 5;
constexpr double OPT_F_INC = 1.1, OPT_F_DEC = 0.5, OPT_ALPHA_START = 0.1, OPT_F_ALPHA = 0.99;

// (F'.v, |F'|^2, |v|^2, max |F'_i|^2); 32-byte aligned: one vector access per workspace slot
struct alignas(32) Sums {
    double fv, ff, vv, fm;
    __device__ __forceinline__ void merge(const Sums &o) { fv += o.fv, ff += o.ff, vv += o.vv, fm = fmax(fm, o.fm); }
    __device__ __forceinline__ Sums shfl_xor(int o) const {
        return {__shfl_xor_sync(0xffffffffu, fv, o), __shfl_xor_sync(0xffffffffu, ff, o), __shfl_xor_sync(0xffffffffu, vv, o),
                __shfl_xor_sync(0xffffffffu, fm, o)};
    }
};

// F' = f A^T (row vector): F'_j = sum_k f_k A[j][k];  A == nullptr: F' = f
__device__ __forceinline__ void gen_force(const float *__restrict__ f, const double *__restrict__ A, double out[3]) {
    const double f0 = f[0], f1 = f[1], f2 = f[2];
    if (A == nullptr) {
        out[0] = f0, out[1] = f1, out[2] = f2;
        return;
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) out[j] = f0 * A[3 * j] + f1 * A[3 * j + 1] + f2 * A[3 * j + 2];
}

__global__ void opt_fire_reduce_pieces_kernel(const float *__restrict__ force, const float *__restrict__ vel,
                                              const double *__restrict__ A, const int *__restrict__ replica,
                                              const int *__restrict__ replica_ptr, int n_atoms, int n_chunks,
                                              Sums *__restrict__ part) {
    hn::reduce_pieces<Sums>(replica, replica_ptr, n_atoms, n_chunks, part, [&](int g) {
        double Ag[9];
        if (A != nullptr) {
#pragma unroll
            for (int k = 0; k < 9; ++k) Ag[k] = __ldg(A + 9 * (size_t)g + k);
        }
        return [=](Sums &acc, int i) {
            double F[3];
            gen_force(force + 3 * (size_t)i, A != nullptr ? Ag : nullptr, F);
            const double v0 = vel[3 * (size_t)i], v1 = vel[3 * (size_t)i + 1], v2 = vel[3 * (size_t)i + 2];
            const double f2 = F[0] * F[0] + F[1] * F[1] + F[2] * F[2];
            acc.fv += F[0] * v0 + F[1] * v1 + F[2] * v2;
            acc.ff += f2;
            acc.vv += v0 * v0 + v1 * v1 + v2 * v2;
            acc.fm = fmax(acc.fm, f2);
        };
    });
}

// out[g] = (F'.v, |F'|^2, |v|^2, max |F'_i|^2)
__global__ void opt_fire_reduce_final_kernel(const Sums *__restrict__ part, const int *__restrict__ replica_ptr,
                                             int n_replicas, int per, double *__restrict__ out) {
    int g;
    Sums acc;
    if (!hn::reduce_slots(part, replica_ptr, n_replicas, per, g, acc)) return;
    double *o = out + 4 * (size_t)g;
    o[0] = acc.fv, o[1] = acc.ff, o[2] = acc.vv, o[3] = acc.fm;
}

__global__ void opt_fire_step_kernel(const double *__restrict__ sums, const float *__restrict__ virial, float *__restrict__ cell,
                                     const double *__restrict__ h0, double *__restrict__ A, double *__restrict__ A_prev,
                                     double *__restrict__ vcell, const double *__restrict__ P0, const double *__restrict__ cf,
                                     double *__restrict__ dt, double *__restrict__ alpha, int *__restrict__ n_pos,
                                     int *__restrict__ steps, int *__restrict__ converged, double fmax2, double dt_max,
                                     double max_step, int move, int n_replicas, double *__restrict__ coef,
                                     double *__restrict__ fmax_out, int *__restrict__ n_active) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_replicas) return;
    double fv = sums[4 * (size_t)g], ff = sums[4 * (size_t)g + 1], vv = sums[4 * (size_t)g + 2], fm = sums[4 * (size_t)g + 3];
    const bool cell_rows = A != nullptr;
    double Ag[9], Fc[9], Vc[9];
    if (cell_rows) {
#pragma unroll
        for (int k = 0; k < 9; ++k) Ag[k] = A[9 * (size_t)g + k], Vc[k] = vcell[9 * (size_t)g + k];
        double h[9], W[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) h[k] = (double)cell[9 * (size_t)g + k], W[k] = (double)__ldg(virial + 9 * (size_t)g + k);
        const double V = fabs(h[0] * (h[4] * h[8] - h[5] * h[7]) - h[1] * (h[3] * h[8] - h[5] * h[6]) +
                              h[2] * (h[3] * h[7] - h[4] * h[6]));
        // A^-1 by cofactors
        const double c00 = Ag[4] * Ag[8] - Ag[5] * Ag[7], c01 = Ag[5] * Ag[6] - Ag[3] * Ag[8], c02 = Ag[3] * Ag[7] - Ag[4] * Ag[6];
        const double idet = 1.0 / (Ag[0] * c00 + Ag[1] * c01 + Ag[2] * c02);
        const double Ai[9] = {c00 * idet, (Ag[2] * Ag[7] - Ag[1] * Ag[8]) * idet, (Ag[1] * Ag[5] - Ag[2] * Ag[4]) * idet,
                              c01 * idet, (Ag[0] * Ag[8] - Ag[2] * Ag[6]) * idet, (Ag[2] * Ag[3] - Ag[0] * Ag[5]) * idet,
                              c02 * idet, (Ag[1] * Ag[6] - Ag[0] * Ag[7]) * idet, (Ag[0] * Ag[4] - Ag[1] * Ag[3]) * idet};
        const double pv = __ldg(P0 + g) * V, icf = 1.0 / __ldg(cf + g);
        double S[9];                          // W_sym - P0 V I
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k) S[3 * j + k] = 0.5 * (W[3 * j + k] + W[3 * k + j]) - (j == k ? pv : 0.0);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            double row = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                Fc[3 * j + k] = (S[3 * j] * Ai[k] + S[3 * j + 1] * Ai[3 + k] + S[3 * j + 2] * Ai[6 + k]) * icf;
                row += Fc[3 * j + k] * Fc[3 * j + k];
                fv += Fc[3 * j + k] * Vc[3 * j + k];
                vv += Vc[3 * j + k] * Vc[3 * j + k];
            }
            ff += row;
            fm = fmax(fm, row);
        }
    }
    fmax_out[g] = sqrt(fm);
    if (converged[g]) return;
    if (fm < fmax2) {                          // sticky: the replica never moves again
        converged[g] = 1;
        return;
    }
    atomicAdd(n_active, 1);
    if (!move) return;

    double a = alpha[g], t = dt[g], cv, cm;
    int np = n_pos[g];
    if (steps[g] == 0) {                       // ASE's first step (v is None): no mixing, v = 0
        cv = 0.0, cm = 0.0;
    } else if (fv > 0.0) {
        cv = 1.0 - a, cm = a * sqrt(vv) / sqrt(ff);
        if (np > OPT_N_MIN) {
            t = fmin(t * OPT_F_INC, dt_max);
            a *= OPT_F_ALPHA;
        }
        np += 1;
    } else {
        cv = 0.0, cm = 0.0, a = OPT_ALPHA_START, t *= OPT_F_DEC, np = 0;
    }
    // v_new = cv v + cfp F: |v_new|^2 from the sums (every term >= 0 in each branch), so the cap needs no atom pass
    const double cfp = cm + t;
    const double dr = t * sqrt(cv * cv * vv + 2.0 * cv * cfp * fv + cfp * cfp * ff);
    const double s = dr > max_step ? max_step / dr : 1.0;
    coef[3 * (size_t)g] = cv, coef[3 * (size_t)g + 1] = cfp, coef[3 * (size_t)g + 2] = s * t;
    alpha[g] = a, dt[g] = t, n_pos[g] = np, steps[g] += 1;
    if (cell_rows) {
        const double c = __ldg(cf + g);
        double An[9];
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double v = cv * Vc[3 * j + k] + cfp * Fc[3 * j + k];
                vcell[9 * (size_t)g + 3 * j + k] = v;
                An[3 * k + j] = (c * Ag[3 * k + j] + s * t * v) / c;     // q_c = c_f A^T + dr,  A = (q_c / c_f)^T
            }
#pragma unroll
        for (int k = 0; k < 9; ++k) A_prev[9 * (size_t)g + k] = Ag[k], A[9 * (size_t)g + k] = An[k];
        const double *H0 = h0 + 9 * (size_t)g;
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k)
                cell[9 * (size_t)g + 3 * j + k] = (float)(H0[3 * j] * An[k] + H0[3 * j + 1] * An[3 + k] + H0[3 * j + 2] * An[6 + k]);
    }
}

__global__ void opt_fire_update_kernel(float *__restrict__ x, float *__restrict__ rp, float *__restrict__ vel,
                                       const float *__restrict__ force, const double *__restrict__ A_prev,
                                       const double *__restrict__ A, const int *__restrict__ replica,
                                       const int *__restrict__ converged, const double *__restrict__ coef, int n_atoms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int g = __ldg(replica + i);
    if (__ldg(converged + g)) return;
    const double cv = __ldg(coef + 3 * (size_t)g), cfp = __ldg(coef + 3 * (size_t)g + 1), sdt = __ldg(coef + 3 * (size_t)g + 2);
    const size_t b = 3 * (size_t)i;
    double F[3], r[3];
    if (A == nullptr) {
        gen_force(force + b, nullptr, F);
    } else {
        double Ap[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) Ap[k] = __ldg(A_prev + 9 * (size_t)g + k);
        gen_force(force + b, Ap, F);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double v = cv * (double)vel[b + k] + cfp * F[k];
        vel[b + k] = (float)v;
        const float q = (float)((double)rp[b + k] + sdt * v);
        rp[b + k] = q;
        r[k] = q;
    }
    if (A == nullptr) return;                  // positions only: x is r' (bitwise)
    const double *Ag = A + 9 * (size_t)g;
#pragma unroll
    for (int k = 0; k < 3; ++k) x[b + k] = (float)(r[0] * __ldg(Ag + k) + r[1] * __ldg(Ag + 3 + k) + r[2] * __ldg(Ag + 6 + k));
}

}  // namespace

extern "C" int64_t hn_opt_fire_reduce_workspace_bytes(int64_t n_atoms, int32_t n_replicas) {
    if (n_atoms <= 0 || n_replicas <= 0) return 0;
    return (hn::reduce_chunks(n_atoms) + n_replicas) * (int64_t)sizeof(Sums);
}

extern "C" int hn_opt_fire_reduce(const float *force, const float *vel, const double *A, const int32_t *replica,
                                  const int32_t *replica_ptr, int32_t n_replicas, int64_t n_atoms, double *sums,
                                  void *workspace, int64_t workspace_bytes, void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_opt_fire_reduce", "n_atoms must be in [0, 2^31)");
    HN_REQUIRE(n_replicas >= 0, "hn_opt_fire_reduce", "n_replicas must be >= 0");
    if (n_replicas == 0 || n_atoms == 0) return 0;
    HN_REQUIRE(force && vel && replica && replica_ptr && sums, "hn_opt_fire_reduce", "null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    HN_REQUIRE(workspace && workspace_bytes >= hn_opt_fire_reduce_workspace_bytes(n_atoms, n_replicas), "hn_opt_fire_reduce",
               "workspace smaller than hn_opt_fire_reduce_workspace_bytes");
    const int64_t chunks = hn::reduce_chunks(n_atoms);
    Sums *part = (Sums *)workspace;
    opt_fire_reduce_pieces_kernel<<<(unsigned)((chunks * 32 + 255) / 256), 256, 0, s>>>(force, vel, A, replica, replica_ptr,
                                                                                         (int)n_atoms, (int)chunks, part);
    HN_CUDA(cudaGetLastError(), "hn_opt_fire_reduce");
    const int per = hn::reduce_slot_threads(chunks, n_replicas);
    opt_fire_reduce_final_kernel<<<(unsigned)(((int64_t)n_replicas * per + 255) / 256), 256, 0, s>>>(part, replica_ptr, n_replicas,
                                                                                                    per, sums);
    return hn::check_launch("hn_opt_fire_reduce");
}

extern "C" int hn_opt_fire_step(const double *sums, const float *virial, float *cell, const double *h0, double *A,
                                double *A_prev, double *vcell, const double *P0, const double *cell_factor, double *dt,
                                double *alpha, int32_t *n_pos, int32_t *steps, int32_t *converged, int32_t n_replicas,
                                double fmax, double dt_max, double max_step, int32_t move, double *coef, double *fmax_out,
                                int32_t *n_active, void *stream) {
    HN_REQUIRE(n_replicas >= 0, "hn_opt_fire_step", "n_replicas must be >= 0");
    HN_REQUIRE(fmax > 0.0 && dt_max > 0.0 && max_step > 0.0, "hn_opt_fire_step", "fmax, dt_max and max_step must be > 0");
    if (n_replicas == 0) return 0;
    HN_REQUIRE(sums && dt && alpha && n_pos && steps && converged && coef && fmax_out && n_active, "hn_opt_fire_step",
               "null pointer");
    HN_REQUIRE(A == nullptr || (virial && cell && h0 && A_prev && vcell && P0 && cell_factor), "hn_opt_fire_step",
               "null pointer among the cell-row arguments");
    cudaStream_t s = (cudaStream_t)stream;
    HN_CUDA(cudaMemsetAsync(n_active, 0, sizeof(int32_t), s), "hn_opt_fire_step");
    opt_fire_step_kernel<<<(unsigned)((n_replicas + 127) / 128), 128, 0, s>>>(
        sums, virial, cell, h0, A, A_prev, vcell, P0, cell_factor, dt, alpha, n_pos, steps, converged, fmax * fmax, dt_max,
        max_step, move != 0, (int)n_replicas, coef, fmax_out, n_active);
    return hn::check_launch("hn_opt_fire_step");
}

extern "C" int hn_opt_fire_update(float *x, float *rp, float *vel, const float *force, const double *A_prev, const double *A,
                                  const int32_t *replica, const int32_t *converged, const double *coef, int64_t n_atoms,
                                  void *stream) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), "hn_opt_fire_update", "n_atoms must be in [0, 2^31)");
    if (n_atoms == 0) return 0;
    HN_REQUIRE(rp && vel && force && replica && converged && coef, "hn_opt_fire_update", "null pointer");
    HN_REQUIRE(A == nullptr || (x && A_prev), "hn_opt_fire_update", "x and A_prev are required with A");
    opt_fire_update_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        x, rp, vel, force, A_prev, A, replica, converged, coef, (int)n_atoms);
    return hn::check_launch("hn_opt_fire_update");
}
