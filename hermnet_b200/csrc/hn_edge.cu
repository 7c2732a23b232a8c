// Fused PaiNN edge kernels (forward, destination-major backward, source-major backward).
//
// Replaces, per layer and sub-network, the reference chain
//   rbf_proj (rmnet.py:55) -> index_select gathers (PyG propagate, rmnet.py:58) -> message (rmnet.py:61-67)
//   -> scatter-add with atomics (rmnet.py:69-73)
// and the RBF x envelope edge embedding (rmnet.py:168-193), none of which is ever materialised here.
//
// Mapping: one warp per row (segment) and per channel slice of 32*VEC channels; lane l owns VEC consecutive
// channels of each of the three F-wide parts, so every gather of a source row is a fully coalesced
// 128*VEC-byte request per part and the segmented reduction is a private register accumulation --
// no atomics, deterministic order (row order of the CSR).
//
// Filter: phi = W.(env*gauss) + b.  With offset = linspace(0,1,K) the Gaussians have sigma = one grid
// step, so only a kBand(=12)-wide band around floor(u*(K-1)) is evaluated; every dropped term is
// < exp(-18) = 1.5e-8 of a unit term (below fp32 rounding of the sum).  Lane j (< kBand) evaluates basis
// function k0+j (one expf per lane per edge), broadcast by shuffle.  The graph builder sorts every row by
// distance (and every transposed row by (module, distance)), so consecutive edges of a warp hit mostly the
// same W rows in L1.
// These row kernels are the fallback for F % 32 == 0 outside {64, 128, 256, 512} and the A/B partner of the tile-sweep
// kernels of hn_edge_quad.cu, which share one band sweep between consecutive edges of a row and are the default
// (hn_edge_params.variant = 1 selects these).
// Verlet-skin superset lists (flags bit 0): the MASKED instantiations skip an entry whose geom[e].w < 0 (the caller stores
// -d for the entries that are not edges now) before its gathers and band; MASKED = false is the unmasked kernel unchanged.
#include <cstdlib>
#include <cstring>

#include "hn_common.cuh"
#include "hn_edge_quad.cuh"

namespace {

using hn::Vec;
using hn::ldv;
using hn::stv;

constexpr unsigned kFull = 0xffffffffu;
constexpr int kBand = 12;   // basis functions floor(x)-5 .. floor(x)+6, x = u*(K-1)

__device__ __forceinline__ float ipow(float u, int p) {
    float r = 1.f;
    for (int i = 0; i < p; ++i) r *= u;
    return r;
}

// Per-edge band: returns k0; lane j < nb gets val = env*g_{k0+j} and (DERIV) dval = d(val)/dd.
template <bool DERIV>
__device__ __forceinline__ int band_setup(float u, const hn_edge_params &P, const float *__restrict__ offset, int lane,
                                          int nb, float &val, float &dval) {
    const int K = P.num_rbf;
    const int kc = (int)floorf(u * (float)(K - 1));
    int k0 = kc - 5;
    k0 = k0 < 0 ? 0 : k0;
    k0 = k0 > K - nb ? K - nb : k0;
    const int p = P.env_p;
    const float a = -0.5f * (float)((p + 1) * (p + 2)), b = (float)(p * (p + 2)), c = -0.5f * (float)(p * (p + 1));
    const float um = ipow(u, p - 1), u0 = um * u, u1 = u0 * u, u2 = u1 * u;
    const float env = 1.f + a * u0 + b * u1 + c * u2;
    val = 0.f;
    dval = 0.f;
    if (lane < nb) {
        const float diff = u - __ldg(offset + k0 + lane);
        const float g = expf(P.coeff * diff * diff);
        val = env * g;
        if (DERIV) {
            const float denv = a * (float)p * um + b * (float)(p + 1) * u0 + c * (float)(p + 2) * u1;
            dval = (denv * g + val * (2.f * P.coeff * diff)) * P.inv_rc;
        }
    }
    return k0;
}

template <int VEC, bool MASKED>
__global__ void __launch_bounds__(256)
edge_fwd_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                const float4 *__restrict__ geom, const int *__restrict__ rowptr, const int *__restrict__ col,
                const int *__restrict__ row_mod, const long long *__restrict__ row_xoff, const float *__restrict__ Wt,
                const float *__restrict__ bias, const float *__restrict__ offset, float *__restrict__ dx,
                float *__restrict__ dvec) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= P.n_rows) return;
    const int F = P.hidden, K = P.num_rbf, F3 = 3 * F;
    const int ch = blockIdx.y * (32 * VEC) + lane * VEC;
    const int m = __ldg(row_mod + row);
    float ax[VEC], av[3][VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { ax[v] = 0.f; av[0][v] = 0.f; av[1][v] = 0.f; av[2][v] = 0.f; }
    if (m >= 0) {
        const int e0 = __ldg(rowptr + row), e1 = __ldg(rowptr + row + 1);
        const float *Wm = Wt + (size_t)m * K * F3 + ch;
        const float *xm = xh + __ldg(row_xoff + row) * F3 + ch;
        const Vec<VEC> ba = ldv<VEC>(bias + (size_t)m * F3 + ch), bb = ldv<VEC>(bias + (size_t)m * F3 + F + ch),
                       bc = ldv<VEC>(bias + (size_t)m * F3 + 2 * F + ch);
        const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
        const int nb = K < kBand ? K : kBand;
        Vec<VEC> vzero;
#pragma unroll
        for (int v = 0; v < VEC; ++v) vzero.v[v] = 0.f;
        for (int e = e0; e < e1; ++e) {
            const int s = __ldg(col + e);
            const float4 g = __ldg(geom + e);
            if (MASKED && g.w < 0.f) continue;     // dead entry of a Verlet-skin list: no gathers, no band
            const float *xs = xm + (size_t)s * F3;
            const Vec<VEC> Pa = ldv<VEC>(xs), Pb = ldv<VEC>(xs + F), Pc = ldv<VEC>(xs + 2 * F);
            Vec<VEC> V0 = vzero, V1 = vzero, V2 = vzero;
            if (vec != nullptr) {      // NULL = identically zero (first layer)
                const float *vs = vec + (size_t)s * F3 + ch;
                V0 = ldv<VEC>(vs), V1 = ldv<VEC>(vs + F), V2 = ldv<VEC>(vs + 2 * F);
            }
            Vec<VEC> fa = ba, fb = bb, fc = bc;
            const float u = g.w * P.inv_rc;
            if (u < 1.f) {
                float val, dval;
                const int k0 = band_setup<false>(u, P, offset, lane, nb, val, dval);
                const float *wk = Wm + (size_t)k0 * F3;
                auto body = [&](int j) {
                    const float gj = __shfl_sync(kFull, val, j);
                    const float *w = wk + (size_t)j * F3;
                    const Vec<VEC> wa = ldv<VEC>(w), wb = ldv<VEC>(w + F), wc = ldv<VEC>(w + 2 * F);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) {
                        fa.v[v] = fmaf(gj, wa.v[v], fa.v[v]);
                        fb.v[v] = fmaf(gj, wb.v[v], fb.v[v]);
                        fc.v[v] = fmaf(gj, wc.v[v], fc.v[v]);
                    }
                };
                if (nb == kBand) {
#pragma unroll
                    for (int j = 0; j < kBand; ++j) body(j);
                } else {
                    for (int j = 0; j < nb; ++j) body(j);
                }
            }
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                ax[v] = fmaf(Pa.v[v], fa.v[v], ax[v]);
                const float tb = Pb.v[v] * fb.v[v] * c1;
                const float tc = Pc.v[v] * fc.v[v] * c2;
                av[0][v] += V0.v[v] * tb + tc * g.x;
                av[1][v] += V1.v[v] * tb + tc * g.y;
                av[2][v] += V2.v[v] * tb + tc * g.z;
            }
        }
    }
    Vec<VEC> o;
#pragma unroll
    for (int v = 0; v < VEC; ++v) o.v[v] = ax[v];
    stv<VEC>(dx + (size_t)row * F + ch, o);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) o.v[v] = av[k][v];
        stv<VEC>(dvec + (size_t)row * F3 + (size_t)k * F + ch, o);
    }
}

// Destination-major backward: per row-edge (dL/du, dL/dd) for this channel slice.
template <int VEC, bool MASKED>
__global__ void __launch_bounds__(256)
edge_bwd_dst_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                    const float4 *__restrict__ geom, const int *__restrict__ rowptr, const int *__restrict__ col,
                    const int *__restrict__ row_mod, const long long *__restrict__ row_xoff, const float *__restrict__ Wt,
                    const float *__restrict__ bias, const float *__restrict__ offset, const float *__restrict__ g_dx,
                    const float *__restrict__ g_dvec, float4 *__restrict__ g_geom, long long n_edges) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= P.n_rows) return;
    const int F = P.hidden, K = P.num_rbf, F3 = 3 * F;
    const int ch = blockIdx.y * (32 * VEC) + lane * VEC;
    const int m = __ldg(row_mod + row);
    const int e0 = __ldg(rowptr + row), e1 = __ldg(rowptr + row + 1);
    float4 *out = g_geom + (size_t)blockIdx.y * n_edges;
    if (m < 0) {
        for (int e = e0 + lane; e < e1; e += 32) out[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    const float *Wm = Wt + (size_t)m * K * F3 + ch;
    const float *xm = xh + __ldg(row_xoff + row) * F3 + ch;
    const Vec<VEC> bc = ldv<VEC>(bias + (size_t)m * F3 + 2 * F + ch);
    const Vec<VEC> gx = ldv<VEC>(g_dx + (size_t)row * F + ch);
    const Vec<VEC> gv0 = ldv<VEC>(g_dvec + (size_t)row * F3 + ch), gv1 = ldv<VEC>(g_dvec + (size_t)row * F3 + F + ch),
                   gv2 = ldv<VEC>(g_dvec + (size_t)row * F3 + 2 * F + ch);
    const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
    const int nb = K < kBand ? K : kBand;
    for (int e = e0; e < e1; ++e) {
        const int s = __ldg(col + e);
        const float4 g = __ldg(geom + e);
        if (MASKED && g.w < 0.f) {             // dead entry of a Verlet-skin list: exact zeros, no gathers, no band
            if (lane == 0) out[e] = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        const float *xs = xm + (size_t)s * F3;
        const Vec<VEC> Pa = ldv<VEC>(xs), Pb = ldv<VEC>(xs + F), Pc = ldv<VEC>(xs + 2 * F);
        Vec<VEC> V0, V1, V2;
#pragma unroll
        for (int v = 0; v < VEC; ++v) V0.v[v] = V1.v[v] = V2.v[v] = 0.f;
        if (vec != nullptr) {          // NULL = identically zero (first layer)
            const float *vs = vec + (size_t)s * F3 + ch;
            V0 = ldv<VEC>(vs), V1 = ldv<VEC>(vs + F), V2 = ldv<VEC>(vs + 2 * F);
        }
        Vec<VEC> fc = bc, da, db, dc;
#pragma unroll
        for (int v = 0; v < VEC; ++v) { da.v[v] = 0.f; db.v[v] = 0.f; dc.v[v] = 0.f; }
        const float u = g.w * P.inv_rc;
        if (u < 1.f) {
            float val, dval;
            const int k0 = band_setup<true>(u, P, offset, lane, nb, val, dval);
            const float *wk = Wm + (size_t)k0 * F3;
            auto body = [&](int j) {
                const float gj = __shfl_sync(kFull, val, j);
                const float hj = __shfl_sync(kFull, dval, j);
                const float *w = wk + (size_t)j * F3;
                const Vec<VEC> wa = ldv<VEC>(w), wb = ldv<VEC>(w + F), wc = ldv<VEC>(w + 2 * F);
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    fc.v[v] = fmaf(gj, wc.v[v], fc.v[v]);
                    da.v[v] = fmaf(hj, wa.v[v], da.v[v]);
                    db.v[v] = fmaf(hj, wb.v[v], db.v[v]);
                    dc.v[v] = fmaf(hj, wc.v[v], dc.v[v]);
                }
            };
            if (nb == kBand) {
#pragma unroll
                for (int j = 0; j < kBand; ++j) body(j);
            } else {
                for (int j = 0; j < nb; ++j) body(j);
            }
        }
        float gd = 0.f, gu0 = 0.f, gu1 = 0.f, gu2 = 0.f;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const float tb = (gv0.v[v] * V0.v[v] + gv1.v[v] * V1.v[v] + gv2.v[v] * V2.v[v]) * c1;   // dL/d(Pb*phib)
            const float tc = (gv0.v[v] * g.x + gv1.v[v] * g.y + gv2.v[v] * g.z) * c2;               // dL/d(Pc*phic)
            gd += gx.v[v] * Pa.v[v] * da.v[v] + tb * Pb.v[v] * db.v[v] + tc * Pc.v[v] * dc.v[v];
            const float cphi = Pc.v[v] * fc.v[v] * c2;
            gu0 += gv0.v[v] * cphi;
            gu1 += gv1.v[v] * cphi;
            gu2 += gv2.v[v] * cphi;
        }
        gd = hn::warp_sum(gd);
        gu0 = hn::warp_sum(gu0);
        gu1 = hn::warp_sum(gu1);
        gu2 = hn::warp_sum(gu2);
        if (lane == 0) out[e] = make_float4(gu0, gu1, gu2, gd);
    }
}

// Source-major backward over the transposed view: grad_xh[m][s] (+=, buffer zero-filled by the caller;
// each (m, s) row is only ever touched by the warp that owns s) and grad_vec[s].
template <int VEC, bool MASKED>
__global__ void __launch_bounds__(256)
edge_bwd_src_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                    const float4 *__restrict__ geom, const int *__restrict__ t_rowptr, const int *__restrict__ t_eid,
                    const int *__restrict__ edge_row, const int *__restrict__ row_mod, const long long *__restrict__ row_xoff,
                    const float *__restrict__ Wt, const float *__restrict__ bias, const float *__restrict__ offset,
                    const float *__restrict__ g_dx, const float *__restrict__ g_dvec, float *__restrict__ grad_xh,
                    float *__restrict__ grad_vec) {
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (s >= P.n_atoms) return;
    const int F = P.hidden, K = P.num_rbf, F3 = 3 * F;
    const int ch = blockIdx.y * (32 * VEC) + lane * VEC;
    const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
    const int nb = K < kBand ? K : kBand;
    const float *vs = vec + (size_t)s * F3 + ch;
    const Vec<VEC> V0 = ldv<VEC>(vs), V1 = ldv<VEC>(vs + F), V2 = ldv<VEC>(vs + 2 * F);
    float gV[3][VEC], gP[3][VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        gV[0][v] = gV[1][v] = gV[2][v] = 0.f;
        gP[0][v] = gP[1][v] = gP[2][v] = 0.f;
    }
    int cur_m = -1;
    long long cur_off = -1;   // element offset of the xh block the accumulators belong to (-1: none)
    bool have = false;
    Vec<VEC> Pb, ba, bb, bc;
#pragma unroll
    for (int v = 0; v < VEC; ++v) Pb.v[v] = ba.v[v] = bb.v[v] = bc.v[v] = 0.f;

    auto flush = [&]() {
        if (!have) return;
        float *dst = grad_xh + cur_off + (long long)s * F3 + ch;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Vec<VEC> o;
#pragma unroll
            for (int v = 0; v < VEC; ++v) o.v[v] = dst[(size_t)k * F + v] + gP[k][v];
            stv<VEC>(dst + (size_t)k * F, o);
#pragma unroll
            for (int v = 0; v < VEC; ++v) gP[k][v] = 0.f;
        }
    };

    const int q0 = __ldg(t_rowptr + s), q1 = __ldg(t_rowptr + s + 1);
    for (int q = q0; q < q1; ++q) {
        const int e = __ldg(t_eid + q);
        if (MASKED && __ldg(&geom[e].w) < 0.f) continue;    // dead entry of a Verlet-skin list
        const int row = __ldg(edge_row + e);
        const int m = __ldg(row_mod + row);
        if (m < 0) continue;
        const long long off = __ldg(row_xoff + row) * F3;
        if (!have || off != cur_off) {
            flush();
            cur_off = off;
            have = true;
            Pb = ldv<VEC>(xh + off + (long long)s * F3 + F + ch);
        }
        if (m != cur_m) {
            cur_m = m;
            ba = ldv<VEC>(bias + (size_t)m * F3 + ch);
            bb = ldv<VEC>(bias + (size_t)m * F3 + F + ch);
            bc = ldv<VEC>(bias + (size_t)m * F3 + 2 * F + ch);
        }
        const float4 g = __ldg(geom + e);
        const Vec<VEC> gx = ldv<VEC>(g_dx + (size_t)row * F + ch);
        const Vec<VEC> gv0 = ldv<VEC>(g_dvec + (size_t)row * F3 + ch), gv1 = ldv<VEC>(g_dvec + (size_t)row * F3 + F + ch),
                       gv2 = ldv<VEC>(g_dvec + (size_t)row * F3 + 2 * F + ch);
        Vec<VEC> fa = ba, fb = bb, fc = bc;
        const float u = g.w * P.inv_rc;
        if (u < 1.f) {
            float val, dval;
            const int k0 = band_setup<false>(u, P, offset, lane, nb, val, dval);
            const float *wk = Wt + ((size_t)m * K + k0) * F3 + ch;
            auto body = [&](int j) {
                const float gj = __shfl_sync(kFull, val, j);
                const float *w = wk + (size_t)j * F3;
                const Vec<VEC> wa = ldv<VEC>(w), wb = ldv<VEC>(w + F), wc = ldv<VEC>(w + 2 * F);
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    fa.v[v] = fmaf(gj, wa.v[v], fa.v[v]);
                    fb.v[v] = fmaf(gj, wb.v[v], fb.v[v]);
                    fc.v[v] = fmaf(gj, wc.v[v], fc.v[v]);
                }
            };
            if (nb == kBand) {
#pragma unroll
                for (int j = 0; j < kBand; ++j) body(j);
            } else {
                for (int j = 0; j < nb; ++j) body(j);
            }
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const float tb = (gv0.v[v] * V0.v[v] + gv1.v[v] * V1.v[v] + gv2.v[v] * V2.v[v]) * c1;
            const float tc = (gv0.v[v] * g.x + gv1.v[v] * g.y + gv2.v[v] * g.z) * c2;
            gP[0][v] = fmaf(gx.v[v], fa.v[v], gP[0][v]);
            gP[1][v] = fmaf(tb, fb.v[v], gP[1][v]);
            gP[2][v] = fmaf(tc, fc.v[v], gP[2][v]);
            const float bphi = Pb.v[v] * fb.v[v] * c1;
            gV[0][v] = fmaf(gv0.v[v], bphi, gV[0][v]);
            gV[1][v] = fmaf(gv1.v[v], bphi, gV[1][v]);
            gV[2][v] = fmaf(gv2.v[v], bphi, gV[2][v]);
        }
    }
    flush();
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        Vec<VEC> o;
#pragma unroll
        for (int v = 0; v < VEC; ++v) o.v[v] = gV[k][v];
        stv<VEC>(grad_vec + (size_t)s * F3 + (size_t)k * F + ch, o);
    }
}

// Filter-weight gradient (only needed when rbf_proj parameters require grad on the fused path):
//   gW[m][k][c] = sum_e env*g_k(d_e) * gphi_e[c],   gb[m][c] = sum_e gphi_e[c]
// One CTA = one (row chunk, module, column slice of <= 384 columns); thread t owns column t of the slice, the
// [K][cols] accumulator lives in shared memory and is updated without atomics (each thread only touches its own
// column).  Partials per chunk are reduced by the caller (fixed order -> deterministic).  edge_live (NULL: every
// entry is an edge) drops the dead entries of a Verlet-skin list from both sums.
__global__ void __launch_bounds__(384)
edge_bwd_w_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                  const float4 *__restrict__ geom, const int *__restrict__ rowptr, const int *__restrict__ col,
                  const int *__restrict__ row_mod, const long long *__restrict__ row_xoff,
                  const unsigned char *__restrict__ edge_live, const float *__restrict__ offset,
                  const float *__restrict__ g_dx, const float *__restrict__ g_dvec, float *__restrict__ gW_part,
                  float *__restrict__ gb_part, int n_chunks, int cols_per_cta) {
    extern __shared__ float acc[];  // [K][cols_per_cta]
    const int F = P.hidden, K = P.num_rbf, F3 = 3 * F;
    const int chunk = blockIdx.x, m = blockIdx.z;
    const int c = blockIdx.y * cols_per_cta + threadIdx.x;  // column in [0, 3F)
    const bool live = threadIdx.x < cols_per_cta && c < F3;
    const int lane = threadIdx.x & 31;
    const int part = live ? c / F : 0, f = live ? c - part * F : 0;
    for (int i = threadIdx.x; i < K * cols_per_cta; i += blockDim.x) acc[i] = 0.f;
    __syncthreads();
    const int rows_per_chunk = (P.n_rows + n_chunks - 1) / n_chunks;
    const int r0 = chunk * rows_per_chunk, r1 = min(P.n_rows, r0 + rows_per_chunk);
    const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
    const int nb = K < kBand ? K : kBand;
    float gb = 0.f;
    for (int row = r0; row < r1; ++row) {
        if (__ldg(row_mod + row) != m) continue;
        const int e0 = __ldg(rowptr + row), e1 = __ldg(rowptr + row + 1);
        const long long xoff = __ldg(row_xoff + row) * F3;
        float gx = 0.f, gv0 = 0.f, gv1 = 0.f, gv2 = 0.f;
        if (live) {
            if (part == 0) gx = __ldg(g_dx + (size_t)row * F + f);
            else {
                gv0 = __ldg(g_dvec + (size_t)row * F3 + f);
                gv1 = __ldg(g_dvec + (size_t)row * F3 + F + f);
                gv2 = __ldg(g_dvec + (size_t)row * F3 + 2 * F + f);
            }
        }
        for (int e = e0; e < e1; ++e) {
            if (edge_live != nullptr && __ldg(edge_live + e) == 0) continue;   // uniform across the CTA
            const int s = __ldg(col + e);
            const float4 g = __ldg(geom + e);
            float gphi = 0.f;
            if (live) {
                const float Pc_ = __ldg(xh + xoff + (long long)s * F3 + c);
                if (part == 0) gphi = gx * Pc_;
                else if (part == 1) {
                    const float *vs = vec + (size_t)s * F3 + f;
                    gphi = (gv0 * __ldg(vs) + gv1 * __ldg(vs + F) + gv2 * __ldg(vs + 2 * F)) * c1 * Pc_;
                } else gphi = (gv0 * g.x + gv1 * g.y + gv2 * g.z) * c2 * Pc_;
            }
            gb += gphi;
            const float u = g.w * P.inv_rc;
            if (u < 1.f) {
                float val, dval;
                const int k0 = band_setup<false>(u, P, offset, lane, nb, val, dval);
                for (int j = 0; j < nb; ++j) {
                    const float gj = __shfl_sync(kFull, val, j);
                    if (live) acc[(k0 + j) * cols_per_cta + threadIdx.x] += gj * gphi;
                }
            }
        }
    }
    __syncthreads();
    if (live) {
        float *dst = gW_part + ((size_t)chunk * P.n_modules + m) * K * F3;
        for (int k = 0; k < K; ++k) dst[(size_t)k * F3 + c] = acc[k * cols_per_cta + threadIdx.x];
        gb_part[((size_t)chunk * P.n_modules + m) * F3 + c] = gb;
    }
}

int pick_vec(int F) { return F % 128 == 0 ? 4 : (F % 64 == 0 ? 2 : (F % 32 == 0 ? 1 : 0)); }

// Every entry point honours flags bit 0 (Verlet-skin superset lists): the row and tile-sweep kernels read the mask from the
// sign of geom[e].w, hn_painn_edge_bwd_w from its live argument.
int validate(const char *where, const hn_edge_params *p) {
    HN_REQUIRE(p != nullptr, where, "null params");
    HN_REQUIRE(pick_vec(p->hidden) != 0, where, "hidden_channels must be a multiple of 32");
    HN_REQUIRE(p->num_rbf >= 2, where, "num_rbf must be >= 2");
    HN_REQUIRE(p->env_p >= 1, where, "envelope exponent must be >= 1");
    HN_REQUIRE(p->n_modules >= 1, where, "n_modules must be >= 1");
    return 0;
}

// p->variant == 1 forces the row-per-warp kernels of this file (A/B measurements, debugging); the default (0) routes
// F % 64 == 0 through the quad-tile kernels of hn_edge_quad.cu.  A per-call flag: the library keeps no selector state.
bool use_quad(const hn_edge_params *p) { return p->variant == 0 && hn::quad::supported(p); }

int row_slices(int hidden) {
    const int v = pick_vec(hidden);
    return v == 0 ? 0 : hidden / (32 * v);
}

}  // namespace

extern "C" int32_t hn_painn_edge_num_slices(int32_t hidden, int32_t variant) {
    hn_edge_params q = {};
    q.hidden = hidden;
    q.variant = variant;
    if (row_slices(hidden) != 0 && use_quad(&q)) return hn::quad::bwd_dst_slices(hidden);
    return row_slices(hidden);
}

// VEC from F; MASKED from flags bit 0 (Verlet-skin superset list, dead entries stored as -d in geom)
#define HN_DISPATCH_VEC(F, FLAGS, CALL)                                         \
    hn::dispatch_bool((FLAGS) & 1, [&](auto masked_) {                          \
        constexpr bool MASKED = decltype(masked_)::value;                       \
        switch (pick_vec(F)) {                                                  \
            case 4: { constexpr int VEC = 4; CALL; break; }                     \
            case 2: { constexpr int VEC = 2; CALL; break; }                     \
            default: { constexpr int VEC = 1; CALL; break; }                    \
        }                                                                       \
    })

extern "C" int hn_painn_edge_fwd(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                                 const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                                 const float *Wt, const float *bias, const float *offset, float *dx, float *dvec,
                                 void *stream) {
    const char *where = "hn_painn_edge_fwd";
    if (int rc = validate(where, p)) return rc;
    if (p->n_rows <= 0) return 0;
    if (use_quad(p)) {
        hn::quad::fwd(p, xh, vec, geom, rowptr, col, row_mod, row_xoff, Wt, bias, offset, dx, dvec, (cudaStream_t)stream);
        return hn::check_launch(where);
    }
    const int wpb = 8;
    dim3 grid((p->n_rows + wpb - 1) / wpb, row_slices(p->hidden));
    HN_DISPATCH_VEC(p->hidden, p->flags, (edge_fwd_kernel<VEC, MASKED><<<grid, 32 * wpb, 0, (cudaStream_t)stream>>>(
                                   *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod, (const long long *)row_xoff, Wt, bias, offset, dx,
                                   dvec)));
    return hn::check_launch(where);
}

extern "C" int hn_painn_edge_bwd_dst(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                                     const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                                     const float *Wt, const float *bias, const float *offset, const float *g_dx,
                                     const float *g_dvec, float *g_geom, int64_t n_edges, void *stream) {
    const char *where = "hn_painn_edge_bwd_dst";
    if (int rc = validate(where, p)) return rc;
    if (p->n_rows <= 0 || n_edges <= 0) return 0;
    if (use_quad(p)) {
        hn::quad::bwd_dst(p, xh, vec, geom, rowptr, col, row_mod, row_xoff, Wt, bias, offset, g_dx, g_dvec, g_geom, n_edges,
                          (cudaStream_t)stream);
        return hn::check_launch(where);
    }
    const int wpb = 8;
    dim3 grid((p->n_rows + wpb - 1) / wpb, row_slices(p->hidden));
    HN_DISPATCH_VEC(p->hidden, p->flags, (edge_bwd_dst_kernel<VEC, MASKED><<<grid, 32 * wpb, 0, (cudaStream_t)stream>>>(
                                   *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod, (const long long *)row_xoff, Wt, bias, offset,
                                   g_dx, g_dvec, (float4 *)g_geom, n_edges)));
    return hn::check_launch(where);
}

extern "C" int hn_painn_edge_bwd_src(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                                     const int32_t *t_rowptr, const int32_t *t_eid, const int32_t *edge_row,
                                     const int32_t *row_mod, const int64_t *row_xoff, const float *Wt, const float *bias,
                                     const float *offset, const float *g_dx, const float *g_dvec, float *grad_xh,
                                     float *grad_vec, void *stream) {
    const char *where = "hn_painn_edge_bwd_src";
    if (int rc = validate(where, p)) return rc;
    if (p->n_atoms <= 0) return 0;
    if (use_quad(p)) {
        hn::quad::bwd_src(p, xh, vec, geom, t_rowptr, t_eid, edge_row, row_mod, row_xoff, Wt, bias, offset, g_dx, g_dvec, grad_xh,
                          grad_vec, (cudaStream_t)stream);
        return hn::check_launch(where);
    }
    const int wpb = 8;
    dim3 grid((p->n_atoms + wpb - 1) / wpb, row_slices(p->hidden));
    HN_DISPATCH_VEC(p->hidden, p->flags, (edge_bwd_src_kernel<VEC, MASKED><<<grid, 32 * wpb, 0, (cudaStream_t)stream>>>(
                                   *p, xh, vec, (const float4 *)geom, t_rowptr, t_eid, edge_row, row_mod, (const long long *)row_xoff, Wt,
                                   bias, offset, g_dx, g_dvec, grad_xh, grad_vec)));
    return hn::check_launch(where);
}

extern "C" int hn_painn_edge_bwd_w(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                                   const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                                   const uint8_t *live, const float *offset, const float *g_dx, const float *g_dvec,
                                   float *gW_part, float *gb_part, int32_t n_chunks, void *stream) {
    const char *where = "hn_painn_edge_bwd_w";
    if (int rc = validate(where, p)) return rc;
    HN_REQUIRE(!(p->flags & 1) || live != nullptr, where, "a Verlet-skin list (flags bit 0) needs the live mask");
    HN_REQUIRE(n_chunks >= 1, where, "n_chunks must be >= 1");
    // column slice: the widest multiple of 32 (F % 32 == 0, so 3F is one) up to 384 whose [K][cols] fp32 accumulator fits in
    // shared memory; several slices when 3F is wider, the last one partly filled
    const int F3 = 3 * p->hidden;
    const int fit = (int)((size_t)227 * 1024 / ((size_t)p->num_rbf * sizeof(float))) / 32 * 32;
    int cols = F3 < 384 ? F3 : 384;
    cols = cols < fit ? cols : fit;
    HN_REQUIRE(cols >= 32, where, "num_rbf too large for the shared-memory accumulator (K * 32 columns * 4 bytes > 227 KB)");
    const size_t smem = (size_t)p->num_rbf * cols * sizeof(float);
    HN_CUDA(cudaFuncSetAttribute(edge_bwd_w_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), where);
    dim3 grid(n_chunks, (F3 + cols - 1) / cols, p->n_modules);
    edge_bwd_w_kernel<<<grid, cols, smem, (cudaStream_t)stream>>>(*p, xh, vec, (const float4 *)geom, rowptr, col, row_mod,
                                                                  (const long long *)row_xoff, (p->flags & 1) ? live : nullptr,
                                                                  offset, g_dx, g_dvec, gW_part, gb_part, n_chunks, cols);
    return hn::check_launch(where);
}
