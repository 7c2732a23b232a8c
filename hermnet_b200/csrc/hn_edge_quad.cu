// Tile-sweep PaiNN edge kernels: forward and destination-major backward (default for F in {64, 128, 256, 512}).
//
// Same arithmetic and reference lines as hn_edge.cu (rmnet.py:55-73 message/aggregate, rmnet.py:168-193 Gaussian RBF x
// polynomial envelope, hermnet.py:51-61 per-element sub-networks):
//   phi_e = W[m] . (env(u) * gauss_k(u)) + b[m],  u = d_e / rc
//   dx[r] = sum_e xh[m][s][0:F] * phi_e[0:F],   dvec[r][k] = sum_e (vec[s][k]*xh_b*phi_b/sqrt(3) + xh_c*phi_c*u_e[k]) / sqrt(F)
//
// Why another loop nest.  The row-per-warp kernels re-read a 12 x 3F band of W for EVERY edge: 18 KB of L1 traffic
// per edge at F=128 against 3 KB of gathered features, and ncu shows them pinned at >80 % of the L1/LSU peak.  Rows
// are sorted by distance by the graph builder, so CONSECUTIVE edges of a row have overlapping bands.  Here a warp
// walks its row in tiles of T consecutive edges (forward T=4, backward T=2) and sweeps the UNION of the tile's bands
// once: every W row it loads feeds T edges of packed FMAs (fma.rn.f32x2).
//   * per tile, lane (q = lane % T, sub = lane / T) evaluates env*gauss_k(d_q) for k = kmin+sub, +32/T, ... of the
//     union (exact Gaussian values, also outside the edge's own 12-wide band -- those terms are < 1.5e-8 and were
//     dropped by the row kernels) into a per-warp shared-memory table of (g,g) pairs; the sweep broadcasts them with
//     LDS.128 and needs no shuffles;
//   * the union is a 64-bit mask relative to kmin (holes between distance shells are skipped); when the bands of a
//     tile span more than 64 basis functions (rows that are no longer distance-sorted because the graph is re-used
//     after the atoms moved) the tile falls back to a single edge: sharing is lost, accuracy never;
//   * accumulation per row stays private to the warp: no atomics, deterministic order;
//   * F is a template parameter, so every address inside the sweep is base + immediate;
//   * Verlet-skin superset lists (flags bit 0, geom.w = -d on the dead entries) run the MASKED instantiations: a dead entry
//     is padding to its tile (no band, no gathers, exact-zero g_geom) and is dropped by the source-major pipeline.
#include "hn_common.cuh"
#include "hn_edge_quad.cuh"

namespace {

typedef unsigned long long u64;

constexpr unsigned kFull = 0xffffffffu;
constexpr int kTabW = 64;         // basis functions a tile's union may span
constexpr int kLo = 5, kHi = 6;   // band = floor(x)-5 .. floor(x)+6, x = u*(K-1)  (same band as hn_edge.cu)
constexpr int kWarps = 8;
constexpr int kBig = 1 << 20;
#ifndef HN_FWD_PIPE
#define HN_FWD_PIPE 0
#endif

__device__ __forceinline__ u64 pk(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
// NP packed pairs (= 2*NP consecutive channels) from global memory through the read-only path
template <int NP>
struct Pairs {
    u64 p[NP];
};
template <int NP>
__device__ __forceinline__ Pairs<NP> ldp(const float *ptr) {
    Pairs<NP> r;
    if constexpr (NP == 2) {
        const ulonglong2 t = __ldg(reinterpret_cast<const ulonglong2 *>(ptr));
        r.p[0] = t.x;
        r.p[1] = t.y;
    } else {
        r.p[0] = __ldg(reinterpret_cast<const u64 *>(ptr));
    }
    return r;
}

// Same loads as ordered (volatile) asm: inside the sweeps every filter row is re-loaded IN PLACE right after its last use
// (the next row's values travel while the remaining FMAs of this row issue), which only works if the compiler keeps the
// load where it is written.
template <int NP>
__device__ __forceinline__ Pairs<NP> ldp_ordered(const float *ptr) {
    Pairs<NP> r;
    if constexpr (NP == 2) {
        asm volatile("ld.global.nc.v2.u64 {%0, %1}, [%2];" : "=l"(r.p[0]), "=l"(r.p[1]) : "l"(ptr));
    } else {
        asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(r.p[0]) : "l"(ptr));
    }
    return r;
}
__device__ __forceinline__ void lds_pair2(unsigned addr, u64 &a, u64 &b) {
    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ void fma2v(u64 &acc, u64 a, u64 b) {   // ordered acc += a * b
    asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ u64 mul2v(u64 a, u64 b) {
    u64 d;
    asm volatile("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// polynomial envelope (rmnet.py:183-193) and its derivative with respect to u
template <bool DERIV>
__device__ __forceinline__ void envelope(float u, int p, float &env, float &denv) {
    const float a = -0.5f * (float)((p + 1) * (p + 2)), b = (float)(p * (p + 2)), c = -0.5f * (float)(p * (p + 1));
    float um;
    if (p == 5) {
        const float u2 = u * u;
        um = u2 * u2;
    } else {
        um = 1.f;
        for (int i = 0; i < p - 1; ++i) um *= u;
    }
    const float u0 = um * u, u1 = u0 * u, u2 = u1 * u;
    env = 1.f + a * u0 + b * u1 + c * u2;
    denv = 0.f;
    if (DERIV) denv = a * (float)p * um + b * (float)(p + 1) * u0 + c * (float)(p + 2) * u1;
}

// Edge eb + (lane % T) of the row: source atom and geometry (zeros past the end of the row).  MASKED: a dead entry of a
// Verlet-skin list (geom.w = -d < 0) gets s = -1 like the padding past the row end, so it adds nothing to the tile's band
// union and takes no gathers; it still counts as one of the tile's edges.
template <int T>
struct Head {
    float4 g;
    int s;
};
template <int T, bool MASKED>
__device__ __forceinline__ Head<T> load_head(const float4 *__restrict__ geom, const int *__restrict__ col, int eb, int e1,
                                             int lane) {
    Head<T> h;
    const int e = eb + (lane & (T - 1));
    h.g = make_float4(0.f, 0.f, 0.f, 0.f);
    h.s = -1;
    if (e < e1) {
        h.g = __ldg(geom + e);
        h.s = __ldg(col + e);
        if (MASKED && h.g.w < 0.f) h.s = -1;
    }
    return h;
}

// Sets up the tile whose head (edges eb .. eb+T-1, h.s < 0 past the row end) was loaded by load_head.  Returns the
// number of edges the tile takes (T, fewer at the end of a row, 1 when the bands span >= kTabW basis functions) and
// fills tab[kk][2q..2q+1] = env*gauss_{kmin+kk}(d_q) (DERIV: tab[kTabW + kk] = d/dd of it) for every kk of the mask.
template <int T, bool DERIV>
__device__ __forceinline__ int tile_setup(const hn_edge_params &P, const float *__restrict__ offset, const Head<T> &h,
                                          int n_left, int lane, float *tab, int &kmin, u64 &mask) {
    constexpr int NSUB = 32 / T;
    const int q = lane & (T - 1), sub = lane / T;
    const int K = P.num_rbf;
    const float u = h.g.w * P.inv_rc;
    const bool valid = h.s >= 0 && u < 1.f;
    int lo = kBig, hi = -1;
    if (valid) {
        const int kc = (int)(u * (float)(K - 1));
        lo = max(kc - kLo, 0);
        hi = min(kc + kHi, K - 1);
    }
    int mn = lo, mx = hi;
#pragma unroll
    for (int o = 1; o < T; o <<= 1) {
        mn = min(mn, __shfl_xor_sync(kFull, mn, o));
        mx = max(mx, __shfl_xor_sync(kFull, mx, o));
    }
    int cnt = n_left < T ? n_left : T;
    if (mx - mn >= kTabW) {        // not distance-sorted: take the first edge alone
        cnt = 1;
        mn = __shfl_sync(kFull, lo, 0);
        mx = __shfl_sync(kFull, hi, 0);
    }
    const bool act = valid && q < cnt;
    u64 bits = 0ull;
    if (act) bits = ((2ull << (hi - lo)) - 1ull) << (lo - mn);
    const unsigned b_lo = __reduce_or_sync(kFull, (unsigned)bits), b_hi = __reduce_or_sync(kFull, (unsigned)(bits >> 32));
    mask = ((u64)b_hi << 32) | (u64)b_lo;
    kmin = mn;
    const int width = mx - mn + 1;    // <= kTabW; <= 0 when no edge of the tile is inside the cutoff
    float env = 0.f, denv = 0.f;
    if (act) envelope<DERIV>(u, P.env_p, env, denv);
    const float *off = offset + mn;
    for (int kk = sub; kk < width; kk += NSUB) {
        if ((mask >> kk) & 1ull) {
            float val = 0.f, dval = 0.f;
            if (act) {
                const float diff = u - __ldg(off + kk);
                const float gg = __expf(P.coeff * diff * diff);
                val = env * gg;
                if (DERIV) dval = (denv * gg + val * (2.f * P.coeff * diff)) * P.inv_rc;
            }
            *reinterpret_cast<float2 *>(tab + kk * (2 * T) + 2 * q) = make_float2(val, val);
            if (DERIV) *reinterpret_cast<float2 *>(tab + (kTabW + kk) * (2 * T) + 2 * q) = make_float2(dval, dval);
        }
    }
    __syncwarp();
    return cnt;
}

// (g,g) pairs of the T edges of a tile for table row kk
template <int T>
__device__ __forceinline__ void load_pairs(const float *tab_row, u64 (&gg)[T]) {
    if constexpr (T == 4) {
        const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(tab_row), b = *reinterpret_cast<const ulonglong2 *>(tab_row + 4);
        gg[0] = a.x;
        gg[1] = a.y;
        gg[2] = b.x;
        gg[3] = b.y;
    } else {
        const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(tab_row);
        gg[0] = a.x;
        gg[1] = a.y;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// forward.  One warp = one (row, slice of 64*NP channels); the slices of a row sit in the same CTA.
// ---------------------------------------------------------------------------------------------------------------
// HV = false: vec is identically zero (first layer, hermnet.py:124): the b part of the filter and the vec gathers vanish.
template <int F, int NP, bool HV, bool MASKED>
__global__ void __launch_bounds__(32 * kWarps, 2)
edge_fwd_quad_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                     const float4 *__restrict__ geom, const int *__restrict__ rowptr, const int *__restrict__ col,
                     const int *__restrict__ row_mod, const long long *__restrict__ row_xoff, const float *__restrict__ Wt,
                     const float *__restrict__ bias, const float *__restrict__ offset, float *__restrict__ dx,
                     float *__restrict__ dvec) {
    constexpr int T = 4, VEC = 2 * NP, F3 = 3 * F, NS = F / (32 * VEC);
    __shared__ __align__(16) float s_tab[kWarps][kTabW * 2 * T];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int unit = blockIdx.x * kWarps + warp;
    const int row = unit / NS, slice = unit % NS;
    if (row >= P.n_rows) return;
    const int ch = slice * (32 * VEC) + lane * VEC;
    const int m = __ldg(row_mod + row);
    float *tab = s_tab[warp];
    float ax[VEC], av[3][VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) ax[v] = av[0][v] = av[1][v] = av[2][v] = 0.f;
    if (m >= 0) {
        const int e0 = __ldg(rowptr + row), e1 = __ldg(rowptr + row + 1);
        const float *Wm = Wt + (size_t)m * P.num_rbf * F3 + ch;
        const float *xm = xh + __ldg(row_xoff + row) * F3 + ch;
        const float *vm = vec + ch;
        const float *bm = bias + (size_t)m * F3 + ch;
        const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
        int eb = e0;
        Head<T> h = load_head<T, MASKED>(geom, col, eb, e1, lane);
        while (eb < e1) {
            int kmin;
            u64 mask;
            const int cnt = tile_setup<T, false>(P, offset, h, e1 - eb, lane, tab, kmin, mask);
            const Head<T> hn = load_head<T, MASKED>(geom, col, eb + cnt, e1, lane);    // next tile's head, in flight during the sweep
            u64 fa[T][NP], fb[T][NP], fc[T][NP];
            {
                const Pairs<NP> ba = ldp<NP>(bm), bb = ldp<NP>(bm + F), bc = ldp<NP>(bm + 2 * F);
#pragma unroll
                for (int j = 0; j < T; ++j)
#pragma unroll
                    for (int n = 0; n < NP; ++n) {
                        fa[j][n] = ba.p[n];
                        fb[j][n] = HV ? bb.p[n] : 0ull;
                        fc[j][n] = bc.p[n];
                    }
            }
            // sweep the runs of consecutive basis functions of the union mask; software-pipelined in place
            const unsigned tab_s = (unsigned)__cvta_generic_to_shared(tab);
            for (u64 mk = mask; mk != 0ull;) {
                const int k0 = __ffsll((long long)mk) - 1;
                const u64 inv = ~(mk >> k0);
                const int len = inv == 0ull ? 64 - k0 : __ffsll((long long)inv) - 1;
                mk = (k0 + len >= 64) ? 0ull : (mk >> (k0 + len)) << (k0 + len);
                const float *w = Wm + (size_t)(kmin + k0) * F3;
                unsigned t = tab_s + k0 * (2 * T * 4);
                Pairs<NP> wa = ldp_ordered<NP>(w), wb, wc = ldp_ordered<NP>(w + 2 * F);
                if constexpr (HV) wb = ldp_ordered<NP>(w + F);
                u64 gg[T];
                lds_pair2(t, gg[0], gg[1]);
                lds_pair2(t + 16, gg[2], gg[3]);
#pragma unroll 1
                for (int i = 1; i <= len; ++i) {
                    if (i < len) {       // the last pass re-loads its own row (harmless, stays inside the matrix)
                        w += F3;
                        t += 2 * T * 4;
                    }
#pragma unroll
                    for (int j = 0; j < T; ++j)
#pragma unroll
                        for (int n = 0; n < NP; ++n) fma2v(fa[j][n], gg[j], wa.p[n]);
                    wa = ldp_ordered<NP>(w);
                    if constexpr (HV) {
#pragma unroll
                        for (int j = 0; j < T; ++j)
#pragma unroll
                            for (int n = 0; n < NP; ++n) fma2v(fb[j][n], gg[j], wb.p[n]);
                        wb = ldp_ordered<NP>(w + F);
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j)
#pragma unroll
                        for (int n = 0; n < NP; ++n) fma2v(fc[j][n], gg[j], wc.p[n]);
                    lds_pair2(t, gg[0], gg[1]);
#pragma unroll
                    for (int j = 2; j < T; ++j)
#pragma unroll
                        for (int n = 0; n < NP; ++n) fma2v(fc[j][n], gg[j], wc.p[n]);
                    wc = ldp_ordered<NP>(w + 2 * F);
                    lds_pair2(t + 16, gg[2], gg[3]);
                }
            }
            __syncwarp();    // table reads done before the next tile's fill
            Pairs<NP> G0[6], G1[6];      // gathered (Pa, Pb, Pc, V0, V1, V2) of the current / next edge
            float U0[3], U1[3];
            auto gather = [&](int j, Pairs<NP>(&G)[6], float(&U)[3]) {
                const int sj = __shfl_sync(kFull, h.s, j);
                U[0] = __shfl_sync(kFull, h.g.x, j);
                U[1] = __shfl_sync(kFull, h.g.y, j);
                U[2] = __shfl_sync(kFull, h.g.z, j);
                const float *xs = xm + (size_t)sj * F3;
                const float *vs = vm + (size_t)sj * F3;
                G[0] = ldp<NP>(xs);
                G[2] = ldp<NP>(xs + 2 * F);
                if constexpr (HV) {
                    G[1] = ldp<NP>(xs + F);
                    G[3] = ldp<NP>(vs);
                    G[4] = ldp<NP>(vs + F);
                    G[5] = ldp<NP>(vs + 2 * F);
                }
            };
            auto fold = [&](int j, const Pairs<NP>(&G)[6], const float(&U)[3]) {
#pragma unroll
                for (int n = 0; n < NP; ++n) {
                    float pa[2], pb[2] = {0.f, 0.f}, pc[2], v0[2] = {0.f, 0.f}, v1[2] = {0.f, 0.f}, v2[2] = {0.f, 0.f}, qa[2],
                          qb[2] = {0.f, 0.f}, qc[2];
                    upk(G[0].p[n], pa[0], pa[1]);
                    upk(G[2].p[n], pc[0], pc[1]);
                    upk(fa[j][n], qa[0], qa[1]);
                    upk(fc[j][n], qc[0], qc[1]);
                    if constexpr (HV) {
                        upk(G[1].p[n], pb[0], pb[1]);
                        upk(G[3].p[n], v0[0], v0[1]);
                        upk(G[4].p[n], v1[0], v1[1]);
                        upk(G[5].p[n], v2[0], v2[1]);
                        upk(fb[j][n], qb[0], qb[1]);
                    }
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int v = 2 * n + hh;
                        ax[v] = fmaf(pa[hh], qa[hh], ax[v]);
                        const float tc = pc[hh] * qc[hh] * c2;
                        if constexpr (HV) {
                            const float tb = pb[hh] * qb[hh] * c1;
                            av[0][v] += v0[hh] * tb + tc * U[0];
                            av[1][v] += v1[hh] * tb + tc * U[1];
                            av[2][v] += v2[hh] * tb + tc * U[2];
                        } else {
                            av[0][v] = fmaf(tc, U[0], av[0][v]);
                            av[1][v] = fmaf(tc, U[1], av[1][v]);
                            av[2][v] = fmaf(tc, U[2], av[2][v]);
                        }
                    }
                }
            };
            if constexpr ((!HV || HN_FWD_PIPE) && !MASKED) {
            gather(0, G0, U0);
            if (cnt > 1) gather(1, G1, U1);
            fold(0, G0, U0);
            if (cnt > 1) {
                if (cnt > 2) gather(2, G0, U0);
                fold(1, G1, U1);
                if (cnt > 2) {
                    if (cnt > 3) gather(3, G1, U1);
                    fold(2, G0, U0);
                    if (cnt > 3) fold(3, G1, U1);
                }
            }
            } else {
                // MASKED: lane j < T holds edge j of the tile; a dead edge (s < 0) is neither gathered nor folded
                const unsigned live = MASKED ? __ballot_sync(kFull, h.s >= 0) : ~0u;
#pragma unroll
                for (int j = 0; j < T; ++j)
                    if (j < cnt && ((live >> j) & 1u)) {
                        gather(j, G0, U0);
                        fold(j, G0, U0);
                    }
            }
            eb += cnt;
            h = hn;
        }
    }
    hn::Vec<VEC> o;
#pragma unroll
    for (int v = 0; v < VEC; ++v) o.v[v] = ax[v];
    hn::stv<VEC>(dx + (size_t)row * F + ch, o);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) o.v[v] = av[k][v];
        hn::stv<VEC>(dvec + (size_t)row * F3 + (size_t)k * F + ch, o);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// destination-major backward: per row-edge (dL/du_x, dL/du_y, dL/du_z, dL/dd), one plane per channel slice.
//   dL/dd  = sum_c [ gx Pa phi_a' + tb Pb phi_b' + tc Pc phi_c' ],  phi' = sum_k W_k d(env g_k)/dd
//          = sum_k h_k(d) . sum_c (qa W_a[k] + qb W_b[k] + qc W_c[k]),  qa = gx Pa, qb = tb Pb, qc = tc Pc
//   dL/du  = sum_c gv[.] Pc phi_c / sqrt(F)
// tb = <gv, V>/sqrt(3F), tc = <gv, u>/sqrt(F) as in hn_edge.cu.  Tiles of 2 edges (the sweep carries 11 packed
// registers per edge); the gathers are issued before the sweep, so their latency hides behind it.  The 8 per-tile
// partial sums (2 edges x 4 values) are reduced across the warp with a halving exchange (8 shuffles instead of 40).
// ---------------------------------------------------------------------------------------------------------------
template <int F, int NP, bool HV, bool MASKED>
__global__ void __launch_bounds__(32 * kWarps, 2)
edge_bwd_dst_quad_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                         const float4 *__restrict__ geom, const int *__restrict__ rowptr, const int *__restrict__ col,
                         const int *__restrict__ row_mod, const long long *__restrict__ row_xoff, const float *__restrict__ Wt,
                         const float *__restrict__ bias, const float *__restrict__ offset, const float *__restrict__ g_dx,
                         const float *__restrict__ g_dvec, float4 *__restrict__ g_geom, long long n_edges) {
    constexpr int T = 2, VEC = 2 * NP, F3 = 3 * F, NS = F / (32 * VEC);
    __shared__ __align__(16) float s_tab[kWarps][2 * kTabW * 2 * T];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int unit = blockIdx.x * kWarps + warp;
    const int row = unit / NS, slice = unit % NS;
    if (row >= P.n_rows) return;
    const int ch = slice * (32 * VEC) + lane * VEC;
    const int m = __ldg(row_mod + row);
    const int e0 = __ldg(rowptr + row), e1 = __ldg(rowptr + row + 1);
    float4 *out = g_geom + (size_t)slice * n_edges;
    if (m < 0) {
        for (int e = e0 + lane; e < e1; e += 32) out[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    float *tab = s_tab[warp];
    const float *Wm = Wt + (size_t)m * P.num_rbf * F3 + ch;
    const float *xm = xh + __ldg(row_xoff + row) * F3 + ch;
    const float *vm = vec + ch;
    const Pairs<NP> bc = ldp<NP>(bias + (size_t)m * F3 + 2 * F + ch);
    float gx[VEC], gv[3][VEC];
    {
        const hn::Vec<VEC> t = hn::ldv<VEC>(g_dx + (size_t)row * F + ch);
        const hn::Vec<VEC> t0 = hn::ldv<VEC>(g_dvec + (size_t)row * F3 + ch), t1 = hn::ldv<VEC>(g_dvec + (size_t)row * F3 + F + ch),
                           t2 = hn::ldv<VEC>(g_dvec + (size_t)row * F3 + 2 * F + ch);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            gx[v] = t.v[v];
            gv[0][v] = t0.v[v];
            gv[1][v] = t1.v[v];
            gv[2][v] = t2.v[v];
        }
    }
    const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
    int eb = e0;
    Head<T> h = load_head<T, MASKED>(geom, col, eb, e1, lane);
    while (eb < e1) {
        // gathers of the T edges first (independent of the table), then the table, then the sweep
        Pairs<NP> Pa[T], Pb[T], Pc[T], V0[T], V1[T], V2[T];
        float ux[T], uy[T], uz[T];
        // MASKED: lane j < T holds edge j of the tile; a dead edge (s < 0) is not gathered and its outputs are exact zeros
        const unsigned live = MASKED ? __ballot_sync(kFull, h.s >= 0) : ~0u;
#pragma unroll
        for (int j = 0; j < T; ++j) {
            int sj = __shfl_sync(kFull, h.s, j);
            ux[j] = __shfl_sync(kFull, h.g.x, j);
            uy[j] = __shfl_sync(kFull, h.g.y, j);
            uz[j] = __shfl_sync(kFull, h.g.z, j);
            if (MASKED && sj < 0) {    // dead or past the row end: zeros feed the sweep, nothing is loaded
#pragma unroll
                for (int n = 0; n < NP; ++n) Pa[j].p[n] = Pb[j].p[n] = Pc[j].p[n] = V0[j].p[n] = V1[j].p[n] = V2[j].p[n] = 0ull;
                continue;
            }
            if (sj < 0) sj = __shfl_sync(kFull, h.s, 0);   // past the row end: a valid address, the result is discarded
            const float *xs = xm + (size_t)sj * F3;
            const float *vs = vm + (size_t)sj * F3;
            Pa[j] = ldp<NP>(xs);
            Pc[j] = ldp<NP>(xs + 2 * F);
            if constexpr (HV) {
                Pb[j] = ldp<NP>(xs + F);
                V0[j] = ldp<NP>(vs);
                V1[j] = ldp<NP>(vs + F);
                V2[j] = ldp<NP>(vs + 2 * F);
            }
        }
        int kmin;
        u64 mask;
        const int cnt = tile_setup<T, true>(P, offset, h, e1 - eb, lane, tab, kmin, mask);
        const Head<T> hn = load_head<T, MASKED>(geom, col, eb + cnt, e1, lane);
        u64 qa[T][NP], qb[T][NP], qc[T][NP], fc[T][NP], ds[T];
        float rc_[T][VEC];    // Pc / sqrt(F): the u-independent factor of dL/du
#pragma unroll
        for (int j = 0; j < T; ++j) {
            ds[j] = 0ull;
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                fc[j][n] = bc.p[n];
                float pa[2], pb[2] = {0.f, 0.f}, pc[2], v0[2] = {0.f, 0.f}, v1[2] = {0.f, 0.f}, v2[2] = {0.f, 0.f}, a_[2], b_[2], c_[2];
                upk(Pa[j].p[n], pa[0], pa[1]);
                upk(Pc[j].p[n], pc[0], pc[1]);
                if constexpr (HV) {
                    upk(Pb[j].p[n], pb[0], pb[1]);
                    upk(V0[j].p[n], v0[0], v0[1]);
                    upk(V1[j].p[n], v1[0], v1[1]);
                    upk(V2[j].p[n], v2[0], v2[1]);
                }
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int v = 2 * n + hh;
                    const float tb = (gv[0][v] * v0[hh] + gv[1][v] * v1[hh] + gv[2][v] * v2[hh]) * c1;
                    const float tc = (gv[0][v] * ux[j] + gv[1][v] * uy[j] + gv[2][v] * uz[j]) * c2;
                    a_[hh] = gx[v] * pa[hh];
                    b_[hh] = tb * pb[hh];
                    c_[hh] = tc * pc[hh];
                    rc_[j][v] = pc[hh] * c2;
                }
                qa[j][n] = pk(a_[0], a_[1]);
                qb[j][n] = pk(b_[0], b_[1]);
                qc[j][n] = pk(c_[0], c_[1]);
            }
        }
        const unsigned tab_s = (unsigned)__cvta_generic_to_shared(tab);
        for (u64 mk = mask; mk != 0ull;) {
            const int k0 = __ffsll((long long)mk) - 1;
            const u64 inv = ~(mk >> k0);
            const int len = inv == 0ull ? 64 - k0 : __ffsll((long long)inv) - 1;
            mk = (k0 + len >= 64) ? 0ull : (mk >> (k0 + len)) << (k0 + len);
            const float *w = Wm + (size_t)(kmin + k0) * F3;
            unsigned t = tab_s + k0 * (2 * T * 4);
            Pairs<NP> wa = ldp_ordered<NP>(w), wb, wc = ldp_ordered<NP>(w + 2 * F);
            if constexpr (HV) wb = ldp_ordered<NP>(w + F);
            u64 gg[T], hh[T];
            lds_pair2(t, gg[0], gg[1]);
            lds_pair2(t + kTabW * 2 * T * 4, hh[0], hh[1]);
#pragma unroll 1
            for (int i = 1; i <= len; ++i) {
                if (i < len) {           // the last pass re-loads its own row (harmless, stays inside the matrix)
                    w += F3;
                    t += 2 * T * 4;
                }
                // per edge and channel pair: tt = qa Wa + qb Wb + qc Wc, then ds += h * tt; fc += g * Wc
                u64 tt[T][NP];
#pragma unroll
                for (int j = 0; j < T; ++j)
#pragma unroll
                    for (int n = 0; n < NP; ++n) tt[j][n] = mul2v(qa[j][n], wa.p[n]);
                wa = ldp_ordered<NP>(w);
                if constexpr (HV) {
#pragma unroll
                    for (int j = 0; j < T; ++j)
#pragma unroll
                        for (int n = 0; n < NP; ++n) fma2v(tt[j][n], qb[j][n], wb.p[n]);
                    wb = ldp_ordered<NP>(w + F);
                }
#pragma unroll
                for (int j = 0; j < T; ++j)
#pragma unroll
                    for (int n = 0; n < NP; ++n) {
                        fma2v(tt[j][n], qc[j][n], wc.p[n]);
                        fma2v(fc[j][n], gg[j], wc.p[n]);
                    }
                wc = ldp_ordered<NP>(w + 2 * F);
                lds_pair2(t, gg[0], gg[1]);
#pragma unroll
                for (int j = 0; j < T; ++j)
#pragma unroll
                    for (int n = 0; n < NP; ++n) fma2v(ds[j], hh[j], tt[j][n]);
                lds_pair2(t + kTabW * 2 * T * 4, hh[0], hh[1]);
            }
        }
        __syncwarp();
        // per-lane partial sums: val[4*j + {0,1,2}] = dL/du, val[4*j + 3] = dL/dd
        float val[4 * T];
#pragma unroll
        for (int j = 0; j < T; ++j) {
            float d0, d1, gu0 = 0.f, gu1 = 0.f, gu2 = 0.f;
            upk(ds[j], d0, d1);
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                float f_[2];
                upk(fc[j][n], f_[0], f_[1]);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int v = 2 * n + hh;
                    const float cphi = rc_[j][v] * f_[hh];
                    gu0 = fmaf(gv[0][v], cphi, gu0);
                    gu1 = fmaf(gv[1][v], cphi, gu1);
                    gu2 = fmaf(gv[2][v], cphi, gu2);
                }
            }
            val[4 * j + 0] = gu0;
            val[4 * j + 1] = gu1;
            val[4 * j + 2] = gu2;
            val[4 * j + 3] = d0 + d1;
        }
        // halving exchange over lane bits 16, 8, 4 (value-index bits 4, 2, 1), then plain butterflies over bits 2, 1
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const bool up = lane & 16;
            const float send = up ? val[i] : val[i + 4], keep = up ? val[i + 4] : val[i];
            val[i] = keep + __shfl_xor_sync(kFull, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const bool up = lane & 8;
            const float send = up ? val[i] : val[i + 2], keep = up ? val[i + 2] : val[i];
            val[i] = keep + __shfl_xor_sync(kFull, send, 8);
        }
        {
            const bool up = lane & 4;
            const float send = up ? val[0] : val[1], keep = up ? val[1] : val[0];
            val[0] = keep + __shfl_xor_sync(kFull, send, 4);
        }
        val[0] += __shfl_xor_sync(kFull, val[0], 2);
        val[0] += __shfl_xor_sync(kFull, val[0], 1);
        // lane holds the total of value index idx = lane >> 2: edge idx >> 2, component idx & 3
        const int idx = lane >> 2;
        if ((lane & 3) == 0 && (idx >> 2) < cnt)
            reinterpret_cast<float *>(out + eb)[idx] = ((live >> (idx >> 2)) & 1u) ? val[0] : 0.f;
        eb += cnt;
        h = hn;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// source-major backward over the transposed view (entries of a source sorted by (module, distance)):
//   grad_xh[m][s] (+=; zero-filled by the caller, each (m, s) row is only touched by the warp that owns s)
//   grad_vec[s]
// A source's entries of one sub-network are few (N_neigh / n_modules) and spread over the whole distance range, so
// their bands barely overlap: one edge per sweep here.  What this kernel changes against edge_bwd_src_kernel is
// latency, not bytes: the index chain t_eid -> edge_row -> (row_mod, row_xoff) is software-pipelined three entries
// deep, the 4F gathered gradient values are in flight during the sweep, the filter rows are re-loaded in place, the
// band values come from a 12-entry shared-memory table (one LDS.64 per basis function instead of a shuffle) and
// the FMAs are packed.
// ---------------------------------------------------------------------------------------------------------------
template <int F, int NP, bool MASKED>
__global__ void __launch_bounds__(32 * kWarps, 2)
edge_bwd_src_sweep_kernel(const hn_edge_params P, const float *__restrict__ xh, const float *__restrict__ vec,
                          const float4 *__restrict__ geom, const int *__restrict__ t_rowptr, const int *__restrict__ t_eid,
                          const int *__restrict__ edge_row, const int *__restrict__ row_mod,
                          const long long *__restrict__ row_xoff, const float *__restrict__ Wt, const float *__restrict__ bias,
                          const float *__restrict__ offset, const float *__restrict__ g_dx, const float *__restrict__ g_dvec,
                          float *__restrict__ grad_xh, float *__restrict__ grad_vec) {
    constexpr int VEC = 2 * NP, F3 = 3 * F, NS = F / (32 * VEC), NB = kLo + kHi + 1;
    __shared__ __align__(16) float s_tab[kWarps][2 * 16];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int unit = blockIdx.x * kWarps + warp;
    const int s = unit / NS, slice = unit % NS;
    if (s >= P.n_atoms) return;
    const int K = P.num_rbf;
    const int ch = slice * (32 * VEC) + lane * VEC;
    const float c1 = 1.0f / sqrtf(3.0f * (float)F), c2 = 1.0f / sqrtf((float)F);
    float *tab = s_tab[warp];
    const unsigned tab_s = (unsigned)__cvta_generic_to_shared(tab);
    float V[3][VEC], gV[3][VEC], gP[3][VEC], Pb[VEC];
    {
        const float *vs = vec + (size_t)s * F3 + ch;
        const hn::Vec<VEC> a = hn::ldv<VEC>(vs), b = hn::ldv<VEC>(vs + F), c = hn::ldv<VEC>(vs + 2 * F);
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            V[0][v] = a.v[v];
            V[1][v] = b.v[v];
            V[2][v] = c.v[v];
            gV[0][v] = gV[1][v] = gV[2][v] = 0.f;
            gP[0][v] = gP[1][v] = gP[2][v] = 0.f;
            Pb[v] = 0.f;
        }
    }
    long long cur_off = -1;     // element offset of the xh block the gP accumulators belong to (-1: none)
    auto flush = [&]() {
        if (cur_off < 0) return;
        float *dst = grad_xh + cur_off + (long long)s * F3 + ch;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            hn::Vec<VEC> o = hn::ldv<VEC>(dst + (size_t)k * F);
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                o.v[v] += gP[k][v];
                gP[k][v] = 0.f;
            }
            hn::stv<VEC>(dst + (size_t)k * F, o);
        }
    };
    const int q0 = __ldg(t_rowptr + s), q1 = __ldg(t_rowptr + s + 1);
    // index pipeline: stage A holds e of entry q+2, stage B (row, geometry) of entry q+1, stage C everything of entry q
    int eA = -1, rowB = -1, rowC = -1, mC = -1;
    float4 gB = make_float4(0.f, 0.f, 0.f, 0.f), gC = gB;
    long long offC = 0;
    if (q0 < q1) {
        const int e0 = __ldg(t_eid + q0);
        rowC = __ldg(edge_row + e0);
        gC = __ldg(geom + e0);
        mC = __ldg(row_mod + rowC);
        offC = __ldg(row_xoff + rowC);
        if (q0 + 1 < q1) {
            const int e1 = __ldg(t_eid + q0 + 1);
            rowB = __ldg(edge_row + e1);
            gB = __ldg(geom + e1);
        }
        if (q0 + 2 < q1) eA = __ldg(t_eid + q0 + 2);
    }
    for (int q = q0; q < q1; ++q) {
        // current entry, then advance the pipeline (loads only; nothing below waits for them before the next pass)
        const int row = rowC, m = mC;
        const float4 g = gC;
        const long long off = offC * F3;
        int mN = -1;
        long long offN = 0;
        if (q + 1 < q1) {
            mN = __ldg(row_mod + rowB);
            offN = __ldg(row_xoff + rowB);
        }
        const int rowN = rowB;
        const float4 gN = gB;
        if (q + 2 < q1) {
            rowB = __ldg(edge_row + eA);
            gB = __ldg(geom + eA);
        }
        if (q + 3 < q1) eA = __ldg(t_eid + q + 3);
        if (m >= 0 && (!MASKED || g.w >= 0.f)) {     // MASKED: a dead entry of a Verlet-skin list (g.w = -d) is skipped
            if (off != cur_off) {
                flush();
                cur_off = off;
                const hn::Vec<VEC> t = hn::ldv<VEC>(xh + off + (long long)s * F3 + F + ch);
#pragma unroll
                for (int v = 0; v < VEC; ++v) Pb[v] = t.v[v];
            }
            // gathered gradients of the destination row: in flight during the sweep
            const Pairs<NP> Gx = ldp<NP>(g_dx + (size_t)row * F + ch);
            const float *gvp = g_dvec + (size_t)row * F3 + ch;
            const Pairs<NP> G0 = ldp<NP>(gvp), G1 = ldp<NP>(gvp + F), G2 = ldp<NP>(gvp + 2 * F);
            const float *bm = bias + (size_t)m * F3 + ch;
            Pairs<NP> fa = ldp<NP>(bm), fb = ldp<NP>(bm + F), fc = ldp<NP>(bm + 2 * F);
            const float u = g.w * P.inv_rc;
            if (u < 1.f) {
                const int kc = (int)(u * (float)(K - 1));
                const int lo = max(kc - kLo, 0), hi = min(kc + kHi, K - 1);
                const int len = hi - lo + 1;
                if (lane < len) {
                    float env, denv;
                    envelope<false>(u, P.env_p, env, denv);
                    const float diff = u - __ldg(offset + lo + lane);
                    const float val = env * __expf(P.coeff * diff * diff);
                    *reinterpret_cast<float2 *>(tab + 2 * lane) = make_float2(val, val);
                }
                __syncwarp();
                const float *w = Wt + ((size_t)m * K + lo) * F3 + ch;
                unsigned t = tab_s;
                Pairs<NP> wa = ldp_ordered<NP>(w), wb = ldp_ordered<NP>(w + F), wc = ldp_ordered<NP>(w + 2 * F);
                u64 gg;
                asm volatile("ld.shared.u64 %0, [%1];" : "=l"(gg) : "r"(t));
#pragma unroll 1
                for (int i = 1; i <= len; ++i) {
                    if (i < len) {       // the last pass re-loads its own row (harmless, stays inside the matrix)
                        w += F3;
                        t += 8;
                    }
#pragma unroll
                    for (int n = 0; n < NP; ++n) fma2v(fa.p[n], gg, wa.p[n]);
                    wa = ldp_ordered<NP>(w);
#pragma unroll
                    for (int n = 0; n < NP; ++n) fma2v(fb.p[n], gg, wb.p[n]);
                    wb = ldp_ordered<NP>(w + F);
#pragma unroll
                    for (int n = 0; n < NP; ++n) fma2v(fc.p[n], gg, wc.p[n]);
                    wc = ldp_ordered<NP>(w + 2 * F);
                    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(gg) : "r"(t));
                }
                __syncwarp();    // table reads done before the next entry's fill
            }
#pragma unroll
            for (int n = 0; n < NP; ++n) {
                float gx[2], g0[2], g1[2], g2[2], pa[2], pb[2], pc[2];
                upk(Gx.p[n], gx[0], gx[1]);
                upk(G0.p[n], g0[0], g0[1]);
                upk(G1.p[n], g1[0], g1[1]);
                upk(G2.p[n], g2[0], g2[1]);
                upk(fa.p[n], pa[0], pa[1]);
                upk(fb.p[n], pb[0], pb[1]);
                upk(fc.p[n], pc[0], pc[1]);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int v = 2 * n + hh;
                    const float tb = (g0[hh] * V[0][v] + g1[hh] * V[1][v] + g2[hh] * V[2][v]) * c1;
                    const float tc = (g0[hh] * g.x + g1[hh] * g.y + g2[hh] * g.z) * c2;
                    gP[0][v] = fmaf(gx[hh], pa[hh], gP[0][v]);
                    gP[1][v] = fmaf(tb, pb[hh], gP[1][v]);
                    gP[2][v] = fmaf(tc, pc[hh], gP[2][v]);
                    const float bphi = Pb[v] * pb[hh] * c1;
                    gV[0][v] = fmaf(g0[hh], bphi, gV[0][v]);
                    gV[1][v] = fmaf(g1[hh], bphi, gV[1][v]);
                    gV[2][v] = fmaf(g2[hh], bphi, gV[2][v]);
                }
            }
        }
        rowC = rowN;
        gC = gN;
        mC = mN;
        offC = offN;
    }
    flush();
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        hn::Vec<VEC> o;
#pragma unroll
        for (int v = 0; v < VEC; ++v) o.v[v] = gV[k][v];
        hn::stv<VEC>(grad_vec + (size_t)s * F3 + (size_t)k * F + ch, o);
    }
}

}  // namespace

namespace hn {
namespace quad {

bool supported(const hn_edge_params *p) { return p->hidden == 64 || p->hidden == 128 || p->hidden == 256 || p->hidden == 512; }

int bwd_dst_slices(int hidden) { return hidden == 64 ? 1 : hidden / 128; }

// MASKED: flags bit 0 (Verlet-skin superset list, dead entries stored as -d in geom), a template argument so that the
// kernels of plain lists are the ones they were before masking existed
#define HN_QUAD_DISPATCH(KERNEL, MASKED, ...)                                                         \
    switch (p->hidden) {                                                                              \
        case 64: KERNEL<64, 1, MASKED><<<grid(1), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;      \
        case 128: KERNEL<128, 2, MASKED><<<grid(1), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;    \
        case 256: KERNEL<256, 2, MASKED><<<grid(2), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;    \
        default: KERNEL<512, 2, MASKED><<<grid(4), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;     \
    }
#define HN_QUAD_DISPATCH_HV(KERNEL, HV, MASKED, ...)                                                      \
    switch (p->hidden) {                                                                                  \
        case 64: KERNEL<64, 1, HV, MASKED><<<grid(1), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;      \
        case 128: KERNEL<128, 2, HV, MASKED><<<grid(1), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;    \
        case 256: KERNEL<256, 2, HV, MASKED><<<grid(2), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;    \
        default: KERNEL<512, 2, HV, MASKED><<<grid(4), 32 * kWarps, 0, stream>>>(__VA_ARGS__); break;     \
    }

int fwd(const hn_edge_params *p, const float *xh, const float *vec, const float *geom, const int32_t *rowptr,
        const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff, const float *Wt, const float *bias,
        const float *offset, float *dx, float *dvec, cudaStream_t stream) {
    auto grid = [&](int ns) { return (unsigned)(((long long)p->n_rows * ns + kWarps - 1) / kWarps); };
    dispatch_bool(p->flags & 1, [&](auto masked) {
        constexpr bool MASKED = decltype(masked)::value;
        if (vec != nullptr) {
            HN_QUAD_DISPATCH_HV(edge_fwd_quad_kernel, true, MASKED, *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod,
                                (const long long *)row_xoff, Wt, bias, offset, dx, dvec)
        } else {
            HN_QUAD_DISPATCH_HV(edge_fwd_quad_kernel, false, MASKED, *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod,
                                (const long long *)row_xoff, Wt, bias, offset, dx, dvec)
        }
    });
    return 0;
}

int bwd_dst(const hn_edge_params *p, const float *xh, const float *vec, const float *geom, const int32_t *rowptr,
            const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff, const float *Wt, const float *bias,
            const float *offset, const float *g_dx, const float *g_dvec, float *g_geom, int64_t n_edges, cudaStream_t stream) {
    auto grid = [&](int ns) { return (unsigned)(((long long)p->n_rows * ns + kWarps - 1) / kWarps); };
    dispatch_bool(p->flags & 1, [&](auto masked) {
        constexpr bool MASKED = decltype(masked)::value;
        if (vec != nullptr) {
            HN_QUAD_DISPATCH_HV(edge_bwd_dst_quad_kernel, true, MASKED, *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod,
                                (const long long *)row_xoff, Wt, bias, offset, g_dx, g_dvec, (float4 *)g_geom, (long long)n_edges)
        } else {
            HN_QUAD_DISPATCH_HV(edge_bwd_dst_quad_kernel, false, MASKED, *p, xh, vec, (const float4 *)geom, rowptr, col, row_mod,
                                (const long long *)row_xoff, Wt, bias, offset, g_dx, g_dvec, (float4 *)g_geom, (long long)n_edges)
        }
    });
    return 0;
}

int bwd_src(const hn_edge_params *p, const float *xh, const float *vec, const float *geom, const int32_t *t_rowptr,
            const int32_t *t_eid, const int32_t *edge_row, const int32_t *row_mod, const int64_t *row_xoff, const float *Wt,
            const float *bias, const float *offset, const float *g_dx, const float *g_dvec, float *grad_xh, float *grad_vec,
            cudaStream_t stream) {
    auto grid = [&](int ns) { return (unsigned)(((long long)p->n_atoms * ns + kWarps - 1) / kWarps); };
    dispatch_bool(p->flags & 1, [&](auto masked) {
        constexpr bool MASKED = decltype(masked)::value;
        HN_QUAD_DISPATCH(edge_bwd_src_sweep_kernel, MASKED, *p, xh, vec, (const float4 *)geom, t_rowptr, t_eid, edge_row, row_mod,
                         (const long long *)row_xoff, Wt, bias, offset, g_dx, g_dvec, grad_xh, grad_vec)
    });
    return 0;
}

}  // namespace quad
}  // namespace hn
