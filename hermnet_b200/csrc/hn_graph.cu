// Graph construction kernels: cell-list radius graph (periodic / non-periodic), stable sort-by-key
// (COO -> row CSR, CSR transpose), row expansion, triplet enumeration.
//
// Replaces HermNet/data.py:14-24 (ASE primitive_neighbor_list / torch_cluster radius_graph, both CPU in
// the reference) and the O(N*E) `torch.where` scans of HermNet/utils.py:11-24.
//
// HBM layout of the cell list (inside the caller's workspace): atoms are counting-sorted by bin with a
// stable radix sort, so a bin is a contiguous run of (float4 pos+index, int4 wrap+group) records and the
// traversal order -- hence the row order of the CSR -- is deterministic.
#include <cub/cub.cuh>

#include "hn_common.cuh"

namespace {

constexpr int kMaxGroups = 16;
constexpr int kMaxCap = 64;
constexpr double kSkin = 1.0 + 1e-6;  // bins are sized for rc*(1+1e-6) plus the fp32 bound below

struct GraphMeta {
    double cell[9];    // row vectors (periodic) or diag(extent) (non-periodic)
    double inv[9];     // inverse, frac_k = sum_r (p_r - origin_r) * inv[r*3+k]
    double origin[3];
    int nb[3];         // bins per axis
    int m[3];          // bins to search on each side
    int bin_offset;    // first global bin id of this graph
    int periodic;
    int atom_begin, atom_end;
};

struct Workspace {
    GraphMeta *meta;
    int *bin_start;    // [max_bins + 1] (histogram, then exclusive scan in place)
    int *atom_bin;     // [N]
    int *atom_bin_sorted;
    int *iota;
    int *sorted_atom;
    float4 *spos;      // [N] (x, y, z, bitcast atom index) in bin order
    int4 *swrap;       // [N] (wx, wy, wz, group) in bin order
    int4 *awrap;       // [N] unsorted
    int *agraph;       // [N] graph of atom (unsorted)
    int *sgraph;       // [N] graph of sorted atom
    void *cub_temp;
    size_t cub_bytes;
    int64_t max_bins;
    int64_t total;
};

size_t cub_temp_bytes(int64_t n, int64_t max_bins) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (int *)nullptr, (int *)nullptr, (int *)nullptr, (int *)nullptr,
                                    (int)n, 0, 32);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int *)nullptr, (int *)nullptr, (int)(max_bins + 1));
    return a > b ? a : b;
}

Workspace carve(void *base, int64_t n, int32_t n_graphs) {
    Workspace w;
    w.max_bins = 8 * (int64_t)n_graphs + 2 * n;
    char *p = (char *)base;
    auto take = [&](int64_t bytes) {
        char *q = p;
        p += hn::align_up(bytes, 256);
        return (void *)q;
    };
    w.meta = (GraphMeta *)take(sizeof(GraphMeta) * (int64_t)n_graphs);
    w.bin_start = (int *)take(4 * (w.max_bins + 2));
    w.atom_bin = (int *)take(4 * n);
    w.atom_bin_sorted = (int *)take(4 * n);
    w.iota = (int *)take(4 * n);
    w.sorted_atom = (int *)take(4 * n);
    w.spos = (float4 *)take(16 * n);
    w.swrap = (int4 *)take(16 * n);
    w.awrap = (int4 *)take(16 * n);
    w.agraph = (int *)take(4 * n);
    w.sgraph = (int *)take(4 * n);
    w.cub_bytes = cub_temp_bytes(n, w.max_bins);
    w.cub_temp = take((int64_t)w.cub_bytes);
    w.total = p - (char *)base;
    return w;
}

// ---------------------------------------------------------------------------------------------------
// per-graph setup: one block per graph
// ---------------------------------------------------------------------------------------------------
__device__ void invert3(const double *c, double *o, double &det) {
    det = c[0] * (c[4] * c[8] - c[5] * c[7]) - c[1] * (c[3] * c[8] - c[5] * c[6]) + c[2] * (c[3] * c[7] - c[4] * c[6]);
    double id = 1.0 / det;
    o[0] = (c[4] * c[8] - c[5] * c[7]) * id; o[1] = (c[2] * c[7] - c[1] * c[8]) * id; o[2] = (c[1] * c[5] - c[2] * c[4]) * id;
    o[3] = (c[5] * c[6] - c[3] * c[8]) * id; o[4] = (c[0] * c[8] - c[2] * c[6]) * id; o[5] = (c[2] * c[3] - c[0] * c[5]) * id;
    o[6] = (c[3] * c[7] - c[4] * c[6]) * id; o[7] = (c[1] * c[6] - c[0] * c[7]) * id; o[8] = (c[0] * c[4] - c[1] * c[3]) * id;
}

__global__ void graph_setup_kernel(const float *__restrict__ pos, const float *__restrict__ cell,
                                   const int *__restrict__ graph_ptr, int n_graphs, double rc, GraphMeta *meta) {
    const int g = blockIdx.x;
    const int a0 = graph_ptr[g], a1 = graph_ptr[g + 1];
    __shared__ float smin[3][128], smax[3][128];
    GraphMeta M;
    if (cell == nullptr) {
        float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
        for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x)
            for (int k = 0; k < 3; ++k) {
                float v = pos[3 * (size_t)a + k];
                lo[k] = fminf(lo[k], v);
                hi[k] = fmaxf(hi[k], v);
            }
        for (int k = 0; k < 3; ++k) { smin[k][threadIdx.x] = lo[k]; smax[k][threadIdx.x] = hi[k]; }
        __syncthreads();
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if (threadIdx.x < s)
                for (int k = 0; k < 3; ++k) {
                    smin[k][threadIdx.x] = fminf(smin[k][threadIdx.x], smin[k][threadIdx.x + s]);
                    smax[k][threadIdx.x] = fmaxf(smax[k][threadIdx.x], smax[k][threadIdx.x + s]);
                }
            __syncthreads();
        }
    } else {
        // largest |coordinate| of the graph: bounds the rounding of the periodic pair test below
        float big = 0.f;
        for (long long q = 3ll * a0 + threadIdx.x; q < 3ll * a1; q += blockDim.x) big = fmaxf(big, fabsf(pos[q]));
        smax[0][threadIdx.x] = big;
        __syncthreads();
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if (threadIdx.x < s) smax[0][threadIdx.x] = fmaxf(smax[0][threadIdx.x], smax[0][threadIdx.x + s]);
            __syncthreads();
        }
    }
    if (threadIdx.x != 0) return;
    // The periodic test subtracts the positions in fp32 (ASE): each component of pos_j - pos_i is off by up to 2^-24 of
    // itself, at most 2^-23 max|pos|, so a kept pair can lie up to sqrt(3) 2^-23 max|pos| beyond rc -- more than the
    // 1e-6 relative margin once |pos| reaches a few hundred A (large boxes, unwrapped trajectories).  The bins cover it.
    const double rcs = rc * kSkin + (cell != nullptr ? ldexp((double)smax[0][0], -22) : 0.0);
    const int n_atoms = a1 - a0;
    double h[3];
    if (cell != nullptr) {
        for (int k = 0; k < 9; ++k) M.cell[k] = (double)cell[9 * (size_t)g + k];
        double det;
        invert3(M.cell, M.inv, det);
        const double vol = fabs(det);
        for (int a = 0; a < 3; ++a) {
            const double *u = &M.cell[3 * ((a + 1) % 3)], *v = &M.cell[3 * ((a + 2) % 3)];
            double cx = u[1] * v[2] - u[2] * v[1], cy = u[2] * v[0] - u[0] * v[2], cz = u[0] * v[1] - u[1] * v[0];
            h[a] = vol / sqrt(cx * cx + cy * cy + cz * cz);
            M.origin[a] = 0.0;
        }
        M.periodic = 1;
    } else {
        for (int k = 0; k < 9; ++k) { M.cell[k] = 0.0; M.inv[k] = 0.0; }
        for (int a = 0; a < 3; ++a) {
            double lo = n_atoms > 0 ? (double)smin[a][0] : 0.0, hi = n_atoms > 0 ? (double)smax[a][0] : 1.0;
            double ext = fmax(hi - lo, 1e-3) * (1.0 + 1e-9) + 1e-6;
            M.cell[4 * a] = ext;
            M.inv[4 * a] = 1.0 / ext;
            M.origin[a] = lo - 5e-7;
            h[a] = ext;
        }
        M.periodic = 0;
    }
    double limit = fmax(8.0, 2.0 * (double)n_atoms);
    long long nb[3];
    for (int a = 0; a < 3; ++a) {
        double q = floor(h[a] / rcs);
        nb[a] = q < 1.0 ? 1 : (q > 1.0e6 ? 1000000 : (long long)q);
    }
    for (int it = 0; it < 64 && (double)nb[0] * (double)nb[1] * (double)nb[2] > limit; ++it) {
        double f = cbrt(limit / ((double)nb[0] * (double)nb[1] * (double)nb[2]));
        for (int a = 0; a < 3; ++a) {
            long long q = (long long)floor((double)nb[a] * f);
            nb[a] = q < 1 ? 1 : (q < nb[a] ? q : (nb[a] > 1 ? nb[a] - 1 : 1));
        }
    }
    for (int a = 0; a < 3; ++a) {
        M.nb[a] = (int)nb[a];
        double width = h[a] / (double)nb[a];
        int m = (int)ceil(rcs / width);
        M.m[a] = m < 1 ? 1 : m;
        if (!M.periodic && M.m[a] > M.nb[a]) M.m[a] = M.nb[a];
    }
    M.bin_offset = 0;
    M.atom_begin = a0;
    M.atom_end = a1;
    meta[g] = M;
}

__global__ void graph_scan_kernel(GraphMeta *meta, int n_graphs) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    int off = 0;
    for (int g = 0; g < n_graphs; ++g) {
        meta[g].bin_offset = off;
        off += meta[g].nb[0] * meta[g].nb[1] * meta[g].nb[2];
    }
}

__global__ void bin_atoms_kernel(const float *__restrict__ pos, int n, const int *__restrict__ graph_ptr, int n_graphs,
                                 const GraphMeta *__restrict__ meta, const int *__restrict__ group, int *atom_bin,
                                 int4 *awrap, int *agraph, int *iota, int *bin_count) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n) return;
    int lo = 0, hi = n_graphs;  // largest g with graph_ptr[g] <= a
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (graph_ptr[mid] <= a) lo = mid; else hi = mid;
    }
    const GraphMeta &M = meta[lo];
    double p[3];
    for (int k = 0; k < 3; ++k) p[k] = (double)pos[3 * (size_t)a + k] - M.origin[k];
    int w[3], b[3];
    for (int k = 0; k < 3; ++k) {
        double f = p[0] * M.inv[k] + p[1] * M.inv[3 + k] + p[2] * M.inv[6 + k];
        double fl = M.periodic ? floor(f) : 0.0;
        w[k] = (int)fl;
        f -= fl;
        int q = (int)(f * (double)M.nb[k]);
        b[k] = q < 0 ? 0 : (q >= M.nb[k] ? M.nb[k] - 1 : q);
    }
    const int bin = M.bin_offset + (b[0] * M.nb[1] + b[1]) * M.nb[2] + b[2];
    atom_bin[a] = bin;
    awrap[a] = make_int4(w[0], w[1], w[2], group ? group[a] : 0);
    agraph[a] = lo;
    iota[a] = a;
    atomicAdd(&bin_count[bin], 1);
}

__global__ void gather_sorted_kernel(const float *__restrict__ pos, int n, const int *__restrict__ sorted_atom,
                                     const int4 *__restrict__ awrap, const int *__restrict__ agraph, float4 *spos,
                                     int4 *swrap, int *sgraph) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int a = sorted_atom[p];
    spos[p] = make_float4(pos[3 * (size_t)a], pos[3 * (size_t)a + 1], pos[3 * (size_t)a + 2], __int_as_float(a));
    swrap[p] = awrap[a];
    sgraph[p] = agraph[a];
}

// ---------------------------------------------------------------------------------------------------
// neighbour traversal (shared by count and fill)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool pair_within_pbc(float3 pi, float3 pj, int S0, int S1, int S2, const double *c, double rc) {
    // ASE arithmetic: float32 difference, promoted; S.cell in float64; no FMA contraction.
    const float dx = __fsub_rn(pj.x, pi.x), dy = __fsub_rn(pj.y, pi.y), dz = __fsub_rn(pj.z, pi.z);
    const double s0 = (double)S0, s1 = (double)S1, s2 = (double)S2;
    const double ox = __dadd_rn(__dadd_rn(__dmul_rn(s0, c[0]), __dmul_rn(s1, c[3])), __dmul_rn(s2, c[6]));
    const double oy = __dadd_rn(__dadd_rn(__dmul_rn(s0, c[1]), __dmul_rn(s1, c[4])), __dmul_rn(s2, c[7]));
    const double oz = __dadd_rn(__dadd_rn(__dmul_rn(s0, c[2]), __dmul_rn(s1, c[5])), __dmul_rn(s2, c[8]));
    const double X = __dadd_rn((double)dx, ox), Y = __dadd_rn((double)dy, oy), Z = __dadd_rn((double)dz, oz);
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(X, X), __dmul_rn(Y, Y)), __dmul_rn(Z, Z));
    return __dsqrt_rn(d2) < rc;
}

__device__ __forceinline__ bool pair_within_open(float3 pi, float3 pj, float r2) {
    // torch_cluster arithmetic: float32 squared distance < r*r
    const float dx = __fsub_rn(pj.x, pi.x), dy = __fsub_rn(pj.y, pi.y), dz = __fsub_rn(pj.z, pi.z);
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    return d2 < r2;
}

__device__ __forceinline__ int floor_div(int a, int n) { return a >= 0 ? a / n : -((-a + n - 1) / n); }

template <typename Visit>
__device__ __forceinline__ void visit_neighbours(int p, const Workspace &w, double rc, Visit &&visit) {
    const float4 me = w.spos[p];
    const int4 mw = w.swrap[p];
    const int a = __float_as_int(me.w);
    const GraphMeta &M = w.meta[w.sgraph[p]];
    const float3 pi = make_float3(me.x, me.y, me.z);
    const int lb = w.atom_bin_sorted[p] - M.bin_offset;
    const int n0 = M.nb[0], n1 = M.nb[1], n2 = M.nb[2];
    const int b0 = lb / (n1 * n2), b1 = (lb / n2) % n1, b2 = lb % n2;
    const float rcf = (float)rc;
    const float r2 = __fmul_rn(rcf, rcf);
    const bool periodic = M.periodic != 0;
    for (int d0 = -M.m[0]; d0 <= M.m[0]; ++d0) {
        int c0 = b0 + d0, s0 = 0;
        if (periodic) { s0 = floor_div(c0, n0); c0 -= s0 * n0; } else if (c0 < 0 || c0 >= n0) continue;
        for (int d1 = -M.m[1]; d1 <= M.m[1]; ++d1) {
            int c1 = b1 + d1, s1 = 0;
            if (periodic) { s1 = floor_div(c1, n1); c1 -= s1 * n1; } else if (c1 < 0 || c1 >= n1) continue;
            for (int d2 = -M.m[2]; d2 <= M.m[2]; ++d2) {
                int c2 = b2 + d2, s2 = 0;
                if (periodic) { s2 = floor_div(c2, n2); c2 -= s2 * n2; } else if (c2 < 0 || c2 >= n2) continue;
                const int bin = M.bin_offset + (c0 * n1 + c1) * n2 + c2;
                const int q0 = w.bin_start[bin], q1 = w.bin_start[bin + 1];
                for (int q = q0; q < q1; ++q) {
                    const float4 o = w.spos[q];
                    const int j = __float_as_int(o.w);
                    const float3 pj = make_float3(o.x, o.y, o.z);
                    if (periodic) {
                        const int4 ow = w.swrap[q];
                        const int S0 = s0 - ow.x + mw.x, S1 = s1 - ow.y + mw.y, S2 = s2 - ow.z + mw.z;
                        if (j == a && S0 == 0 && S1 == 0 && S2 == 0) continue;
                        if (pair_within_pbc(pi, pj, S0, S1, S2, M.cell, rc)) visit(j, ow.w, S0, S1, S2);
                    } else {
                        if (j == a) continue;
                        if (pair_within_open(pi, pj, r2)) visit(j, w.swrap[q].w, 0, 0, 0);
                    }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(128) rg_count_kernel(Workspace w, int n, double rc, int n_groups, int cap, int *counts) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int cnt[kMaxGroups];
#pragma unroll
    for (int g = 0; g < kMaxGroups; ++g) cnt[g] = 0;
    visit_neighbours(p, w, rc, [&](int, int grp, int, int, int) { cnt[grp] += 1; });
    const int a = __float_as_int(w.spos[p].w);
    for (int g = 0; g < n_groups; ++g) {
        int c = cnt[g];
        if (cap > 0 && c > cap) c = cap;
        counts[(size_t)a * n_groups + g] = c;
    }
}

__global__ void __launch_bounds__(128) rg_fill_kernel(Workspace w, int n, double rc, int n_groups, int cap,
                                                       const int *__restrict__ rowptr, int *col, char4 *shift) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int a = __float_as_int(w.spos[p].w);
    if (cap > 0) {
        // capped rows keep the `cap` smallest neighbour indices, ascending (n_groups == 1 enforced by the host)
        const int r0 = rowptr[a], room = rowptr[a + 1] - r0;
        int best[kMaxCap];
        int have = 0;
        visit_neighbours(p, w, rc, [&](int j, int, int, int, int) {
            int pos = have;
            if (have == room) {
                if (room == 0 || j > best[room - 1]) return;
                pos = room - 1;
            } else {
                have += 1;
            }
            while (pos > 0 && best[pos - 1] > j) { best[pos] = best[pos - 1]; --pos; }
            best[pos] = j;
        });
        for (int q = 0; q < have; ++q) { col[r0 + q] = best[q]; shift[r0 + q] = make_char4(0, 0, 0, 0); }
        return;
    }
    int cur[kMaxGroups];
#pragma unroll
    for (int g = 0; g < kMaxGroups; ++g) cur[g] = 0;
    for (int g = 0; g < n_groups; ++g) cur[g] = rowptr[(size_t)a * n_groups + g];
    visit_neighbours(p, w, rc, [&](int j, int grp, int S0, int S1, int S2) {
        const int q = cur[grp]++;
        col[q] = j;
        shift[q] = make_char4((signed char)S0, (signed char)S1, (signed char)S2, 0);
    });
}

int build_cell_list(const float *pos, int64_t n, const float *cell, const int32_t *graph_ptr, int32_t n_graphs,
                    double rc, const int32_t *group, const Workspace &w, cudaStream_t st) {
    const char *where = "hn_radius_graph(cell list)";
    graph_setup_kernel<<<n_graphs, 128, 0, st>>>(pos, cell, graph_ptr, n_graphs, rc, w.meta);
    graph_scan_kernel<<<1, 32, 0, st>>>(w.meta, n_graphs);
    HN_CUDA(cudaMemsetAsync(w.bin_start, 0, 4 * (w.max_bins + 2), st), where);
    const int nb = (int)((n + 255) / 256);
    bin_atoms_kernel<<<nb, 256, 0, st>>>(pos, (int)n, graph_ptr, n_graphs, w.meta, group, w.atom_bin, w.awrap,
                                          w.agraph, w.iota, w.bin_start);
    size_t bytes = w.cub_bytes;
    HN_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, bytes, w.bin_start, w.bin_start, (int)(w.max_bins + 1), st), where);
    int end_bit = 1;
    while (end_bit < 31 && (1ll << end_bit) <= w.max_bins) ++end_bit;
    bytes = w.cub_bytes;
    HN_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, bytes, w.atom_bin, w.atom_bin_sorted, w.iota, w.sorted_atom,
                                            (int)n, 0, end_bit, st), where);
    gather_sorted_kernel<<<nb, 256, 0, st>>>(pos, (int)n, w.sorted_atom, w.awrap, w.agraph, w.spos, w.swrap, w.sgraph);
    return hn::check_launch(where);
}

int rg_validate(const char *where, int64_t n, int32_t n_graphs, int32_t n_groups, int32_t cap, const float *cell,
                const Workspace &w, int64_t workspace_bytes) {
    HN_REQUIRE(n > 0 && n < (1ll << 30), where, "n_atoms out of range");
    HN_REQUIRE(n_graphs > 0, where, "n_graphs must be positive");
    HN_REQUIRE(n_groups >= 1 && n_groups <= kMaxGroups, where, "n_groups must be in [1,16]");
    HN_REQUIRE(cap <= kMaxCap, where, "max_neighbors must be <= 64");
    HN_REQUIRE(!(cap > 0 && n_groups != 1), where, "max_neighbors requires n_groups == 1");
    HN_REQUIRE(!(cap > 0 && cell != nullptr), where, "max_neighbors is only defined for the non-periodic branch");
    HN_REQUIRE(workspace_bytes >= w.total, where, "workspace too small");
    return 0;
}

}  // namespace

extern "C" int64_t hn_radius_graph_workspace_bytes(int64_t n_atoms, int32_t n_graphs) {
    if (n_atoms <= 0 || n_graphs <= 0) return 256;
    return carve(nullptr, n_atoms, n_graphs).total;
}

extern "C" int hn_radius_graph_count(const float *pos, int64_t n_atoms, const float *cell, const int32_t *graph_ptr,
                                     int32_t n_graphs, double rc, const int32_t *group, int32_t n_groups,
                                     int32_t max_neighbors, int32_t *counts, void *workspace, int64_t workspace_bytes,
                                     void *stream) {
    const char *where = "hn_radius_graph_count";
    Workspace w = carve(workspace, n_atoms, n_graphs);
    if (int rc_ = rg_validate(where, n_atoms, n_graphs, n_groups, max_neighbors, cell, w, workspace_bytes)) return rc_;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc_ = build_cell_list(pos, n_atoms, cell, graph_ptr, n_graphs, rc, group, w, st)) return rc_;
    rg_count_kernel<<<(int)((n_atoms + 127) / 128), 128, 0, st>>>(w, (int)n_atoms, rc, n_groups, max_neighbors, counts);
    return hn::check_launch(where);
}

extern "C" int hn_radius_graph_fill(const float *pos, int64_t n_atoms, const float *cell, const int32_t *graph_ptr,
                                    int32_t n_graphs, double rc, const int32_t *group, int32_t n_groups,
                                    int32_t max_neighbors, const int32_t *rowptr, int32_t *col, int8_t *shift,
                                    void *workspace, int64_t workspace_bytes, void *stream) {
    const char *where = "hn_radius_graph_fill";
    (void)pos; (void)graph_ptr; (void)group;
    Workspace w = carve(workspace, n_atoms, n_graphs);
    if (int rc_ = rg_validate(where, n_atoms, n_graphs, n_groups, max_neighbors, cell, w, workspace_bytes)) return rc_;
    cudaStream_t st = (cudaStream_t)stream;
    rg_fill_kernel<<<(int)((n_atoms + 127) / 128), 128, 0, st>>>(w, (int)n_atoms, rc, n_groups, max_neighbors, rowptr,
                                                                 col, (char4 *)shift);
    return hn::check_launch(where);
}

// ---------------------------------------------------------------------------------------------------
// stable sort by key -> CSR
// ---------------------------------------------------------------------------------------------------
namespace {

struct SortWs {
    int *keys_out, *iota, *count;
    void *cub_temp;
    size_t cub_bytes;
    int64_t total;
};

SortWs carve_sort(void *base, int64_t n, int32_t n_keys) {
    SortWs w;
    char *p = (char *)base;
    auto take = [&](int64_t bytes) { char *q = p; p += hn::align_up(bytes, 256); return (void *)q; };
    w.keys_out = (int *)take(4 * n);
    w.iota = (int *)take(4 * n);
    w.count = (int *)take(4 * ((int64_t)n_keys + 2));
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (int *)nullptr, (int *)nullptr, (int *)nullptr, (int *)nullptr, (int)n, 0, 32);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int *)nullptr, (int *)nullptr, n_keys + 1);
    w.cub_bytes = a > b ? a : b;
    w.cub_temp = take((int64_t)w.cub_bytes);
    w.total = p - (char *)base;
    return w;
}

// Histogram of the keys (+ the identity permutation the radix sort carries along).  One global atomic per ITEM
// serialises on hot counters (256 distance bins for 3.6e7 edges took 4 ms per call), so:
//   few keys  -> per-CTA histogram in shared memory, flushed once per CTA;
//   many keys -> lanes of a warp holding the same key are merged with __match_any_sync before the global atomic.
constexpr int kHistItems = 16;          // items per thread of the shared-memory variant
constexpr int kHistSmallKeys = 8192;

__global__ void __launch_bounds__(256)
key_hist_small_kernel(const int *__restrict__ keys, int64_t n, int n_keys, int *iota, int *count) {
    extern __shared__ int s_hist[];
    for (int k = threadIdx.x; k < n_keys; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * (blockDim.x * kHistItems);
#pragma unroll 4
    for (int j = 0; j < kHistItems; ++j) {
        const int64_t i = base + (int64_t)j * blockDim.x + threadIdx.x;
        if (i < n) {
            iota[i] = (int)i;
            atomicAdd(&s_hist[keys[i]], 1);
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < n_keys; k += blockDim.x) {
        const int c = s_hist[k];
        if (c != 0) atomicAdd(&count[k], c);
    }
}

__global__ void key_hist_kernel(const int *__restrict__ keys, int64_t n, int *iota, int *count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;
    const int key = live ? keys[i] : -1;
    if (live) iota[i] = (int)i;
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (live && (__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&count[key], __popc(peers));
}

__global__ void expand_rowptr_kernel(const int *__restrict__ rowptr, int n_rows, int *edge_row) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int e1 = rowptr[r + 1];
    for (int e = rowptr[r]; e < e1; ++e) edge_row[e] = r;
}

}  // namespace

extern "C" int64_t hn_sort_by_key_workspace_bytes(int64_t n, int32_t n_keys) {
    return carve_sort(nullptr, n < 1 ? 1 : n, n_keys < 1 ? 1 : n_keys).total;
}

extern "C" int hn_sort_by_key(const int32_t *keys, int64_t n, int32_t n_keys, int32_t *rowptr, int32_t *order,
                              void *workspace, int64_t workspace_bytes, void *stream) {
    const char *where = "hn_sort_by_key";
    HN_REQUIRE(n >= 0 && n < (1ll << 31) - 1, where, "n out of range");
    HN_REQUIRE(n_keys >= 1, where, "n_keys must be >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    SortWs w = carve_sort(workspace, n < 1 ? 1 : n, n_keys);
    HN_REQUIRE(workspace_bytes >= w.total, where, "workspace too small");
    HN_CUDA(cudaMemsetAsync(w.count, 0, 4 * ((int64_t)n_keys + 2), st), where);
    if (n > 0) {
        if (n_keys <= kHistSmallKeys) {
            const int64_t per_cta = 256 * kHistItems;
            key_hist_small_kernel<<<(int)((n + per_cta - 1) / per_cta), 256, (size_t)n_keys * sizeof(int), st>>>(keys, n, n_keys,
                                                                                                                 w.iota, w.count);
        } else {
            key_hist_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(keys, n, w.iota, w.count);
        }
    }
    size_t bytes = w.cub_bytes;
    HN_CUDA(cub::DeviceScan::ExclusiveSum(w.cub_temp, bytes, w.count, rowptr, n_keys + 1, st), where);
    if (n > 0) {
        int end_bit = 1;
        while (end_bit < 31 && (1ll << end_bit) < (long long)n_keys) ++end_bit;
        bytes = w.cub_bytes;
        HN_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, bytes, keys, w.keys_out, w.iota, order, (int)n, 0, end_bit, st),
                where);
    }
    return hn::check_launch(where);
}

extern "C" int hn_expand_rowptr(const int32_t *rowptr, int32_t n_rows, int32_t *edge_row, void *stream) {
    if (n_rows <= 0) return 0;
    expand_rowptr_kernel<<<(n_rows + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rowptr, n_rows, edge_row);
    return hn::check_launch("hn_expand_rowptr");
}

// ---------------------------------------------------------------------------------------------------
// triplets
// ---------------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ bool type_ok(const int *src_type, const int *col, int e, int want) {
    return src_type == nullptr || want < 0 || src_type[col[e]] == want;
}

__global__ void triplets_count_kernel(const int *__restrict__ rowptr, int n_rows, const int *__restrict__ col,
                                      const int *__restrict__ src_type, int ta, int tc, long long *counts) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int e0 = rowptr[r], e1 = rowptr[r + 1];
    long long na = 0, nc = 0, both = 0;
    for (int e = e0; e < e1; ++e) {
        const bool a = type_ok(src_type, col, e, ta), c = type_ok(src_type, col, e, tc);
        na += a; nc += c; both += (a && c);
    }
    counts[r] = na * nc - both;  // ordered pairs (e1 in A, e2 in C) minus e1 == e2
}

__global__ void triplets_fill_kernel(const int *__restrict__ rowptr, int n_rows, const int *__restrict__ col,
                                     const int *__restrict__ src_type, int ta, int tc,
                                     const long long *__restrict__ trip_ptr, int *out1, int *out2) {
    // one warp per row; lanes stride over e2 for each e1 so the output stays sorted by (row, e1, e2)
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int e0 = rowptr[r], e1 = rowptr[r + 1];
    long long base = trip_ptr[r];
    for (int a = e0; a < e1; ++a) {
        if (!type_ok(src_type, col, a, ta)) continue;
        for (int b0 = e0; b0 < e1; b0 += 32) {
            const int b = b0 + lane;
            const bool ok = b < e1 && b != a && type_ok(src_type, col, b, tc);
            const unsigned mask = __ballot_sync(0xffffffffu, ok);
            if (ok) {
                const long long q = base + __popc(mask & ((1u << lane) - 1u));
                out1[q] = a;
                out2[q] = b;
            }
            base += __popc(mask);
        }
    }
}

__global__ void triplet_dots_kernel(const float *__restrict__ m_vec, int F, const long long *__restrict__ trip_ptr,
                                    const int *__restrict__ t1, const int *__restrict__ t2, int n_rows, float *dots) {
    const int r = blockIdx.x;
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        float acc = 0.f;
        for (long long q = trip_ptr[r]; q < trip_ptr[r + 1]; ++q) {
            const float *a = m_vec + (size_t)t1[q] * 3 * F, *b = m_vec + (size_t)t2[q] * 3 * F;
            acc += a[f] * b[f] + a[F + f] * b[F + f] + a[2 * F + f] * b[2 * F + f];
        }
        dots[(size_t)r * F + f] = acc;
    }
}

}  // namespace

extern "C" int hn_triplets_count(const int32_t *rowptr, int32_t n_rows, const int32_t *col, const int32_t *src_type,
                                 int32_t type_a, int32_t type_c, int64_t *counts, void *stream) {
    if (n_rows <= 0) return 0;
    triplets_count_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rowptr, n_rows, col, src_type, type_a,
                                                                                  type_c, (long long *)counts);
    return hn::check_launch("hn_triplets_count");
}

extern "C" int hn_triplets_fill(const int32_t *rowptr, int32_t n_rows, const int32_t *col, const int32_t *src_type,
                                int32_t type_a, int32_t type_c, const int64_t *trip_ptr, int32_t *e1, int32_t *e2,
                                void *stream) {
    if (n_rows <= 0) return 0;
    const int warps_per_block = 4;
    triplets_fill_kernel<<<(n_rows + warps_per_block - 1) / warps_per_block, 32 * warps_per_block, 0,
                           (cudaStream_t)stream>>>(rowptr, n_rows, col, src_type, type_a, type_c,
                                                   (const long long *)trip_ptr, e1, e2);
    return hn::check_launch("hn_triplets_fill");
}

extern "C" int hn_triplet_dots(const float *m_vec, int32_t F, const int64_t *trip_ptr, const int32_t *e1, const int32_t *e2,
                               int32_t n_rows, float *dots, void *stream) {
    if (n_rows <= 0) return 0;
    triplet_dots_kernel<<<n_rows, 128, 0, (cudaStream_t)stream>>>(m_vec, F, (const long long *)trip_ptr, e1, e2, n_rows, dots);
    return hn::check_launch("hn_triplet_dots");
}
