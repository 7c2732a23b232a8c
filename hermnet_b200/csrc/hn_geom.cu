// Edge geometry (forward / backward-to-positions-and-cell) and the gather / segmented-sum primitives.
//
// Replaces HVNet.with_edge (HermNet/hermnet.py:133-152) and, in backward, the autograd chain
// norm -> div -> index_select^T (index_add with atomics) that torch would run.
// HBM layout: geom[e] is one float4 (ux, uy, uz, d) so the edge kernels fetch the whole edge geometry
// with a single 16-byte load.
#include "hn_common.cuh"

namespace {

__global__ void edge_geom_fwd_kernel(const float *__restrict__ pos, const float *__restrict__ cell,
                                     const int *__restrict__ atom_graph, const int *__restrict__ edge_row,
                                     int rows_per_atom, const int *__restrict__ col, const char4 *__restrict__ shift,
                                     float sign, long long n_edges, float4 *__restrict__ geom) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int s = col[e];
    const int r = edge_row[e] / rows_per_atom;
    float dx = pos[3 * (size_t)s] - pos[3 * (size_t)r];
    float dy = pos[3 * (size_t)s + 1] - pos[3 * (size_t)r + 1];
    float dz = pos[3 * (size_t)s + 2] - pos[3 * (size_t)r + 2];
    if (cell != nullptr && shift != nullptr) {
        const char4 S = shift[e];
        if (S.x | S.y | S.z) {
            const float *c = cell + 9 * (size_t)atom_graph[s];
            const float s0 = sign * (float)S.x, s1 = sign * (float)S.y, s2 = sign * (float)S.z;
            dx += s0 * c[0] + s1 * c[3] + s2 * c[6];
            dy += s0 * c[1] + s1 * c[4] + s2 * c[7];
            dz += s0 * c[2] + s1 * c[5] + s2 * c[8];
        }
    }
    float d = sqrtf(dx * dx + dy * dy + dz * dz);
    if (d <= 1.0e-6f) d = 1.0e-6f;  // torch.isclose(d, 0, atol=1e-6) -> 1e-6  (hermnet.py:146-147)
    const float inv = 1.0f / d;
    geom[e] = make_float4(dx * inv, dy * inv, dz * inv, d);
}

// dL/dD of one row-edge from (u, d) and the summed per-part (dL/du, dL/dd)
__device__ __forceinline__ float3 edge_grad_D(const float4 *__restrict__ geom, const float4 *__restrict__ g_geom,
                                              int n_parts, long long n_edges, long long e) {
    const float4 g = __ldg(geom + e);
    float4 t = __ldg(g_geom + e);
    for (int p = 1; p < n_parts; ++p) {
        const float4 q = __ldg(g_geom + (size_t)p * n_edges + e);
        t.x += q.x; t.y += q.y; t.z += q.z; t.w += q.w;
    }
    const float inv = 1.0f / g.w;
    if (g.w == 1.0e-6f)  // clamped: d is a constant, u = D * 1e6
        return make_float3(t.x * inv, t.y * inv, t.z * inv);
    const float dot = t.x * g.x + t.y * g.y + t.z * g.z;
    return make_float3(t.w * g.x + (t.x - dot * g.x) * inv, t.w * g.y + (t.y - dot * g.y) * inv,
                       t.w * g.z + (t.z - dot * g.z) * inv);
}

__global__ void edge_geom_bwd_kernel(const float4 *__restrict__ geom, const float4 *__restrict__ g_geom, int n_parts,
                                     const char4 *__restrict__ shift, const int *__restrict__ rowptr, int rows_per_atom,
                                     const int *__restrict__ t_rowptr, const int *__restrict__ t_eid, float sign,
                                     int n_atoms, long long n_edges, float *__restrict__ grad_pos,
                                     float *__restrict__ cellw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    float ax = 0.f, ay = 0.f, az = 0.f;
    float w[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w[k] = 0.f;
    // destination side: D = pos[src] - pos[dst] + ...  ->  -dL/dD
    const int e0 = rowptr[(size_t)i * rows_per_atom], e1 = rowptr[(size_t)(i + 1) * rows_per_atom];
    for (int e = e0; e < e1; ++e) {
        const float3 gD = edge_grad_D(geom, g_geom, n_parts, n_edges, e);
        ax -= gD.x; ay -= gD.y; az -= gD.z;
        if (cellw != nullptr && shift != nullptr) {
            const char4 S = shift[e];
            if (S.x | S.y | S.z) {
                const float s[3] = {sign * (float)S.x, sign * (float)S.y, sign * (float)S.z};
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    w[3 * a] += s[a] * gD.x; w[3 * a + 1] += s[a] * gD.y; w[3 * a + 2] += s[a] * gD.z;
                }
            }
        }
    }
    // source side (transposed view): +dL/dD
    const int q0 = t_rowptr[i], q1 = t_rowptr[i + 1];
    for (int q = q0; q < q1; ++q) {
        const float3 gD = edge_grad_D(geom, g_geom, n_parts, n_edges, t_eid[q]);
        ax += gD.x; ay += gD.y; az += gD.z;
    }
    grad_pos[3 * (size_t)i] = ax; grad_pos[3 * (size_t)i + 1] = ay; grad_pos[3 * (size_t)i + 2] = az;
    if (cellw != nullptr) {
#pragma unroll
        for (int k = 0; k < 9; ++k) cellw[9 * (size_t)i + k] = w[k];
    }
}

// per-atom virial: every row-edge e gives -1/2 D_e (x) gD_e to each endpoint, D_e = d * u (clamped edges too).  Same
// traversal as edge_geom_bwd_kernel (row CSR, then its transpose), so the summation order is fixed
__global__ void edge_virial_atom_kernel(const float4 *__restrict__ geom, const float4 *__restrict__ g_geom,
                                        const int *__restrict__ rowptr, int rows_per_atom, const int *__restrict__ t_rowptr,
                                        const int *__restrict__ t_eid, int n_atoms, long long n_edges,
                                        float *__restrict__ virial) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    float w[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w[k] = 0.f;
    auto add = [&](long long e) {
        const float4 g = __ldg(geom + e);
        const float3 gD = edge_grad_D(geom, g_geom, 1, n_edges, e);
        const float D[3] = {g.w * g.x, g.w * g.y, g.w * g.z};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            w[3 * a] += D[a] * gD.x; w[3 * a + 1] += D[a] * gD.y; w[3 * a + 2] += D[a] * gD.z;
        }
    };
    const int e0 = rowptr[(size_t)i * rows_per_atom], e1 = rowptr[(size_t)(i + 1) * rows_per_atom];
    for (int e = e0; e < e1; ++e) add(e);
    const int q0 = t_rowptr[i], q1 = t_rowptr[i + 1];
    for (int q = q0; q < q1; ++q) add(t_eid[q]);
#pragma unroll
    for (int k = 0; k < 9; ++k) virial[9 * (size_t)i + k] = -0.5f * w[k];
}

__global__ void gather_rows_kernel(const float *__restrict__ X, const int *__restrict__ idx, long long total, int C,
                                   float *__restrict__ out) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += stride) {
        const long long e = t / C;
        const int c = (int)(t - e * C);
        out[t] = __ldg(X + (size_t)idx[e] * C + c);
    }
}

__global__ void gather_rows4_kernel(const float4 *__restrict__ X, const int *__restrict__ idx, long long total, int C4,
                                    float4 *__restrict__ out) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += stride) {
        const long long e = t / C4;
        const int c = (int)(t - e * C4);
        out[t] = __ldg(X + (size_t)idx[e] * C4 + c);
    }
}

// short rows: one thread per (row, column); consecutive threads = consecutive columns (coalesced)
__global__ void segment_sum_kernel(const float *__restrict__ Y, const int *__restrict__ rowptr, const int *__restrict__ perm,
                                   long long total, int C, float *__restrict__ out) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += stride) {
        const long long r = t / C;
        const int c = (int)(t - r * C);
        float acc = 0.f;
        const int q1 = rowptr[r + 1];
        for (int q = rowptr[r]; q < q1; ++q) {
            const int e = perm ? perm[q] : q;
            acc += __ldg(Y + (size_t)e * C + c);
        }
        out[t] = acc;
    }
}

// long rows (few segments, e.g. per-graph energy): every (row, column) is split over `chunks` blocks that each reduce a
// contiguous chunk with a fixed-shape tree in double precision; a second kernel adds the chunk partials in order
// (deterministic; a single block per row took 3.2 ms for the 1M-atom energy sum)
__global__ void segment_sum_long_kernel(const float *__restrict__ Y, const int *__restrict__ rowptr,
                                        const int *__restrict__ perm, int C, int chunks, double *__restrict__ partial) {
    const int r = blockIdx.x, c = blockIdx.y, z = blockIdx.z;
    __shared__ double part[256];
    double acc = 0.0;
    const long long q0 = rowptr[r], q1 = rowptr[r + 1];
    const long long per = (q1 - q0 + chunks - 1) / chunks;
    const long long a = q0 + (long long)z * per, b = (a + per < q1) ? a + per : q1;
    for (long long q = a + threadIdx.x; q < b; q += blockDim.x) {
        const int e = perm ? perm[q] : (int)q;
        acc += (double)__ldg(Y + (size_t)e * C + c);
    }
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[((size_t)r * C + c) * chunks + z] = part[0];
}

__global__ void segment_sum_finish_kernel(const double *__restrict__ partial, int total, int chunks, float *__restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    double acc = 0.0;
    for (int z = 0; z < chunks; ++z) acc += partial[(size_t)t * chunks + z];
    out[t] = (float)acc;
}

}  // namespace

extern "C" int hn_edge_geom_fwd(const float *pos, const float *cell, const int32_t *atom_graph, const int32_t *edge_row,
                                int32_t rows_per_atom, const int32_t *col, const int8_t *shift, float sign, int64_t n_edges,
                                float *geom, void *stream) {
    if (n_edges <= 0) return 0;
    HN_REQUIRE(rows_per_atom >= 1, "hn_edge_geom_fwd", "rows_per_atom must be >= 1");
    edge_geom_fwd_kernel<<<(unsigned)((n_edges + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        pos, cell, atom_graph, edge_row, rows_per_atom, col, (const char4 *)shift, sign, n_edges, (float4 *)geom);
    return hn::check_launch("hn_edge_geom_fwd");
}

extern "C" int hn_edge_geom_bwd(const float *geom, const float *g_geom, int32_t n_parts, const int8_t *shift,
                                const int32_t *rowptr, int32_t rows_per_atom, const int32_t *t_rowptr, const int32_t *t_eid,
                                float sign, int64_t n_atoms, int64_t n_edges, float *grad_pos, float *cellw, void *stream) {
    if (n_atoms <= 0) return 0;
    HN_REQUIRE(n_parts >= 1, "hn_edge_geom_bwd", "n_parts must be >= 1");
    edge_geom_bwd_kernel<<<(unsigned)((n_atoms + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        (const float4 *)geom, (const float4 *)g_geom, n_parts, (const char4 *)shift, rowptr, rows_per_atom, t_rowptr, t_eid,
        sign, (int)n_atoms, n_edges, grad_pos, cellw);
    return hn::check_launch("hn_edge_geom_bwd");
}

extern "C" int hn_edge_virial_atom(const float *geom, const float *g_geom, const int32_t *rowptr, int32_t rows_per_atom,
                                   const int32_t *t_rowptr, const int32_t *t_eid, int64_t n_atoms, int64_t n_edges,
                                   float *virial, void *stream) {
    if (n_atoms <= 0) return 0;
    HN_REQUIRE(rows_per_atom >= 1, "hn_edge_virial_atom", "rows_per_atom must be >= 1");
    edge_virial_atom_kernel<<<(unsigned)((n_atoms + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        (const float4 *)geom, (const float4 *)g_geom, rowptr, rows_per_atom, t_rowptr, t_eid, (int)n_atoms, n_edges, virial);
    return hn::check_launch("hn_edge_virial_atom");
}

extern "C" int hn_gather_rows(const float *X, const int32_t *idx, int64_t n_out, int32_t C, float *out, void *stream) {
    if (n_out <= 0 || C <= 0) return 0;
    const int sms = hn::num_sms() > 0 ? hn::num_sms() : 148;
    const bool v4 = (C % 4 == 0) && (((uintptr_t)X | (uintptr_t)out) % 16 == 0);
    const long long total = v4 ? n_out * (C / 4) : n_out * (long long)C;
    long long blocks = (total + 255) / 256;
    if (blocks > (long long)sms * 32) blocks = (long long)sms * 32;
    if (v4)
        gather_rows4_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const float4 *)X, idx, total, C / 4,
                                                                               (float4 *)out);
    else
        gather_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(X, idx, total, C, out);
    return hn::check_launch("hn_gather_rows");
}

namespace {
// chunks of the long-row path (few, possibly very long segments); 0: the short-row kernel needs no workspace
int segment_sum_chunks(int32_t n_rows, int32_t C) {
    if (!((long long)n_rows * C <= 4096 && C <= 64)) return 0;
    const int sms = hn::num_sms() > 0 ? hn::num_sms() : 148;
    const int total = n_rows * C;
    int chunks = (sms * 4 + total - 1) / total;
    return chunks < 1 ? 1 : (chunks > 256 ? 256 : chunks);
}
}  // namespace

extern "C" int64_t hn_segment_sum_workspace_bytes(int32_t n_rows, int32_t C) {
    if (n_rows <= 0 || C <= 0) return 0;
    return (int64_t)sizeof(double) * n_rows * C * segment_sum_chunks(n_rows, C);
}

extern "C" int hn_segment_sum(const float *Y, const int32_t *rowptr, const int32_t *perm, int32_t n_rows, int32_t C,
                              float *out, void *workspace, int64_t workspace_bytes, void *stream) {
    if (n_rows <= 0 || C <= 0) return 0;
    const int sms = hn::num_sms() > 0 ? hn::num_sms() : 148;
    const int chunks = segment_sum_chunks(n_rows, C);
    if (chunks > 0) {  // few, possibly very long segments: chunk partials in the CALLER's workspace (no library state)
        const int total = n_rows * C;
        HN_REQUIRE(workspace != nullptr && workspace_bytes >= hn_segment_sum_workspace_bytes(n_rows, C), "hn_segment_sum",
                   "workspace too small (hn_segment_sum_workspace_bytes)");
        double *partial = (double *)workspace;
        dim3 grid(n_rows, C, chunks);
        segment_sum_long_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(Y, rowptr, perm, C, chunks, partial);
        segment_sum_finish_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(partial, total, chunks, out);
    } else {
        const long long total = (long long)n_rows * C;
        long long blocks = (total + 255) / 256;
        if (blocks > (long long)sms * 32) blocks = (long long)sms * 32;
        segment_sum_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(Y, rowptr, perm, total, C, out);
    }
    return hn::check_launch("hn_segment_sum");
}
