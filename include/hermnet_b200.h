/* hermnet_b200 -- C ABI of the B200-native HermNet message-passing hot path.
 *
 * The reference (thu-wangz17/HermNet) has no FFI: its hot path is a chain of implicit PyTorch /
 * PyG / torch_scatter / torch_cluster / ASE library calls.  Each entry point below names the
 * reference call site(s) it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  Every pointer is a DEVICE pointer on the
 *     current CUDA device unless stated otherwise; the caller owns every buffer (outputs, scratch).
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises.
 *   - return value: 0 = ok, non-zero = error; `hn_last_error()` gives a thread-local message.
 *   - variable-size outputs use two phases (count -> caller scans/allocates -> fill).
 *   - indices are int32 (E < 2^31); triplet offsets are int64.
 *   - float data is fp32; the neighbour test runs in fp64 (see hn_radius_graph_*).
 *
 * Graph layout ("row CSR")
 *   A *row* is one segment of the segmented reduction: (destination atom [, module slot]).
 *   rows_per_atom is constant: row r belongs to atom r / rows_per_atom.
 *     rowptr[R+1], col[E] (source atom of each row-edge), shift[E][4] (int8 Sx,Sy,Sz,0),
 *     row_mod[R] (module / weight-set id of the row, -1 = inactive row).
 *   The transposed view (grouped by source atom) is t_rowptr[N+1], t_eid[E] (row-edge ids),
 *   edge_row[E] (row of each row-edge).
 */
#ifndef HERMNET_B200_H
#define HERMNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HN_ABI_VERSION 2

int hn_abi_version(void);
const char *hn_last_error(void);
/* number of SMs of the current device (grid sizing), <0 on error */
int hn_device_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * Radius graph: cell-list neighbour search producing a centre-sorted CSR.
 * Replaces HermNet/data.py:14-24 `neighbor_search` = ase.neighborlist.primitive_neighbor_list
 * (periodic, data.py:19-21) / torch_cluster radius_graph (non-periodic, data.py:16).
 *
 * Row c*n_groups+g lists every (j, S) with group[j]==g and
 *     || pos_j - pos_c + S.cell || < rc ,  not (j==c and S==0)
 * evaluated as  sqrt(sum((double)(float)(pos_j-pos_c) + S.cell)^2) < rc  in fp64, un-fused
 * (the ASE arithmetic).  cell==NULL: non-periodic, fp32 test d2 < rc*rc, S==0, and at most
 * max_neighbors (>0) neighbours per centre, the smallest indices (torch_cluster CUDA semantics).
 * Positions need not lie inside the cell.  Atoms of a graph are contiguous: graph_ptr[B+1].
 * `workspace` (hn_radius_graph_workspace_bytes) carries the cell list from count to fill.
 * Entry order inside a row is deterministic (cell-traversal order).
 * ------------------------------------------------------------------------------------------- */
int64_t hn_radius_graph_workspace_bytes(int64_t n_atoms, int32_t n_graphs);
int hn_radius_graph_count(const float *pos, int64_t n_atoms, const float *cell /*[B,3,3] or NULL*/,
                          const int32_t *graph_ptr, int32_t n_graphs, double rc,
                          const int32_t *group /*[N] or NULL*/, int32_t n_groups, int32_t max_neighbors,
                          int32_t *counts /*[N*n_groups]*/, void *workspace, int64_t workspace_bytes,
                          void *stream);
int hn_radius_graph_fill(const float *pos, int64_t n_atoms, const float *cell, const int32_t *graph_ptr,
                         int32_t n_graphs, double rc, const int32_t *group, int32_t n_groups,
                         int32_t max_neighbors, const int32_t *rowptr /*[N*n_groups+1]*/,
                         int32_t *col /*[E]*/, int8_t *shift /*[E,4]*/, void *workspace,
                         int64_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Stable counting sort of edge ids by an integer key: order[] lists ids grouped by key ascending,
 * original order inside a key; rowptr[n_keys+1].  Used for (a) COO -> row CSR of a user-supplied
 * edge_index (replaces the per-atom `torch.where` scans of HermNet/utils.py:11-24 `in_subgraph`),
 * (b) the transposed (source-major) view needed by the backward pass.
 * ------------------------------------------------------------------------------------------- */
int64_t hn_sort_by_key_workspace_bytes(int64_t n, int32_t n_keys);
int hn_sort_by_key(const int32_t *keys, int64_t n, int32_t n_keys, int32_t *rowptr, int32_t *order,
                   void *workspace, int64_t workspace_bytes, void *stream);
/* edge_row[e] = r for rowptr[r] <= e < rowptr[r+1] */
int hn_expand_rowptr(const int32_t *rowptr, int32_t n_rows, int32_t *edge_row, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Canonical ordered triplets (j,i,k) over row-edge ids (SURVEY.md A.3; HTNet -- not in the
 * reference, HermNet/hermnet.py:155-157 raises): all (e1,e2), e1 != e2, in the same row, sorted
 * by (row, e1, e2).  Typed variant: src_type[col[e1]]==type_a and src_type[col[e2]]==type_c
 * (pass src_type=NULL for untyped).
 * ------------------------------------------------------------------------------------------- */
int hn_triplets_count(const int32_t *rowptr, int32_t n_rows, const int32_t *col, const int32_t *src_type,
                      int32_t type_a, int32_t type_c, int64_t *counts /*[R]*/, void *stream);
int hn_triplets_fill(const int32_t *rowptr, int32_t n_rows, const int32_t *col, const int32_t *src_type,
                     int32_t type_a, int32_t type_c, const int64_t *trip_ptr /*[R+1]*/,
                     int32_t *e1 /*[T]*/, int32_t *e2 /*[T]*/, void *stream);
/* dots[r][f] = sum over triplets (e1,e2) of row r of sum_k m_vec[e1][k][f]*m_vec[e2][k][f] */
int hn_triplet_dots(const float *m_vec /*[E,3,F]*/, int32_t F, const int64_t *trip_ptr, const int32_t *e1,
                    const int32_t *e2, int32_t n_rows, float *dots /*[R,F]*/, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Edge geometry.  Replaces HVNet.with_edge, HermNet/hermnet.py:133-152:
 *   D = pos[col[e]] - pos[atom(row(e))] + sign * S_e . cell[graph[col[e]]]   (sign=+1: reference
 *   quirk F5, -1: physical);  d = |D|, d <= 1e-6 -> 1e-6;  u = D/d.   geom[e] = (ux,uy,uz,d).
 * Backward: g_geom[n_parts][E] = (dL/dux, dL/duy, dL/duz, dL/dd), summed over parts, gives
 *   grad_pos[N,3] (segmented sums over the row CSR and its transpose -- no atomics) and, if
 *   cellw != NULL, the per-atom virial partial cellw[i][a][b] = sign * sum_{e in rows(i)} S_e[a]*gD_e[b].
 * ------------------------------------------------------------------------------------------- */
int hn_edge_geom_fwd(const float *pos, const float *cell, const int32_t *atom_graph, const int32_t *edge_row,
                     int32_t rows_per_atom, const int32_t *col, const int8_t *shift, float sign, int64_t n_edges,
                     float *geom /*[E,4]*/, void *stream);
int hn_edge_geom_bwd(const float *geom, const float *g_geom, int32_t n_parts, const int8_t *shift,
                     const int32_t *rowptr, int32_t rows_per_atom, const int32_t *t_rowptr, const int32_t *t_eid,
                     float sign, int64_t n_atoms, int64_t n_edges, float *grad_pos /*[N,3]*/,
                     float *cellw /*[N,9] or NULL*/, void *stream);
/* Per-atom virial from the same gradient (one part, g_geom[E] as above):
 *   virial[i][a][b] = -1/2 sum_{e in rows(i)} D_e[a]*gD_e[b] - 1/2 sum_{e : col[e] = i} D_e[a]*gD_e[b],
 *   D_e = d*u (clamped edges too); rows(i) = rowptr[i*R] .. rowptr[(i+1)*R], sources from the transpose
 *   (t_rowptr, t_eid).  Row = position component, column = force component; not symmetrised.  Summed
 *   over a graph's atoms: W = sum_i pos_i (x) F_i - cell^T dE/dcell = -sum_e D_e (x) gD_e.  One thread
 *   per atom, fixed order, no atomics (bitwise reproducible); zero g_geom rows (dead Verlet-skin
 *   entries) add nothing; n_edges == 0 writes zeros.
 * ------------------------------------------------------------------------------------------- */
int hn_edge_virial_atom(const float *geom /*[E,4]*/, const float *g_geom /*[E,4]*/, const int32_t *rowptr,
                        int32_t rows_per_atom, const int32_t *t_rowptr, const int32_t *t_eid, int64_t n_atoms,
                        int64_t n_edges, float *virial /*[N][9]*/, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Fused PaiNN edge kernel.  Replaces, per layer and per sub-network, HermNet/rmnet.py:55-73
 * (rbf_proj, propagate/message, scatter aggregate), rmnet.py:168-193 (Gaussian RBF x polynomial
 * envelope) and the sub-graph regrouping of HermNet/utils.py:11-24 / hermnet.py:51-61:
 *   phi_e = W[m] . (env(d/rc) * gauss_k(d/rc)) + b[m]                       (3F)
 *   dx[r]      = sum_e  xh[m][s][0:F]  * phi_e[0:F]
 *   dvec[r][k] = sum_e (vec[s][k] * xh[m][s][F:2F]*phi_e[F:2F]/sqrt(3) + xh[m][s][2F:3F]*phi_e[2F:3F]*u_e[k]) / sqrt(F)
 * with m = row_mod[r], s = col[e]; segmented reduction per row, warp shuffles, no global atomics.
 * xh is ONE flat fp32 buffer holding the projected source features of every sub-network compactly;
 * row r reads source s at row (row_xoff[r] + s) of that [rows][3F] buffer (int64 row offsets; for a dense
 * [M][N][3F] layout row_xoff[r] = m*N).  Wt is rbf_proj.weight transposed: [M][K][3F].  gauss_k uses the `offset` buffer (K values,
 * linspace(0,1,K)) and coeff = -0.5/(offset[1]-offset[0])^2; F % 32 == 0.
 * vec may be NULL in fwd and bwd_dst: vec == 0 identically (the first layer, hermnet.py:124), which removes the vec
 * gathers and the F:2F part of the filter from those two passes.
 * bwd_dst (row-major pass): g_geom[n_slices][E] = per-edge (dL/du, dL/dd).
 * bwd_src (source-major pass over the transpose): grad_xh (same flat layout as xh; must be zero-filled
 *   by the caller) and grad_vec[N][3][F].
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_atoms;      /* N: rows of vec / of each xh[m] */
    int32_t n_rows;       /* R */
    int32_t n_modules;    /* M */
    int32_t hidden;       /* F */
    int32_t num_rbf;      /* K */
    int32_t env_p;        /* polynomial envelope exponent */
    float inv_rc;         /* 1/cutoff */
    float coeff;          /* Gaussian coefficient */
    int32_t variant;      /* kernel family of hn_painn_edge_{fwd,bwd_dst,bwd_src}: 0 = auto (quad-tile kernels for F % 64 == 0,
                             else row-per-warp), 1 = row-per-warp only (A/B measurements).  Per call: no library state. */
    int32_t flags;        /* bit 0: the edge list is a Verlet-skin SUPERSET (built with rc + skin): its dead entries must
                             contribute nothing -- not even the filter bias (rmnet.py:55: the reference has no such edge).
                             Every family reads the mask from its own input:
                               hn_tc_edge_*: the sign of tile_geom[.].w (-d for dead, written by hn_tc_tile_windows(live));
                               hn_painn_edge_{fwd,bwd_dst,bwd_src}: the sign of geom[e].w (the caller stores -d for a
                                 dead entry; a real distance is >= 1e-6).  bwd_dst writes exact zeros to the g_geom rows
                                 of dead entries in every slice plane;
                               hn_painn_edge_bwd_w, hn_layer0_basis_*: their live argument (uint8 [E]). */
} hn_edge_params;

/* Planes of g_geom that hn_painn_edge_bwd_dst writes for this F and kernel family (the caller sums them); 0 = unsupported F. */
int32_t hn_painn_edge_num_slices(int32_t hidden, int32_t variant);
int hn_painn_edge_fwd(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                      const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                      const float *Wt, const float *bias, const float *offset, float *dx /*[R,F]*/,
                      float *dvec /*[R,3,F]*/, void *stream);
int hn_painn_edge_bwd_dst(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                          const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                          const float *Wt, const float *bias, const float *offset, const float *g_dx,
                          const float *g_dvec, float *g_geom /*[n_slices,E,4]*/, int64_t n_edges, void *stream);
int hn_painn_edge_bwd_src(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                          const int32_t *t_rowptr, const int32_t *t_eid, const int32_t *edge_row,
                          const int32_t *row_mod, const int64_t *row_xoff, const float *Wt, const float *bias,
                          const float *offset, const float *g_dx, const float *g_dvec, float *grad_xh /*zeroed*/,
                          float *grad_vec /*[N,3,F]*/, void *stream);

/* Filter-weight gradient of the fused path (autograd of nn.Linear rbf_proj, rmnet.py:45,55):
 *   gW_part[chunk][m][k][c] / gb_part[chunk][m][c] hold per-row-chunk partial sums of
 *   gW[m][k][c] = sum_e env*gauss_k(d_e) * dL/dphi_e[c],  gb[m][c] = sum_e dL/dphi_e[c];
 *   the caller adds the n_chunks partials in fixed order (deterministic).
 *   live: uint8 [E], 0 = entry of a Verlet-skin list that is not an edge now (left out of both sums); required with
 *   p->flags bit 0, ignored (may be NULL) without it.  num_rbf up to 1816 (a [K][32] fp32 accumulator fits in 227 KB). */
int hn_painn_edge_bwd_w(const hn_edge_params *p, const float *xh, const float *vec, const float *geom,
                        const int32_t *rowptr, const int32_t *col, const int32_t *row_mod, const int64_t *row_xoff,
                        const uint8_t *live, const float *offset, const float *g_dx, const float *g_dvec,
                        float *gW_part /*[n_chunks,M,K,3F]*/, float *gb_part /*[n_chunks,M,3F]*/, int32_t n_chunks,
                        void *stream);

/* ---------------------------------------------------------------------------------------------
 * First-layer edge pass of HVNet by basis aggregation.  In the first layer x = Embedding[Z], vec = 0
 * (HermNet/hermnet.py:123-124): the projected source features depend only on the source ELEMENT z, so the message sum of
 * rmnet.py:55-73 is linear in per-(destination, element) sums of the radial basis:
 *   Sa[r][z*K + k]        = sum_{e -> r, elem[e] = z} env * gauss_k(d_e)          Sa[r][n_elem*K + z]    = edge count
 *   Sc[r][c][z*K + k]     = sum ... * u_e[c]                                      Sc[r][c][n_elem*K + z] = sum u_e[c]
 * (rows of `kp` floats, kp % 4 == 0, kp >= n_elem * (K + 1); the pad is written as zeros), and
 *   dx[r] = [Sa[r]] . BigA[m]^T,  dvec[r][c] = [Sc[r][c]] . BigC[m]^T   with  BigA[m][f][z*K+k] = xa[m][z][f] * W_a[m][k][f],
 *   BigA[m][f][n_elem*K+z] = xa[m][z][f] * b_a[m][f]  (BigC likewise with xc / sqrt(F)) -- dense GEMMs (hn_gemm_tf32x3).
 * `elem[e]` = element index of the source of row-edge e; rows with row_mod < 0 are skipped (fwd: their S rows are not
 * written; bwd: zeros in g_geom).  bwd: g_geom[e] = (dL/du, dL/dd) from g_Sa / g_Sc (same layout as Sa / Sc).
 * p: n_rows, num_rbf, env_p, inv_rc, coeff, flags (bit 0: `live` [E] uint8 marks the entries of a Verlet-skin list that are
 * edges right now; else live may be NULL).
 * ------------------------------------------------------------------------------------------- */
int hn_layer0_basis_fwd(const hn_edge_params *p, const int32_t *rowptr, const int32_t *elem, const int32_t *row_mod,
                        const float *geom, const uint8_t *live, const float *offset, int32_t n_elem, int32_t kp,
                        float *Sa /*[R,kp]*/, float *Sc /*[R,3,kp]*/, void *stream);
int hn_layer0_basis_bwd(const hn_edge_params *p, const int32_t *rowptr, const int32_t *elem, const int32_t *row_mod,
                        const float *geom, const uint8_t *live, const float *offset, int32_t n_elem, int32_t kp,
                        const float *g_Sa, const float *g_Sc, float *g_geom /*[E,4]*/, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core PaiNN edge kernels (tcgen05 / TMEM / TMA; hidden_channels == 128, num_rbf <= 256).
 * Same arithmetic and reference lines as hn_painn_edge_* above; the filter projection
 * rbf_proj (HermNet/rmnet.py:45,55) runs as fp16-split (hi + lo) tensor-core tiles with fp32
 * accumulation: PHI^T[3F x 64 edges] = W^T[3F x 32-wide basis window] . BASIS^T.
 *
 * Tile plan (built once per graph, replaces the per-layer regrouping of HermNet/utils.py:11-24):
 *   a *block* is up to hn_tc_block_rows(0|1) rows of ONE sub-network (dst-major: row0 + l*stride) or
 *   consecutive source atoms (src-major); a *tile* is up to hn_tc_tile_edges() edges of a block
 *   (src-major: of one (block, sub-network) group) whose Gaussian bands fit one 32-wide window.
 *     blk_info[n_blocks][4]  dst-major (row0, row stride, n_rows, module | -1), src-major (first atom, 1, n, -1)
 *     blk_tile[n_blocks+1]   tile range of each block
 *     tile_info[n_tiles][4]  (first edge record, count, cumulative ends of the (local % G) groups packed 8 bits each, module)
 *     tile_win[n_tiles][2]   (k0, n_chunks): written by hn_tc_tile_windows for the CURRENT geometry, together with
 *     tile_geom[E][4]        the geometry (ux,uy,uz,d) of every record in record order (the kernels read THIS, not geom)
 *     erec[E][4]             dst-major (xh row, source atom, row_local, edge id),
 *                            src-major (destination row, xh row of the source, source_local, edge id)
 *   Build: kc = hn_tc_basis_index(geom); order = edges sorted by (group, kc) (hn_sort_by_key twice);
 *   hn_tc_plan_count -> caller scans -> hn_tc_plan_fill (tile_start) -> hn_tc_plan_finalize, which
 *   sorts every tile by (local % G, local) and writes erec / tile_info from rec[E][4] (indexed by
 *   edge id, field 2 = local index) and tile_mod[n_tiles].
 * Weights: hn_tc_split_weights turns Wt [M][K][3F] into fp16 hi and lo planes [2][M*3F][K32],
 *   K32 = num_rbf rounded up to 32, scaled by a per-module power of two; wscale[m] = 1/scale.
 * Outputs as in hn_painn_edge_*: fwd dx/dvec (every row of every block is written), bwd_dst one
 *   g_geom plane [E][4] (only edges in tiles are written), bwd_src grad_xh (zero-filled by the
 *   caller) and grad_vec (every atom of every block is written).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_blocks;
    int32_t n_tiles;
    const int32_t *blk_info;
    const int32_t *blk_tile;
    const int32_t *blk_xoff;   /* dst-major [n_blocks]: xh row of source s for the block's rows = blk_xoff[b] + erec[.][1] */
    const int32_t *tile_info;
    int32_t *tile_win;
    const int32_t *erec;
    float *tile_geom;          /* [E][4]: geometry of every record, written by hn_tc_tile_windows */
    const float *zero_row;     /* >= 3F zeros (required when hn_edge_params.flags bit 0 is set, else may be NULL) */
    const int32_t *blk_order;  /* [n_blocks] processing order of the blocks (a permutation; NULL = identity).  Results do not
                                  depend on it; interleaving the element-type slices spatially keeps the rows that several
                                  sub-networks gather (vec, g_dx / g_dvec) in L2 between their uses. */
} hn_tc_plan;

int32_t hn_tc_supported(int32_t hidden, int32_t num_rbf);
int32_t hn_tc_block_rows(int32_t src_major);   /* rows (dst-major) / source atoms (src-major) per block */
int32_t hn_tc_tile_edges(void);
int32_t hn_tc_groups(void);          /* epilogue groups G: tiles are sorted by (local % G, local) */
int64_t hn_tc_split_weights_elems(int32_t n_modules, int32_t hidden, int32_t num_rbf);   /* fp16 elements of wsplit */
int hn_tc_split_weights(const float *Wt, int32_t n_modules, int32_t num_rbf, int32_t hidden, void *wsplit /*fp16*/,
                        float *wscale /*[M]*/, void *stream);
int hn_tc_basis_index(const float *geom, int64_t n_edges, float inv_rc, int32_t num_rbf, int32_t *kc /*[E]*/, void *stream);
/* Per-edge inputs of a plan in one pass: kc[e] = basis index of the edge (as hn_tc_basis_index), rec[e][4] = its record
 * (dst-major: xh row, source, row-local index = atom_local[row / rows_per_atom], edge id; src-major: destination row, xh row,
 * source % src_block, edge id), sub[e] = sort sub-key (dst-major: 0, src-major: sub-network of the row; -1 = inactive row). */
int hn_tc_plan_records(int32_t src_major, const int32_t *edge_row, const int32_t *col, const int64_t *row_xoff, const int32_t *row_mod,
                       const int32_t *atom_local, int32_t rows_per_atom, int32_t src_block, const float *geom, float inv_rc,
                       int32_t num_rbf, int64_t n_edges, int32_t *rec, int32_t *kc, int32_t *sub, void *stream);
/* Segment-local sort of the plan builder: segment s = entries in_ptr[s] .. in_ptr[s+1] of the edge list `ids` (NULL: identity)
 * -- the CSR entries of a destination block or the transposed-CSR entries of a source block; entries are ordered by (sub, kc)
 * inside their segment (sub: NULL = 0; -1 drops the entry), stable and deterministic.  Count pass: counts[s * n_sub + sub]
 * (order_out NULL); fill pass: order_out[out_base[s] + position] = edge id (counts NULL).  n_sub * num_rbf <= 8192. */
int hn_tc_plan_sort(const int32_t *in_ptr, const int32_t *ids, const int32_t *kc, const int32_t *sub, int32_t n_seg, int32_t n_sub,
                    int32_t num_rbf, int32_t *counts, const int32_t *out_base, int32_t *order_out, void *stream);
int hn_tc_plan_count(const int32_t *order, const int32_t *kc, const int32_t *grp_ptr, int32_t n_groups, int32_t num_rbf,
                     int32_t window /* 32, 64, ...: basis-index width of a tile (k-chunks per tile = window / 32) */,
                     int32_t *counts, void *stream);
int hn_tc_plan_fill(const int32_t *order, const int32_t *kc, const int32_t *grp_ptr, int32_t n_groups, int32_t num_rbf,
                    int32_t window, const int32_t *grp_tile, int32_t *tile_start, void *stream);
int hn_tc_plan_finalize(const int32_t *order, const int32_t *tile_start, int32_t n_tiles, int64_t n_edges,
                        const int32_t *rec /*[E][4]*/, const int32_t *tile_mod, int32_t *erec, int32_t *tile_info, void *stream);
/* live: NULL, or uint8 [E] -- 0 marks an entry of a Verlet-skin superset list that is not an edge now (stored as -d in
 * tile_geom; with hn_edge_params.flags bit 0 the edge kernels make it contribute nothing) */
int hn_tc_tile_windows(const hn_tc_plan *plan, const float *geom, const uint8_t *live, float inv_rc, int32_t num_rbf, void *stream);
int hn_tc_edge_fwd(const hn_edge_params *p, const hn_tc_plan *plan, const float *xh, const float *vec /*NULL: vec == 0*/,
                   const float *geom, const void *wsplit, const float *wscale, const float *bias, const float *offset,
                   float *dx, float *dvec, float *dbg /*NULL, or 2*E*3F + 14336 floats: phi | raw accumulators | first operand stage*/,
                   int64_t dbg_edges /*E of the debug layout*/, void *stream);
int hn_tc_edge_bwd_dst(const hn_edge_params *p, const hn_tc_plan *plan, const float *xh, const float *vec, const float *geom,
                       const void *wsplit, const float *wscale, const float *bias, const float *offset, const float *g_dx,
                       const float *g_dvec, float *g_geom /*[E][4]*/, void *stream);
int hn_tc_edge_bwd_src(const hn_edge_params *p, const hn_tc_plan *plan /*src-major*/, const float *xh, const float *vec,
                       const float *geom, const void *wsplit, const float *wscale, const float *bias, const float *offset,
                       const float *g_dx, const float *g_dvec, float *grad_xh /*zeroed*/, float *grad_vec, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Row gather / segmented sum -- mutually adjoint linear primitives used by the differentiable
 * (double-backward, training) formulation.  Replace PyG's index_select gathers (rmnet.py:58) and
 * torch_scatter.scatter's atomicAdd (rmnet.py:71-72, hermnet.py:130) with deterministic kernels.
 *   gather:       out[e][:] = X[idx[e]][:]
 *   segment_sum:  out[r][:] = sum_{q in [rowptr[r],rowptr[r+1])} Y[perm ? perm[q] : q][:]
 * Also used for halo pack (gather) / reverse halo accumulation (segment_sum) in the domain-
 * decomposed path.
 * ------------------------------------------------------------------------------------------- */
int hn_gather_rows(const float *X, const int32_t *idx, int64_t n_out, int32_t C, float *out, void *stream);
int64_t hn_segment_sum_workspace_bytes(int32_t n_rows, int32_t C);   /* 0 when no workspace is needed */
int hn_segment_sum(const float *Y, const int32_t *rowptr, const int32_t *perm, int32_t n_rows, int32_t C,
                   float *out, void *workspace, int64_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Row normalisation of the node features: the nn.LayerNorm of rmnet.py:39,52 without its affine part (the caller folds
 * weight / bias into the Linear that follows).  xhat[i] = (x[i] - mean[i]) * rstd[i], rstd = 1/sqrt(var + eps), biased
 * variance over the `hidden` channels; hidden % 32 == 0, <= 512.  Backward: g_x from g_xhat and the saved x, mean, rstd.
 * ------------------------------------------------------------------------------------------- */
int hn_layernorm_fwd(const float *x, int64_t n, int32_t hidden, float eps, float *xhat, float *mean, float *rstd, void *stream);
int hn_layernorm_bwd(const float *g_xhat, const float *x, const float *mean, const float *rstd, int64_t n, int32_t hidden,
                     float *g_x, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Readout MLP (hermnet.py:112-116,129): e_atom[i] = W2 . ssilu(W1 x[i] + b1) + b2, W1 [F/2, F], W2 [F/2], plain fp32 FMAs
 * (the atomic energies cancel strongly in the sum; this layer does not use the 3xTF32 GEMM).  bwd: g_x[i] = dE/dx[i] given
 * g_e[i] = dL/de_atom[i]; the hidden activations are recomputed.  F = 64 or 128 (W1 lives in shared memory); b2: device
 * pointer to the scalar bias (no host read-back: the call can be captured in a CUDA graph).
 * ------------------------------------------------------------------------------------------- */
int hn_readout_fwd(const float *x, const float *W1, const float *b1, const float *W2, const float *b2, int64_t n, int32_t hidden,
                   float *e_atom, void *stream);
int hn_readout_bwd(const float *x, const float *W1, const float *b1, const float *W2, const float *b2, const float *g_e, int64_t n,
                   int32_t hidden, float *g_x, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Halo exchange of the domain-decomposed path (SURVEY.md 8(b)/(e); no counterpart in the reference, whose only
 * multi-GPU path is DDP, example/dist_train.py).  A landing-buffer row is [x (F) | vec (3F)] floats.
 *   hn_halo_pack:   row i = features of atom src_idx[i]; stored at
 *                   ((float *)dst_base[row_peer[i]]) + row_slot[i] * 4F -- dst_base[] holds device addresses: the PEERS'
 *                   landing buffers mapped into this process (NVLink peer memory), or slices of one local send buffer
 *                   (NCCL all-to-all fallback).
 *   hn_halo_unpack: row i of buf -> x[dst_idx[i]], vec[dst_idx[i]] (the ghost rows).
 * The backward pass calls the same pair with the lists swapped (ghost-row gradients into the owners' buffers, then
 * hn_segment_sum): the reverse force accumulation.
 * ------------------------------------------------------------------------------------------- */
int hn_halo_pack(const float *x, const float *vec, const int32_t *src_idx, const int32_t *row_peer, const int32_t *row_slot,
                 const uint64_t *dst_base, int64_t n_rows, int32_t hidden, void *stream);
int hn_halo_unpack(const float *buf, const int32_t *dst_idx, int64_t n_rows, int32_t hidden, float *x, float *vec, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Node-side dense layers on the tcgen05 tensor cores (3xTF32 split, fp32-class accuracy):
 *   C[M,N] (row pitch ldc) = A[M,K] (row pitch lda) . W[N,K]^T + bias[N]   (bias may be NULL)
 * Replaces the cuBLAS fp32 GEMMs behind nn.Linear in HermNet/rmnet.py:40-49 (x_proj), :84-89
 * (vec_proj, xvec_proj) and hermnet.py:112-116 (out_energy) on the fused path.  W is passed
 * pre-split: W_hi = W & 0xFFFFE000 (bitwise), W_lo = W - W_hi.  K % 32 == 0, N % 64 == 0,
 * pitches % 4 == 0, 16-byte aligned pointers.
 * ------------------------------------------------------------------------------------------- */
int hn_gemm_tf32x3(const float *A, int64_t M, int64_t K, int64_t lda, const float *W_hi, const float *W_lo,
                   int64_t N, const float *bias, float *C, int64_t ldc, void *stream);
/* Same GEMM with a fused epilogue (ScaledSiLU of rmnet.py:110-117 and its derivative):
 *   mode 0: C = A.W^T + bias
 *   mode 1: pre = A.W^T + bias;  C2 = pre (optional, row pitch ldc2);  C = silu(pre)/0.6
 *   mode 2: C = (A.W^T) * d[silu(z)/0.6]/dz at z = aux[row][col] (row pitch ld_aux) -- backward through the activation */
int hn_gemm_tf32x3_ex(const float *A, int64_t M, int64_t K, int64_t lda, const float *W_hi, const float *W_lo,
                      int64_t N, const float *bias, float *C, int64_t ldc, int32_t mode, const float *aux,
                      int64_t ld_aux, float *C2, int64_t ldc2, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Fused element-wise stages of the node update (HermNet/rmnet.py:24-32 residuals of PaiNNModule.forward and
 * rmnet.py:94-107 PaiNNUpdate.forward) and their hand-written backward; n rows, F channels, fp32:
 *   pre : xcat[:,0:F] = (x + dx)/sqrt2 (xcat row pitch 2F);  vecp = vec + dvec      (dx / dvec row pitches given)
 *   mid : v12 = [v1 v2] [n,3,2F]:  vdot = sum_k v1*v2/sqrt(F);  xcat[:,F:2F] = sqrt(sum_k v2^2 + 1e-8)
 *   post: a = [a1 a2 a3] [n,3F]:   x_out = xcat[:,0:F] + (a1 + a2*vdot)/sqrt2;  vec_out = vecp + a3*v1
 *   post_bwd: g_a, g_vdot, g_v12[...,0:F] from (g_x, g_vec);   mid_bwd: completes g_v12 from (g_vdot, g_cat[:,F:2F]);
 *   pre_bwd:  g_x (= g_dx) = (g_xn + g_cat[:,0:F])/sqrt2;  g_vec (= g_dvec) = g_vecn + g_vecp
 * ------------------------------------------------------------------------------------------- */
int hn_node_pre(int64_t n, int32_t F, const float *x, const float *dx, int64_t ld_dx, const float *vec,
                const float *dvec, int64_t ld_dvec, float *xcat, float *vecp, void *stream);
int hn_node_mid(int64_t n, int32_t F, const float *v12, float *vdot, float *xcat, void *stream);
int hn_node_post(int64_t n, int32_t F, const float *xcat, const float *a, const float *vdot, const float *vecp,
                 const float *v12, float *x_out, float *vec_out, void *stream);
int hn_node_post_bwd(int64_t n, int32_t F, const float *g_x, const float *g_vec, const float *a, const float *vdot,
                     const float *v12, float *g_a, float *g_vdot, float *g_v12, void *stream);
int hn_node_mid_bwd(int64_t n, int32_t F, const float *g_vdot, const float *g_cat, const float *v12, const float *vn,
                    int64_t ld_vn, float *g_v12, void *stream);
int hn_node_pre_bwd(int64_t n, int32_t F, const float *g_xn, const float *g_cat, const float *g_vecn,
                    const float *g_vecp, float *g_x, float *g_vec, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Langevin (NVT) step of the device MD loop: BAOAB (Leimkuhler-Matthews), units A, fs, eV.  With
 * c1 = exp(-gamma dt), c2 = sqrt(1 - c1^2) (computed by the caller in float64), inv_m = 1/(mass * 103.642697):
 *   hn_md_langevin_baoa   B  v += dt/2 F(x_n) inv_m;  A  x += dt/2 v;
 *                         O  v = c1 v + c2 sqrt(kT[g] inv_m) xi;  A  x += dt/2 v      (pos, vel in place)
 *   -- the caller evaluates F(x_{n+1}) --
 *   hn_md_kick            B  v += half_dt F(x_{n+1}) inv_m;  kinetic[i] = 1/2 |v_i|^2 / inv_m_i (eV; kinetic may be
 *                         NULL);  one thread advances *step by 1.
 * One thread per atom, caller's atom order.  Replica g owns the contiguous atoms replica_ptr[g] .. replica_ptr[g+1]
 * (replica[N] int32 names each atom's replica, replica_ptr[G+1] int32); kT[G] (eV) and seed[G] (int64, bits read as
 * uint64) are per-replica device arrays; step is a device int64 that baoa reads and only kick writes.  Keeping step and
 * kT in device memory lets a captured CUDA graph replay without any host argument changing: every replay draws fresh
 * noise, and a temperature ramp is a copy into kT.
 *
 * Noise (normative): for atom i of replica g, j = i - replica_ptr[g] (replica-local index),
 *   r = Philox4x32-10(counter = (j, lo32(step), hi32(step), 0), key = (lo32(seed[g]), hi32(seed[g])))
 *       (curand_Philox4x32_10 of <curand_philox4x32_x.h>),
 *   u_k = float((r_k >> 9) * 2 + 1) * 2^-24        (k = 0..3: exact in fp32, in [2^-24, 1 - 2^-24]),
 *   xi_x = sqrt(-2 ln u0) cos(2 pi u1),  xi_y = sqrt(-2 ln u0) sin(2 pi u1),  xi_z = sqrt(-2 ln u2) cos(2 pi u3)
 *       (fp32 logf / sincospif; |xi| <= 5.77).
 * The noise of a replica is a function of its seed, the local index and the step alone: independent of the batch it sits
 * in and of the launch configuration, so a trajectory is bitwise reproducible and restartable from any step.
 * Checks: 0 <= n_atoms < 2^31, n_replicas >= 1, dt > 0, 0 <= c1 <= 1, non-null pointers when n_atoms > 0
 * (n_atoms == 0: no-op, step is not advanced).
 * ------------------------------------------------------------------------------------------- */
int hn_md_langevin_baoa(float *pos /*[N,3]*/, float *vel /*[N,3]*/, const float *force /*[N,3]*/, const float *inv_mass /*[N]*/,
                        const int32_t *replica /*[N]*/, const int32_t *replica_ptr /*[G+1]*/, int32_t n_replicas,
                        const float *kT /*[G]*/, const int64_t *seed /*[G]*/, const int64_t *step /*[1]*/, float c1, float c2,
                        float dt, int64_t n_atoms, void *stream);
int hn_md_kick(float *vel /*[N,3]*/, const float *force /*[N,3]*/, const float *inv_mass /*[N]*/, float half_dt, int64_t n_atoms,
               float *kinetic /*[N] or NULL*/, int64_t *step /*[1]*/, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Constant-pressure cell step of the device MD loop: isotropic stochastic cell rescaling (Bernetti & Bussi,
 * J. Chem. Phys. 153, 114107 (2020)), run after hn_md_kick and a per-replica sum of its kinetic energies.
 * Units A, fs, eV; pressures in eV/A^3, beta (isothermal compressibility) in A^3/eV.
 *   hn_md_scr_barostat    one thread per replica g, float64 inside:
 *                           V = |det cell_g|,  P = (2 kinetic[g] + tr virial_g) / (3 V)   (virial as from the force
 *                           pass: W = sum pos (x) F - cell^T dE/dcell, so tr W / 3V = -dU/dV),
 *                           b = beta[g] dt / tau_p,
 *                           de = -b (P0[g] - P) + sqrt(2 kT[g] b / V) xi,   mu = float(exp(de / 3)),
 *                           cell_g = mu * cell_g (fp32, in place),  mu_out[g] = mu,  pressure[g] = float(P).
 *                         The drift carries no +kT/V term: with the velocity scaling below and noise ~ V^-1/2
 *                         (Ito), the zero-flux density is rho(V) ~ V^N exp(-(U + K + P0 V)/kT) (DESIGN.md).
 *   hn_md_affine_scale    one thread per atom i of replica g = replica[i]:  pos_i = mu[g] pos_i,  vel_i = vel_i / mu[g]
 *                         (fp32, in place; with the cell scaled by the same mu every edge vector scales exactly).
 * Noise (normative): for replica g at counter value n = *step (read after hn_md_kick advanced it),
 *   r = Philox4x32-10(counter = (0, lo32(n), hi32(n), 1), key = (lo32(seed[g]), hi32(seed[g]))),
 *   u_k = float((r_k >> 9) * 2 + 1) * 2^-24 (k = 0, 1; as in hn_md_langevin_baoa),
 *   xi = sqrt(-2 ln u0) cos(2 pi u1)        (float64 log / cospi of the exact fp32 uniforms).
 * Counter word 3 = 1 keeps this stream disjoint from the Langevin noise (word 3 = 0) at every step.  P0, kT, beta, seed,
 * step and cell live in device memory, so a captured replay needs no changing host argument and a pressure ramp is a
 * copy into P0.  beta[g] >= 0 is the caller's precondition (device data are not read on the host).
 * Checks: n_replicas >= 0, dt > 0, tau_p > 0 (so dt / tau_p > 0), 0 <= n_atoms < 2^31, non-null pointers when there
 * is work (n_replicas == 0 / n_atoms == 0: no-op).
 * ------------------------------------------------------------------------------------------- */
int hn_md_scr_barostat(float *cell /*[G,3,3]*/, const float *kinetic /*[G]*/, const float *virial /*[G,3,3]*/,
                       const float *P0 /*[G]*/, const float *kT /*[G]*/, const float *beta /*[G]*/, const int64_t *seed /*[G]*/,
                       const int64_t *step /*[1]*/, int32_t n_replicas, float dt, float tau_p, float *mu /*[G]*/,
                       float *pressure /*[G]*/, void *stream);
int hn_md_affine_scale(float *pos /*[N,3]*/, float *vel /*[N,3]*/, const int32_t *replica /*[N]*/, const float *mu /*[G]*/,
                       int64_t n_atoms, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Constant pressure with the cell shape free: triclinic stochastic cell rescaling of lower-triangular cells (lattice
 * vectors = rows of h, h upper triangle 0, diagonal > 0: a along x, b in the xy plane), run after hn_md_kick.  Units and
 * per-replica device arrays as in hn_md_scr_barostat.  Lower triangles are packed (00, 10, 11, 20, 21, 22).
 *   hn_md_kinetic_tensor     one thread per atom:  out[i] = (m v (x) v) lower triangle, m = 1 / inv_mass[i] (fp32); the
 *                            caller sums it per replica (hn_segment_sum) into kin6[g] = sum_i m v (x) v.
 *   hn_md_scr_barostat_tri   one thread per replica g, float64 inside:
 *                              V = h00 h11 h22,  P = (kin6[g] + W_g) / V on the lower triangle (only the lower triangle of
 *                              virial is read; the force pass's W = sum pos (x) F - h^T dE/dh is symmetric to rounding),
 *                              b = beta[g] dt / tau_p,
 *                              delta = (b/3) (P - P0[g] I) + (b kT[g] / 3V) diag(2, 0, -2) + sqrt(2 b kT[g] / 3V) xi
 *                              (lower-triangular; xi = 6 unit normals),
 *                              mu = expm(delta) in closed form (diagonal exponentials, divided differences of exp for the
 *                              off-diagonal entries, expm1-based / series forms for close diagonal entries),
 *                              cell_g = float(h mu) (lower triangle; the upper triangle is written as exact zeros),
 *                              mu_out[g] = float(mu), mu_inv_t[g] = float(expm(-delta)^T) (upper-triangular),
 *                              pressure[g] = the symmetric tensor with lower triangle float(P) (eV/A^3).
 *                            The drift's diag(2, 0, -2) makes rho ~ exp(-(U + K + P0 V)/kT) / (h11 h22^2) in (h, s = x h^-1,
 *                            pi = p h^T) stationary (DESIGN.md, "Triclinic constant pressure"); tr delta has the law of the
 *                            isotropic barostat's strain.  beta = 0 gives mu = I and the cell unchanged bitwise.
 *   hn_md_affine_deform      one thread per atom i of replica g = replica[i] (fp32, in place, row vectors):
 *                              pos_i = pos_i mu[g],  vel_i = vel_i mu_inv_t[g];  mu = I leaves pos / vel bitwise unchanged.
 *                            With the cell deformed by the same mu every edge vector becomes D mu exactly.
 * Noise (normative): for replica g at counter value n = *step (read after hn_md_kick advanced it),
 *   r_k = Philox4x32-10(counter = (k, lo32(n), hi32(n), 2), key = (lo32(seed[g]), hi32(seed[g])))   (k = 0, 1),
 *   u = float((r >> 9) * 2 + 1) * 2^-24 of each word (as in hn_md_langevin_baoa),
 *   per k: z = sqrt(-2 ln u0) cos(2 pi u1), sqrt(-2 ln u0) sin(2 pi u1), sqrt(-2 ln u2) cos(2 pi u3), sqrt(-2 ln u2) sin(2 pi u3)
 *   (float64), and xi = the first 6 of the 8 values in the packed order.  Counter word 3 = 2 keeps this stream disjoint from
 *   the Langevin noise (0) and the isotropic barostat's (1).
 * Lower-triangular cells with a positive diagonal and beta[g] >= 0 are the caller's precondition.
 * Checks: n_replicas >= 0, dt > 0, tau_p > 0, 0 <= n_atoms < 2^31, non-null pointers when there is work (n_replicas == 0 /
 * n_atoms == 0: no-op).
 * ------------------------------------------------------------------------------------------- */
int hn_md_kinetic_tensor(const float *vel /*[N,3]*/, const float *inv_mass /*[N]*/, int64_t n_atoms, float *out /*[N,6]*/,
                         void *stream);
int hn_md_scr_barostat_tri(float *cell /*[G,3,3]*/, const float *kin6 /*[G,6]*/, const float *virial /*[G,3,3]*/,
                           const float *P0 /*[G]*/, const float *kT /*[G]*/, const float *beta /*[G]*/, const int64_t *seed /*[G]*/,
                           const int64_t *step /*[1]*/, int32_t n_replicas, float dt, float tau_p, float *mu /*[G,3,3]*/,
                           float *mu_inv_t /*[G,3,3]*/, float *pressure /*[G,3,3]*/, void *stream);
int hn_md_affine_deform(float *pos /*[N,3]*/, float *vel /*[N,3]*/, const int32_t *replica /*[N]*/, const float *mu /*[G,3,3]*/,
                        const float *mu_inv_t /*[G,3,3]*/, int64_t n_atoms, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Structure relaxation: FIRE (Bitzek et al., PRL 97, 170201 (2006)) with ASE's rules, per replica g, over the generalized
 * coordinates of ASE's UnitCellFilter in row-vector convention (lattice vectors = rows of h).  Masses are ignored.
 * Replicas are contiguous as in hn_md_langevin_baoa (replica[N], replica_ptr[G+1]).
 *   Deformation A_g = h0_g^-1 h_g (float64 [G][9], row-major).  Atom rows r'_i = x_i A^-1, generalized force F'_i = f_i A^T.
 *   With the cell relaxed (A != NULL) three cell rows q_c = c_f A^T with generalized force
 *     F_c = (W_sym - P0 V I) A^-1 / c_f,   W_sym = (W + W^T)/2,  W = sum pos (x) F - h^T dE/dh  (the per-graph virial of
 *     the force pass; W - P0 V I is ASE's filter virial),  V = |det h|,  c_f = cell_factor[g].
 *   A == NULL: positions only; A = I exactly, F' = f and x = r' bitwise (no multiplication).
 * Fixed constants N_min = 5, f_inc = 1.1, f_dec = 0.5, alpha_start = 0.1, f_alpha = 0.99.  Per iteration, with F the
 * generalized forces at the current coordinates and every sum over replica g's rows (atom rows and cell rows alike):
 *   hn_opt_fire_reduce   one warp per chunk of 256 atoms, float64:  sums[g] = (sum F'.v, sum |F'|^2, sum |v|^2,
 *                        max_i |F'_i|^2) over the atom rows.  The piece (chunk b) x (replica g) is written to workspace slot
 *                        b + g and the pieces of a replica are summed in order (a warp per replica, or a block when replicas
 *                        span many chunks): fixed summation order, no atomics, bitwise reproducible for a given (N, G).
 *   hn_opt_fire_step     one thread per replica, float64.  Adds the cell rows (A != NULL), writes fmax_out[g] = max row |F|,
 *                        then:  converged[g] set: nothing more.  max row |F|^2 < fmax^2: converged[g] = 1 (sticky; the
 *                        replica never moves again).  Otherwise the replica counts in *n_active (zeroed by the call) and,
 *                        with move != 0, takes a FIRE step:
 *                          steps[g] == 0 (ASE's v is None):  c_v = 0, c_m = 0 (dt, alpha unchanged);
 *                          P = F.v > 0:  c_v = 1 - alpha, c_m = alpha |v| / |F|;  if n_pos > N_min: dt = min(f_inc dt, dt_max),
 *                                        alpha *= f_alpha;  n_pos += 1;
 *                          else:         c_v = 0, c_m = 0, alpha = alpha_start, dt *= f_dec, n_pos = 0;
 *                          v_new = c_v v + c_f' F with c_f' = c_m + dt, |v_new|^2 = c_v^2 |v|^2 + 2 c_v c_f' F.v + c_f'^2 |F|^2
 *                          (closed form: no second atom pass), s = min(1, max_step / (dt |v_new|)),
 *                          coef[g] = (c_v, c_f', s dt), steps[g] += 1;
 *                        cell rows: vcell = c_v vcell + c_f' F_c, A_prev = A, A = ((c_f A^T + s dt vcell) / c_f)^T,
 *                        cell = float(h0 A) in place.  move == 0: convergence test only (the last evaluation of a capped run).
 *   hn_opt_fire_update   one thread per atom of a replica with converged[g] == 0:  v = c_v v + c_f' F'_i (F' at A_prev, the
 *                        deformation the forces were evaluated at),  r' += s dt v (fp32 storage, float64 arithmetic),
 *                        x = r' A (the new deformation; A == NULL: r' is the positions and x is not used).
 * State (device memory, caller-owned): dt, alpha [G] float64, n_pos, steps, converged [G] int32, vcell, A, A_prev [G][9]
 * float64, h0 [G][9] float64.  Initial values: dt = the user's dt, alpha = 0.1, zeros, A = I, v = 0, r' = x.
 * Checks: 0 <= n_atoms < 2^31, n_replicas >= 0, fmax, dt_max, max_step > 0, non-null pointers when there is work
 * (n_atoms == 0 / n_replicas == 0: no-op); the reduce workspace holds hn_opt_fire_reduce_workspace_bytes.
 * ------------------------------------------------------------------------------------------- */
int64_t hn_opt_fire_reduce_workspace_bytes(int64_t n_atoms, int32_t n_replicas);
int hn_opt_fire_reduce(const float *force /*[N,3]*/, const float *vel /*[N,3]*/, const double *A /*[G,9] or NULL*/,
                       const int32_t *replica /*[N]*/, const int32_t *replica_ptr /*[G+1]*/, int32_t n_replicas, int64_t n_atoms,
                       double *sums /*[G,4]*/, void *workspace, int64_t workspace_bytes, void *stream);
int hn_opt_fire_step(const double *sums /*[G,4]*/, const float *virial /*[G,3,3]*/, float *cell /*[G,3,3]*/,
                     const double *h0 /*[G,9]*/, double *A /*[G,9] or NULL*/, double *A_prev /*[G,9]*/, double *vcell /*[G,9]*/,
                     const double *P0 /*[G] eV/A^3*/, const double *cell_factor /*[G]*/, double *dt /*[G]*/, double *alpha /*[G]*/,
                     int32_t *n_pos /*[G]*/, int32_t *steps /*[G]*/, int32_t *converged /*[G]*/, int32_t n_replicas, double fmax,
                     double dt_max, double max_step, int32_t move, double *coef /*[G,3]*/, double *fmax_out /*[G]*/,
                     int32_t *n_active /*[1]*/, void *stream);
int hn_opt_fire_update(float *x /*[N,3]*/, float *rp /*[N,3]*/, float *vel /*[N,3]*/, const float *force /*[N,3]*/,
                       const double *A_prev /*[G,9]*/, const double *A /*[G,9] or NULL*/, const int32_t *replica /*[N]*/,
                       const int32_t *converged /*[G]*/, const double *coef /*[G,3]*/, int64_t n_atoms, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Nudged elastic band forces (csrc/hn_neb.cu): ASE's NEB(method="improvedtangent", climb=...) over B bands of K interior
 * images each.  Band-major layout of the N_img = B K images: image g = b K + k of band b is the contiguous atom range
 * [image_ptr[g], image_ptr[g+1]) of n_b atoms (image[i] = g), images 0..K-1 of a band one after the other; the endpoints are
 * `initial` / `final` [sum n_b, 3] with band b at rows band_ptr[b] .. band_ptr[b+1] in the same atom order.  For atom i of
 * image k: R_{k-1} is pos[i - n_b] (k > 0) or initial[band_ptr[b] + local] (k == 0), R_{k+1} is pos[i + n_b] (k < K-1) or
 * final[band_ptr[b] + local] (k == K-1);  D+ = R_{k+1} - R_k,  D- = R_k - R_{k-1}.
 *   hn_neb_reduce    sums[g] = (|D+|^2, |D-|^2, D+.D-, F.D+, F.D-) over the atoms of image g, float64 from fp32 positions and
 *                    forces; the fixed-order chunk / slot scheme of hn_opt_fire_reduce (bitwise reproducible for a given
 *                    layout), workspace of hn_neb_reduce_workspace_bytes.
 *   hn_neb_step      one thread per band, float64 (energies promoted from fp32; end_energy[b] = (E_initial, E_final)):
 *                    imax[b] = 1 + the first k of maximal energy (1..K, the numbering with the endpoints at 0 and K+1);
 *                    tangent tau = a D+ + w D-:  E_{k+1} > E_k > E_{k-1}: (1, 0);  E_{k+1} < E_k < E_{k-1}: (0, 1);  else
 *                    with V_max / V_min the larger / smaller of |E_{k+1} - E_k|, |E_{k-1} - E_k|:  (V_max, V_min) if
 *                    E_{k+1} > E_{k-1} else (V_min, V_max), and (1, 1) when V_max == 0.  T = a^2 S++ + 2 a w S+- + w^2 S--,
 *                    Ft = a F+ + w F-;  q = -2 Ft / T for the climbing image (climb != 0 and k == imax - 1), else
 *                    q = -Ft / T + spring[b] (sqrt S++ - sqrt S--) / sqrt T;  q = 0 when T == 0.  coef[g] = (q a, q w).
 *   hn_neb_project   per atom: F <- F + coef[g][0] D+ + coef[g][1] D-  (float64 arithmetic, fp32 in place).
 * Checks: 0 <= n_atoms < 2^31, n_bands >= 0, n_images >= 1, non-null pointers when there is work (no atoms / no bands:
 * no-op).  No host synchronisation.
 * ------------------------------------------------------------------------------------------- */
int64_t hn_neb_reduce_workspace_bytes(int64_t n_atoms, int32_t n_img);
int hn_neb_reduce(const float *pos /*[M,3]*/, const float *force /*[M,3]*/, const float *initial /*[N,3]*/, const float *final_ /*[N,3]*/,
                  const int32_t *image /*[M]*/, const int32_t *image_ptr /*[B*K+1]*/, const int32_t *band_ptr /*[B+1]*/,
                  int32_t n_bands, int32_t n_images, int64_t n_atoms /*M = K N*/, double *sums /*[B*K,5]*/, void *workspace,
                  int64_t workspace_bytes, void *stream);
int hn_neb_step(const double *sums /*[B*K,5]*/, const float *energy /*[B*K]*/, const float *end_energy /*[B,2]*/,
                const double *spring /*[B]*/, int32_t climb, int32_t n_bands, int32_t n_images, double *coef /*[B*K,2]*/,
                int32_t *imax /*[B]*/, void *stream);
int hn_neb_project(float *force /*[M,3]*/, const float *pos /*[M,3]*/, const float *initial /*[N,3]*/, const float *final_ /*[N,3]*/,
                   const int32_t *image /*[M]*/, const int32_t *image_ptr /*[B*K+1]*/, const int32_t *band_ptr /*[B+1]*/,
                   int32_t n_bands, int32_t n_images, const double *coef /*[B*K,2]*/, int64_t n_atoms, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HERMNET_B200_H */
