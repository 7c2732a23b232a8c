// Deterministic per-segment reduction over contiguous segments of atoms (replicas, images), shared by hn_opt.cu and
// hn_neb.cu.  Two passes with a caller-owned workspace of (chunks + segments) slots:
//   pieces  one warp per REDUCE_CHUNK-atom chunk c; the piece (chunk c) x (segment g) goes to slot c + g, which is unique
//           because c + g strictly increases along the atoms.  Lanes stride over the piece, then a fixed xor tree.
//   slots   `per` threads (32 or 256) merge the slots of one segment in slot order, then the same xor tree and, with 256,
//           the 8 warps in order.
// The order of every operation depends on (n_atoms, segment_ptr) only: two launches are bitwise equal.
//
// Acc is a plain struct with   void merge(const Acc &o)   (this = this (+) o, applied field by field) and
//                              Acc shfl_xor(int o) const  (every field from lane ^ o);
// a zero-initialised Acc{} is the identity of merge.
#pragma once
#include <cuda_runtime.h>

namespace hn {

constexpr int REDUCE_CHUNK = 256;        // atoms of one warp's piece (8 per lane)

inline int64_t reduce_chunks(int64_t n_atoms) { return (n_atoms + REDUCE_CHUNK - 1) / REDUCE_CHUNK; }

template <class Acc>
__device__ __forceinline__ void warp_merge(Acc &a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a.merge(a.shfl_xor(o));
}

// Pieces pass, called by every thread of the grid (blockDim a multiple of 32).  make_atom(g) returns the per-atom
// accumulation of segment g, a callable (Acc &, int atom); per-segment set-up belongs in make_atom.
template <class Acc, class MakeAtom>
__device__ __forceinline__ void reduce_pieces(const int *__restrict__ segment, const int *__restrict__ segment_ptr, int n_atoms,
                                              int n_chunks, Acc *__restrict__ part, MakeAtom make_atom) {
    const int c = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (c >= n_chunks) return;
    const int a0 = c * REDUCE_CHUNK, a1 = min(a0 + REDUCE_CHUNK, n_atoms);
    const int g_last = __ldg(segment + a1 - 1);
    for (int g = __ldg(segment + a0); g <= g_last; ++g) {
        const int s = max(a0, __ldg(segment_ptr + g)), e = min(a1, __ldg(segment_ptr + g + 1));
        if (s >= e) continue;
        auto atom = make_atom(g);
        Acc acc{};
        for (int i = s + lane; i < e; i += 32) atom(acc, i);
        warp_merge(acc);
        if (lane == 0) part[c + g] = acc;
    }
}

// Slots pass, called by every thread of the grid (blockDim 256).  Returns true in the one thread that holds segment g's
// total in `out` (g < n_segments).
template <class Acc>
__device__ __forceinline__ bool reduce_slots(const Acc *__restrict__ part, const int *__restrict__ segment_ptr, int n_segments,
                                             int per, int &g, Acc &out) {
    __shared__ Acc warp_acc[8];
    g = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) / per);
    const int t = threadIdx.x % per;
    Acc acc{};
    if (g < n_segments) {
        const int p0 = __ldg(segment_ptr + g), p1 = __ldg(segment_ptr + g + 1);
        if (p1 > p0) {
            const int c1 = (p1 - 1) / REDUCE_CHUNK;
#pragma unroll 4
            for (int c = p0 / REDUCE_CHUNK + t; c <= c1; c += per) acc.merge(part[c + g]);
        }
    }
    warp_merge(acc);
    if (per > 32) {                           // one segment per block: combine the 8 warps in order
        if ((threadIdx.x & 31) == 0) warp_acc[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x != 0) return false;
        acc = warp_acc[0];
        for (int w = 1; w < 8; ++w) acc.merge(warp_acc[w]);
    } else if (t != 0) {
        return false;
    }
    out = acc;
    return g < n_segments;
}

// a block per segment when segments span many chunks on average, else a warp per segment
inline int reduce_slot_threads(int64_t chunks, int64_t n_segments) { return chunks >= 64 * n_segments ? 256 : 32; }

}  // namespace hn
