"""Minimum-energy paths on the device: climbing-image nudged elastic band (NEB) over batched bands.

The host route is ASE's ``NEB(images, climb=True, method="improvedtangent")`` driven by ``FIRE`` over ``NNCalculator``: one
``calculate`` per image per iteration, each with a host round trip and a fresh neighbour list, one band at a time.  Here
the interior images of many bands are the replicas of one device evaluation, the NEB force is three kernels
(``hn_neb_{reduce,step,project}``) and FIRE runs per band with the kernels of ``fire_relax_device``."""
from __future__ import annotations

import numpy as np
import torch

from .. import ops
from .md import VerletGraph, _host, _replica_floats, _setup, _stack
from .relax import _Fire, _fire_params


def neb_device(model, numbers, initial, final, cell, n_images=5, images=None, batch=None, spring_constant=0.1, climb=False,
               fmax=0.05, max_steps=1000, dt=0.1, dt_max=1.0, max_step=0.2, skin=0.0, cuda_graph=False, stats=None,
               device="cuda"):
    """Relax ``B`` bands of ``K = n_images`` interior images between fixed endpoints to the minimum-energy path with ASE's
    improved-tangent NEB and FIRE.  Returns ``(images [K,N,3], energies [B,K+2])``: ``images[k]`` is image ``k`` of every
    band in the atom order of ``initial``, and ``energies[b]`` holds ``E(initial)``, the energies of the returned images and
    ``E(final)``.

    ``numbers [N]``, ``initial`` / ``final [N,3]``, ``cell`` (``None`` for clusters, ``[3,3]`` or ``[B,3,3]``, fixed) and
    ``batch`` (``None`` for one band, or a PyG batch vector over ``B`` bands, which may differ in size) follow
    ``fire_relax_device``; every image uses the same ``numbers`` and ``batch``.  The endpoints never move and are evaluated
    once, together.  The NEB force of interior image ``k`` with ``D+ = R_{k+1} - R_k`` and ``D- = R_k - R_{k-1}`` is the
    improved tangent of Henkelman & Jonsson (2000) ``tau = a D+ + b D-`` (the weights ``a``, ``b`` from the energies; (1, 1)
    when three neighbouring energies are equal, where ASE divides by zero): the force perpendicular to ``tau`` plus the
    spring ``k (|D+| - |D-|) tau / |tau|`` with ``spring_constant`` (eV/A^2, a float or ``B`` values).  With ``climb`` the
    first image of highest energy in each band (lowest ``k`` on ties) climbs from the first iteration: ``F - 2 (F.tau) tau /
    |tau|^2`` without spring (Henkelman, Uberuaga & Jonsson 2000).

    FIRE treats a whole band as one system, as ASE's FIRE does on an NEB: one ``dt`` / ``alpha`` / ``n_pos`` per band, the
    ``max_step`` cap on the band's whole step and convergence when every interior atom of the band has ``|F_NEB| < fmax``.
    ``fmax``, ``max_steps``, ``dt``, ``dt_max``, ``max_step``, ``skin`` and ``cuda_graph`` mean what they mean in
    ``fire_relax_device``; convergence is sticky per band (a converged band keeps its coordinates bitwise), and the run ends on
    an evaluation, so returned images and energies belong together.

    Initial band.  ``images=None``: the linear interpolation ``initial + (k+1)/(K+1) (final' - initial)``.  ``images``
    ``[K,N,3]`` (for example the result of a plain run, to continue with ``climb=True``): used as given.  In a periodic cell
    every configuration is first re-expressed next to its predecessor along the band with the fractional wrap ``d -> (s -
    round(s)) h`` of the displacement ``d`` (``s = d h^-1``, per atom): ``final' = initial + wrap(final - initial)`` without
    ``images``, else ``R_0``, ..., ``R_{K-1}`` and then ``final`` in turn from ``initial``.  This is the minimum image only
    in cells that are not strongly skewed.  The band then lives in unwrapped coordinates.

    ``stats`` (optional dict) receives ``converged [B]`` (bool) and ``steps [B]``; per evaluation ``energy [iters,B,K]``,
    ``fmax [iters,B]`` (the largest NEB force of the band) and ``imax [iters,B]`` (the first highest image, numbered
    ``1..K`` as in ``energies``; reported with or without ``climb``); the FIRE state after each step ``dt``, ``alpha`` and
    ``n_pos [iters,B]``; and ``builds`` / ``reuses`` of the images' neighbour lists.

    ``ValueError`` for the parameters ``fire_relax_device`` rejects, ``n_images < 1``, spring constants that are not finite
    and > 0, endpoints or images of the wrong shape or not finite, a singular cell, and a band in which ``initial`` and
    ``final'``, or two consecutive configurations, coincide in every atom.

    Example: relax the endpoints, run plain NEB, then continue with the climbing image::

        xa, _, _ = fire_relax_device(model, Z, a, cell, fmax=0.01)
        xb, _, _ = fire_relax_device(model, Z, b, cell, fmax=0.01)
        path, _ = neb_device(model, Z, xa, xb, cell, n_images=7, fmax=0.1)
        path, energies = neb_device(model, Z, xa, xb, cell, n_images=7, images=path, climb=True, fmax=0.02)
        barrier = energies.max(1).values - energies[:, 0]
    """
    name = "neb_device"
    max_steps = _fire_params(name, fmax, dt, dt_max, max_step, max_steps)
    if not (int(n_images) == n_images and n_images >= 1):
        raise ValueError(f"{name}: n_images must be an integer >= 1 (got {n_images})")
    K = int(n_images)
    n = len(_host(numbers))
    if n == 0:
        raise ValueError(f"{name}: there are no atoms")
    x0, x1 = (_configurations(v, (n, 3), what, name) for v, what in ((initial, "initial"), (final, "final")))
    R = None if images is None else _configurations(images, (K, n, 3), "images", name)
    st = _setup(name, numbers, x0, cell, batch, device,
                cell_error=None if cell is None else "cell must be finite and non-singular")
    B, sizes = st.G, st.sizes
    rptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    spring = _replica_floats(spring_constant, B, "spring_constant", name, lambda v: np.isfinite(v) & (v > 0.0),
                             "spring constants must be finite and > 0")
    rep = np.repeat(np.arange(B), sizes)

    # the band in float64 on the host, once: re-expressed along the band, then rounded to fp32
    wrap = _fractional_wrap(cell, B, rep)
    if R is None:
        x1 = x0 + wrap(x1 - x0)
        R = x0 + (np.arange(1, K + 1) / (K + 1))[:, None, None] * (x1 - x0)
    else:
        prev = x0
        for k in range(K):
            R[k] = prev = prev + wrap(R[k] - prev)
        x1 = prev + wrap(x1 - prev)
    band = np.concatenate([x0[None], R, x1[None]]).astype(np.float32)
    ends_equal = np.logical_and.reduceat((band[-1] == band[0]).all(1), rptr[:-1])                    # [B]
    if ends_equal.any():
        raise ValueError(f"{name}: initial and final coincide in band(s) {np.flatnonzero(ends_equal).tolist()}")
    same = np.logical_and.reduceat((band[1:] == band[:-1]).all(2), rptr[:-1], axis=1)              # [K+1, B]
    if same.any():
        raise ValueError(f"{name}: two consecutive configurations of band(s) {np.flatnonzero(same.any(0)).tolist()} coincide "
                         "in every atom")

    # band-major layout: band b holds images 0..K-1 of its n_b atoms; public (k, atom a) sits at internal row dst[k, a]
    local = np.arange(n) - rptr[rep]
    dst = K * rptr[rep][None, :] + np.arange(K)[:, None] * sizes[rep][None, :] + local[None, :]
    dev = st.pos.device
    perm = torch.from_numpy(dst.reshape(-1)).to(dev)
    pos = torch.empty((K * n, 3), dtype=torch.float32, device=dev)
    pos[perm] = torch.from_numpy(band[1:-1].reshape(-1, 3)).to(dev)
    inner = np.empty(K * n, dtype=np.int64)
    inner[dst.reshape(-1)] = (rep[None, :] * K + np.arange(K)[:, None]).reshape(-1)
    image = torch.from_numpy(inner.astype(np.int32)).to(dev)
    image_ptr = torch.from_numpy(np.append((K * rptr[:-1, None] + np.arange(K)[None, :] * sizes[:, None]).reshape(-1),
                                           K * n).astype(np.int32)).to(dev)
    band_of = torch.from_numpy((inner // K).astype(np.int32)).to(dev)
    band_rows = torch.from_numpy((K * rptr).astype(np.int32)).to(dev)
    Z = torch.empty(K * n, dtype=st.Z.dtype, device=dev)
    Z[perm] = st.Z.repeat(K)
    c = None if st.c is None else st.c.repeat_interleave(K, 0)
    x0_t, x1_t = st.pos, torch.from_numpy(band[-1]).to(dev)
    spring_t = torch.from_numpy(spring).to(dev)

    ends = VerletGraph(model, batch=torch.cat([st.replica, st.replica + B]).long())
    e_end = ends.evaluate(torch.cat([x0_t, x1_t]), torch.cat([st.Z, st.Z]), None if st.c is None else torch.cat([st.c, st.c]))[0]
    e_end = torch.stack([e_end[:B], e_end[B:]], 1).contiguous()

    vg = VerletGraph(model, skin, cuda_graph, batch=None if B * K == 1 else image.long())
    fire = _Fire(pos, band_of, band_rows, B, fmax, dt, dt_max, max_step)
    coef = torch.zeros((B * K, 2), dtype=torch.float64, device=dev)
    imax = torch.zeros(B, dtype=torch.int32, device=dev)
    energy, imaxs = [], []
    for it in range(max_steps + 1):
        e, f = vg.evaluate(pos, Z, c)
        e = e.contiguous()
        sums = ops.neb_reduce(pos, f, x0_t, x1_t, image, image_ptr, st.replica_ptr, K)
        ops.neb_step(sums, e, e_end, spring_t, climb, coef, imax)
        ops.neb_project(f, pos, x0_t, x1_t, image, image_ptr, st.replica_ptr, K, coef)
        energy.append(e.view(B, K))
        imaxs.append(imax.clone())
        if fire.step(f, it < max_steps):
            break
        fire.update(f)
    if stats is not None:
        tr = fire.trace
        stats.update(vg.counts(), converged=fire.converged.bool(), steps=fire.steps.clone(), energy=_stack(energy, e, B, K),
                     fmax=_stack(tr["fmax"], e, B), imax=_stack(imaxs, imax, B),
                     **{k: _stack(tr[k], e, B) for k in ("dt", "alpha", "n_pos")})
    return pos[perm].view(K, n, 3), torch.cat([e_end[:, :1], e.view(B, K), e_end[:, 1:]], 1)


def _configurations(value, shape, what, name) -> np.ndarray:
    """``value`` as a float64 host array of ``shape`` with finite entries (``ValueError`` otherwise)."""
    v = _host(value).astype(np.float64)
    if v.shape != shape:
        raise ValueError(f"{name}: {what} must be {list(shape)}, got {list(v.shape)}")
    if not np.isfinite(v).all():
        raise ValueError(f"{name}: {what} must be finite")
    return v.copy()


def _fractional_wrap(cell, B, rep):
    """``d -> (s - round(s)) h`` per atom with ``s = d h^-1`` and ``h`` the cell of the atom's band (identity for clusters)."""
    if cell is None:
        return lambda d: d
    h = np.broadcast_to(_host(cell).astype(np.float64).reshape(-1, 3, 3), (B, 3, 3))
    h_inv = np.linalg.inv(h)

    def wrap(d):
        s = np.einsum("ni,nij->nj", d, h_inv[rep])
        return np.einsum("ni,nij->nj", s - np.round(s), h[rep])
    return wrap
