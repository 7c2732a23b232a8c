"""Minimum-energy paths on the device: ``hn_neb_reduce`` / ``hn_neb_step`` / ``hn_neb_project`` (``ops.neb_*``) and
``plugin.neb.neb_device``.

Two float64 references:
- ``ref_neb_forces`` is the NEB force in vector form, image by image, as the papers and ASE's ``improvedtangent`` method
  write it (explicit tangent, normalised; projection, spring, climb).  It does not use the coefficient algebra of the
  kernels, so it checks that algebra;
- ``ref_reduce`` / ``ref_step`` / ``ref_project`` follow the header of include/hermnet_b200.h on the band-major layout; they
  are the oracle of the kernels on the GPU and stand in for the three ops in the CPU cases over the kernel emulator.
The driver is checked against ``host_fire`` of tests/test_relax.py driving the concatenated interior images of a band with
``ref_neb_forces`` as the force, and on a Mueller-Brown surface against its saddle point found by Newton's method."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import hermnet_b200 as H
from hermnet_b200 import ops, synthetic
from hermnet_b200.plugin.neb import neb_device
from hermnet_b200.plugin.relax import fire_relax_device
from tests.test_langevin import _cpu_model, _cpu_systems, _replica_tensors, _water_model
from tests.test_relax import emu_relax, host_fire  # noqa: F401  (emu_relax is a fixture)

DEV = "cuda:0"


def _np(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------
def _weights(em, e, ep):
    """Improved-tangent weights ``(a, b)`` of ``tau = a D+ + b D-`` and the name of the branch taken."""
    if ep > e > em:
        return 1.0, 0.0, "up"
    if ep < e < em:
        return 0.0, 1.0, "down"
    vmax, vmin = max(abs(ep - e), abs(em - e)), min(abs(ep - e), abs(em - e))
    if vmax == 0.0:
        return 1.0, 1.0, "flat"
    if ep > em:
        return vmax, vmin, "extremum, E+ > E-"
    return vmin, vmax, "extremum, E+ <= E-"


def ref_neb_forces(R, E, F, k, climb):
    """NEB forces ``[K,n,3]`` of one band in vector form: ``R [K+2,n,3]`` the band with its endpoints, ``E [K+2]`` its
    energies, ``F [K,n,3]`` the model forces of the interior images, ``k`` the spring constant.  Returns ``(F_neb, imax)``
    with ``imax`` in ``1..K``."""
    R, E, F = (np.asarray(a, dtype=np.float64) for a in (R, E, F))
    K = len(R) - 2
    imax = 1 + int(np.argmax(E[1:-1]))                    # the first maximum
    out = np.empty_like(F)
    for i in range(1, K + 1):
        t_plus, t_minus = R[i + 1] - R[i], R[i] - R[i - 1]
        a, b, _ = _weights(E[i - 1], E[i], E[i + 1])
        tau = a * t_plus + b * t_minus
        f = F[i - 1]
        norm = np.sqrt(np.vdot(tau, tau))
        if norm == 0.0:
            out[i - 1] = f
            continue
        tau = tau / norm
        if climb and i == imax:
            out[i - 1] = f - 2.0 * np.vdot(f, tau) * tau
        else:
            out[i - 1] = f - np.vdot(f, tau) * tau + tau * k * (np.linalg.norm(t_plus) - np.linalg.norm(t_minus))
    return out, imax


def _neighbours(pos, initial, final, image, image_ptr, band_ptr, K):
    """``(x, R_{k-1}, R_{k+1})`` of every band-major atom, float64."""
    x, x0, x1 = (_np(t).astype(np.float64) for t in (pos, initial, final))
    img, ip, bp = (_np(t).astype(np.int64) for t in (image, image_ptr, band_ptr))
    i = np.arange(len(x))
    b, k = img // K, img % K
    nb = ip[img + 1] - ip[img]
    end = bp[b] + i - ip[img]
    prev = np.where((k == 0)[:, None], x0[np.minimum(end, len(x0) - 1)], x[np.maximum(i - nb, 0)])
    nxt = np.where((k == K - 1)[:, None], x1[np.minimum(end, len(x1) - 1)], x[np.minimum(i + nb, len(x) - 1)])
    return x, prev, nxt


def ref_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K):
    """``[B K,5]``: ``(|D+|^2, |D-|^2, D+.D-, F.D+, F.D-)`` per image."""
    x, prev, nxt = _neighbours(pos, initial, final, image, image_ptr, band_ptr, K)
    dp, dm, f = nxt - x, x - prev, _np(force).astype(np.float64)
    img, n_img = _np(image).astype(np.int64), _np(image_ptr).size - 1
    terms = [(dp * dp).sum(1), (dm * dm).sum(1), (dp * dm).sum(1), (f * dp).sum(1), (f * dm).sum(1)]
    return np.stack([np.bincount(img, t, n_img) for t in terms], 1)


def ref_step(sums, energy, end_energy, spring, climb, branches=None):
    """``(coef [B K,2], imax [B])`` of the header's rules, per band and image."""
    E, ends, ks = _np(energy).astype(np.float64), _np(end_energy).astype(np.float64).reshape(-1, 2), _np(spring)
    B = len(ks)
    K = len(E) // B
    coef, imax = np.zeros((B * K, 2)), np.zeros(B, dtype=np.int32)
    for b in range(B):
        Eb = np.concatenate([[ends[b, 0]], E[b * K:(b + 1) * K], [ends[b, 1]]])
        top = int(np.argmax(Eb[1:-1]))
        imax[b] = top + 1
        for k in range(K):
            g = b * K + k
            a, w, name = _weights(Eb[k], Eb[k + 1], Eb[k + 2])
            spp, smm, spm, fp, fm = sums[g]
            T, ft = a * a * spp + 2 * a * w * spm + w * w * smm, a * fp + w * fm
            q = 0.0
            if T > 0.0:
                q = -2.0 * ft / T if (climb and k == top) else -ft / T + ks[b] * (np.sqrt(spp) - np.sqrt(smm)) / np.sqrt(T)
            coef[g] = q * a, q * w
            if branches is not None:
                branches.add("T = 0" if T == 0.0 else name)
    return coef, imax


def ref_project(force, pos, initial, final, image, image_ptr, band_ptr, K, coef):
    """The projected forces ``[M,3]`` (float32)."""
    x, prev, nxt = _neighbours(pos, initial, final, image, image_ptr, band_ptr, K)
    c = _np(coef)[_np(image).astype(np.int64)]
    return (_np(force).astype(np.float64) + c[:, :1] * (nxt - x) + c[:, 1:] * (x - prev)).astype(np.float32)


# --- CPU stand-ins of the three ops (same contracts) ---
def emu_neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, n_images):
    return torch.from_numpy(ref_reduce(pos, force, initial, final, image, image_ptr, band_ptr, n_images))


def emu_neb_step(sums, energy, end_energy, spring, climb, coef, imax):
    c, m = ref_step(_np(sums), energy, end_energy, spring, climb)
    coef.copy_(torch.from_numpy(c))
    imax.copy_(torch.from_numpy(m))


def emu_neb_project(force, pos, initial, final, image, image_ptr, band_ptr, n_images, coef):
    force.copy_(torch.from_numpy(ref_project(force, pos, initial, final, image, image_ptr, band_ptr, n_images, coef)))


@pytest.fixture
def emu_neb(emu_relax, monkeypatch):
    monkeypatch.setattr(ops, "neb_reduce", emu_neb_reduce)
    monkeypatch.setattr(ops, "neb_step", emu_neb_step)
    monkeypatch.setattr(ops, "neb_project", emu_neb_project)
    return emu_relax


def band_major(bands, K):
    """Band-major layout of ``bands`` (list of ``[K+2,n_b,3]`` arrays, endpoints included): ``(pos [K N,3], initial [N,3],
    final [N,3], image, image_ptr, band_ptr)`` as tensors."""
    sizes = [b.shape[1] for b in bands]
    pos = np.concatenate([b[1:-1].reshape(-1, 3) for b in bands]).astype(np.float32)
    initial = np.concatenate([b[0] for b in bands]).astype(np.float32)
    final = np.concatenate([b[-1] for b in bands]).astype(np.float32)
    image_sizes = [n for n in sizes for _ in range(K)]
    image, image_ptr = _replica_tensors(image_sizes, "cpu")
    band_ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32)
    return torch.from_numpy(pos), torch.from_numpy(initial), torch.from_numpy(final), image, image_ptr, band_ptr


# Energy patterns of 5-image bands that take every branch of the tangent between them (endpoints at both ends).
PATTERNS = [
    [0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0],          # monotone up
    [6.0, 5.0, 4.0, 3.0, 2.0, 1.0, 0.0],          # monotone down
    [0.0, 1.0, 3.0, 2.5, 3.0, 1.0, 0.5],          # local maxima, a local minimum, E+ = E- at the minimum
    [0.0, 1.0, 3.0, 3.0, 3.0, 2.0, 0.0],          # three equal energies, ties for the climbing image
    [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0],          # flat everywhere
]


def _random_bands(seed, K=5):
    """Bands with the energy patterns above, random sizes and geometry; the middle image of the flat band sits on the midpoint
    of its neighbours' coincident positions (T = 0)."""
    rng = np.random.default_rng(seed)
    bands, E = [], []
    for p, pat in enumerate(PATTERNS):
        n = int(rng.integers(1, 40))
        R = np.cumsum(rng.normal(0.0, 0.3, (K + 2, n, 3)), 0)
        if p == len(PATTERNS) - 1:
            R[3] = R[1]                               # R_{k+1} = R_{k-1} around image k = 1: tau = D+ + D- = 0
        bands.append(R)
        E.append(np.asarray(pat, dtype=np.float64))
    return bands, np.array(E)


def _coefficient_forces(bands, E, springs, climb, K=5, branches=None):
    pos, initial, final, image, image_ptr, band_ptr = band_major(bands, K)
    gen = torch.Generator().manual_seed(1)
    force = torch.randn(pos.shape, generator=gen)
    energy = torch.from_numpy(E[:, 1:-1].reshape(-1).astype(np.float32))
    end_energy = torch.from_numpy(E[:, [0, -1]].astype(np.float32))
    sums = ref_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K)
    coef, imax = ref_step(sums, energy, end_energy, torch.from_numpy(springs), climb, branches)
    return pos, force, ref_project(force, pos, initial, final, image, image_ptr, band_ptr, K, coef), imax


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the references
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("climb", [False, True], ids=["plain", "climb"])
def test_coefficient_form_matches_vector_form(climb):
    bands, E = _random_bands(0)
    K = 5
    springs = np.linspace(0.05, 2.0, len(bands))
    branches = set()
    pos, force, got, imax = _coefficient_forces(bands, E, springs, climb, K, branches)
    assert branches == {"up", "down", "extremum, E+ > E-", "extremum, E+ <= E-", "flat", "T = 0"}, branches
    # the vector form on the fp32-rounded band the coefficient form saw
    off = 0
    for b, R in enumerate(bands):
        n = R.shape[1]
        Rb = np.concatenate([R[:1], _np(pos)[off:off + K * n].reshape(K, n, 3), R[-1:]]).astype(np.float32)
        Fb = _np(force)[off:off + K * n].reshape(K, n, 3)
        ref, im = ref_neb_forces(Rb, E[b].astype(np.float32), Fb, springs[b], climb)
        assert im == imax[b], b
        assert np.abs(got[off:off + K * n].reshape(K, n, 3) - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), b
        off += K * n
    assert list(imax[3:5]) == [2, 1]                  # ties: the lowest image


def test_imax_ties_and_the_plain_force_at_t_zero():
    bands, E = _random_bands(1)
    K = 5
    pos, force, got, imax = _coefficient_forces(bands, E, np.full(len(bands), 0.1), True, K)
    n = [R.shape[1] for R in bands]
    start = K * sum(n[:-1])
    # flat band: the first image climbs (a tie), the second has T = 0 and keeps the plain force exactly
    k1 = slice(start + n[-1], start + 2 * n[-1])
    assert imax[-1] == 1 and np.array_equal(got[k1], _np(force)[k1])
    assert not np.array_equal(got[start:start + n[-1]], _np(force)[start:start + n[-1]])


# ---------------------------------------------------------------------------------------------------------------------
# Mueller-Brown surface on a one-atom cluster
# ---------------------------------------------------------------------------------------------------------------------
MB_A = np.array([-200.0, -100.0, -170.0, 15.0])
MB_a = np.array([-1.0, -1.0, -6.5, 0.7])
MB_b = np.array([0.0, 0.0, 11.0, 0.6])
MB_c = np.array([-10.0, -10.0, -6.5, 0.7])
MB_x0 = np.array([1.0, 0.0, -0.5, -1.0])
MB_y0 = np.array([0.0, 0.5, 1.5, 1.0])
MB_SCALE, MB_KZ = 0.01, 5.0                       # eV per MB unit; harmonic z (eV/A^2)


class MuellerBrown(torch.nn.Module):
    """``E = s V_MB(x, y) + kz z^2 / 2`` per atom, summed per graph: the ``build_graph`` / ``forward_graph`` interface that
    ``VerletGraph`` calls, without parameters or a neighbour list.  float64 inside, fp32 out like the real models."""

    def build_graph(self, pos, atomic_number, cell=None, batch=None, skin=0.0):
        n_graphs = 1 if batch is None else int(batch.max()) + 1
        return SimpleNamespace(batch=batch, n_graphs=n_graphs, list_rc=0.0)

    def forward_graph(self, pos, atomic_number, cell, g):
        p = pos.double()
        x, y, z = p[:, 0:1], p[:, 1:2], p[:, 2]
        t = lambda v: torch.as_tensor(v, dtype=torch.float64, device=pos.device)  # noqa: E731
        dx, dy = x - t(MB_x0), y - t(MB_y0)
        e = MB_SCALE * (t(MB_A) * torch.exp(t(MB_a) * dx * dx + t(MB_b) * dx * dy + t(MB_c) * dy * dy)).sum(1) + 0.5 * MB_KZ * z * z
        batch = torch.zeros_like(z, dtype=torch.long) if g.batch is None else g.batch
        return torch.zeros(g.n_graphs, dtype=torch.float64, device=pos.device).index_add(0, batch, e).float(), None, None


def mb_grad_hess(x, y):
    """Gradient and Hessian of ``s V_MB`` at ``(x, y)`` (float64)."""
    dx, dy = x - MB_x0, y - MB_y0
    ex = MB_SCALE * MB_A * np.exp(MB_a * dx * dx + MB_b * dx * dy + MB_c * dy * dy)
    ux, uy = 2 * MB_a * dx + MB_b * dy, MB_b * dx + 2 * MB_c * dy
    g = np.array([(ex * ux).sum(), (ex * uy).sum()])
    h = np.array([[(ex * (ux * ux + 2 * MB_a)).sum(), (ex * (ux * uy + MB_b)).sum()],
                  [(ex * (ux * uy + MB_b)).sum(), (ex * (uy * uy + 2 * MB_c)).sum()]])
    return g, h


def mb_stationary(x, y):
    """Newton's method on the gradient from ``(x, y)``: the stationary point and its Hessian eigenvalues."""
    p = np.array([x, y], dtype=np.float64)
    for _ in range(100):
        g, h = mb_grad_hess(*p)
        p = p - np.linalg.solve(h, g)
    g, h = mb_grad_hess(*p)
    assert np.abs(g).max() < 1e-12
    return p, np.linalg.eigvalsh(h)


MB_MIN_A, MB_MIN_C, MB_SADDLE = (-0.558, 1.442), (-0.050, 0.467), (-0.822, 0.624)
MB_KW = dict(n_images=7, climb=True, fmax=2e-3, max_steps=3000, spring_constant=0.5)


def _mb_endpoints():
    (a, ea), (c, ec) = mb_stationary(*MB_MIN_A), mb_stationary(*MB_MIN_C)
    assert (ea > 0).all() and (ec > 0).all()
    return np.array([[a[0], a[1], 0.0]]), np.array([[c[0], c[1], 0.0]])


def _check_mb_saddle(images, energies, st, fmax):
    """The climbing image sits on the Newton saddle within ``|F| / lambda_min``: ``|F| < fmax`` at convergence (the climbing
    force is the model force reflected along the tangent, so it has the same norm), the Hessian's smallest eigenvalue
    magnitude turns that into a distance; plus the fp32 rounding of positions and forces."""
    s, eig = mb_stationary(*MB_SADDLE)
    assert eig[0] < 0 < eig[1] and np.abs(s - MB_SADDLE).max() < 2e-3
    tol = 1.5 * fmax / np.abs(eig).min() + 1e-5
    im = int(st["imax"][-1, 0])
    x = _np(images)[im - 1, 0].astype(np.float64)
    assert bool(st["converged"][0]), st["steps"]
    assert np.abs(x[:2] - s).max() < tol, (x, s, tol)
    assert abs(x[2]) < tol
    # the straight line between the minima misses the saddle: projection and spring carried the band there
    a, c = _mb_endpoints()
    u = (c[0, :2] - a[0, :2]) / np.linalg.norm(c[0, :2] - a[0, :2])
    d = s - a[0, :2]
    assert np.linalg.norm(d - np.dot(d, u) * u) > 50 * tol
    e = _np(energies)[0]
    assert int(np.argmax(e)) == im and e[im] == e.max()


def test_emulated_mueller_brown_climbing_image_finds_the_saddle(emu_neb):
    a, c = _mb_endpoints()
    st = {}
    images, energies = neb_device(MuellerBrown(), [1], a, c, None, stats=st, device="cpu", **MB_KW)
    print("Mueller-Brown (CPU emulator): steps", st["steps"].tolist())
    assert images.shape == (7, 1, 3) and energies.shape == (1, 9)
    _check_mb_saddle(images, energies, st, MB_KW["fmax"])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the driver over the kernel emulator
# ---------------------------------------------------------------------------------------------------------------------
def _two_lattice_bands():
    """Two periodic bands of different sizes (64 and 59 atoms): a rattled lattice and the same lattice with one atom moved
    by 1 A and every atom rattled again."""
    pos, Z, cell, batch = _cpu_systems((41, 42))
    keep = np.ones(len(Z), dtype=bool)
    keep[np.flatnonzero(batch == 1)[-5:]] = False
    pos, Z, batch = pos[keep], Z[keep], batch[keep]
    rng = np.random.default_rng(3)
    final = pos + rng.normal(0.0, 0.05, pos.shape).astype(np.float32)
    for b in (0, 1):
        final[np.flatnonzero(batch == b)[7], 0] += 1.0
    return pos, final, Z, cell, batch


def image_evaluator(model, Z, h, dev):
    """``evaluate(configs [m,n,3]) -> (E [m], F [m,n,3])`` one configuration at a time at the fp32-rounded geometry."""
    Zt = torch.as_tensor(Z).long().to(dev)

    def evaluate(xs):
        E, F = [], []
        for x in xs:
            out = model.energy_forces_virial(H.Data(pos=torch.from_numpy(np.asarray(x, dtype=np.float32)).to(dev), atomic_number=Zt,
                                                    cell=torch.from_numpy(np.asarray(h, dtype=np.float32)).reshape(1, 3, 3).to(dev)))
            E.append(float(out["energy"][0]))
            F.append(_np(out["forces"]).astype(np.float64))
        return np.array(E), np.array(F)
    return evaluate


def host_neb(model, x0, x1, R0, Z, h, dev, k, climb, steps, **kw):
    """ASE's NEB + FIRE on one band: ``host_fire`` on the concatenated interior images with ``ref_neb_forces`` as the force.
    Returns ``(images [K,n,3], [(dt, alpha, n_pos) after each step])``."""
    K, n = R0.shape[:2]
    ev = image_evaluator(model, Z, h, dev)
    E_ends, _ = ev([x0, x1])

    def evaluate(x, _h):
        R = x.reshape(K, n, 3)
        E, F = ev(R)
        f, _ = ref_neb_forces(np.concatenate([x0[None], R, x1[None]]), np.concatenate([[E_ends[0]], E, [E_ends[1]]]), F, k, climb)
        return f.reshape(K * n, 3), np.zeros((3, 3))
    x, _, trace = host_fire(evaluate, R0.reshape(K * n, 3).astype(np.float64), h, steps, False, **kw)
    return x.reshape(K, n, 3), trace


def check_against_host_neb(model, x0, x1, Z, cell, batch, dev, K, springs, climb, steps, **kw):
    st = {}
    images, energies = neb_device(model, Z, x0, x1, cell, n_images=K, batch=batch, spring_constant=springs, climb=climb,
                                  max_steps=steps, stats=st, device=dev, **kw)
    assert st["steps"].tolist() == [steps] * len(springs), "the comparison wants every band still moving"
    # the starting band the driver built (max_steps = 0 returns it untouched)
    start, _ = neb_device(model, Z, x0, x1, cell, n_images=K, batch=batch, max_steps=0, device=dev)
    for b, k in enumerate(springs):
        sl = batch == b
        R, trace = host_neb(model, x0[sl].astype(np.float64), _np(x1)[sl].astype(np.float64), _np(start)[:, sl], Z[sl], cell[b], dev,
                            k, climb, steps, **kw)
        assert len(trace) == steps
        tr = np.array(trace)
        assert np.allclose(_np(st["dt"])[:steps, b], tr[:, 0], rtol=1e-12, atol=0)
        assert np.allclose(_np(st["alpha"])[:steps, b], tr[:, 1], rtol=1e-12, atol=0)
        assert np.array_equal(_np(st["n_pos"])[:steps, b], tr[:, 2].astype(np.int32))
        assert np.abs(_np(images)[:, sl] - R).max() < 1e-4, b
    return st


def test_emulated_driver_matches_host_neb_and_fire(emu_neb):
    model = _cpu_model()
    x0, x1, Z, cell, batch = _two_lattice_bands()
    for climb in (False, True):
        check_against_host_neb(model, x0, x1, Z, cell, batch, "cpu", 3, [0.1, 0.7], climb, 8, fmax=1e-6)


def test_emulated_periodic_re_expression(emu_neb):
    model = _cpu_model()
    x0, x1, Z, cell, batch = _two_lattice_bands()
    kw = dict(n_images=3, batch=batch, max_steps=3, device="cpu")
    ref_images, ref_e = neb_device(model, Z, x0, x1, cell, **kw)
    # whole lattice vectors added to some atoms of the final configuration
    rng = np.random.default_rng(5)
    shifts = rng.integers(-2, 3, (len(Z), 3)).astype(np.float64)
    x1s = (x1 + np.einsum("ni,nij->nj", shifts, cell.astype(np.float64)[batch])).astype(np.float32)
    images, e = neb_device(model, Z, x0, x1s, cell, **kw)
    assert float((images - ref_images).abs().max()) < 1e-5 and float((e - ref_e).abs().max()) < 1e-5
    # images given wrapped into the cell: re-expressed along the band, they are the unwrapped ones
    h = cell.astype(np.float64)[batch]
    s = np.einsum("kni,nij->knj", _np(ref_images).astype(np.float64), np.linalg.inv(h))
    wrapped = np.einsum("kni,nij->knj", s - np.floor(s), h)
    assert np.abs(wrapped - _np(ref_images)).max() > 1.0
    a, ea = neb_device(model, Z, x0, x1s, cell, images=wrapped, **dict(kw, max_steps=0))
    b, eb = neb_device(model, Z, x0, x1, cell, images=ref_images, **dict(kw, max_steps=0))
    assert float((a - b).abs().max()) < 1e-5 and float((ea - eb).abs().max()) < 1e-5


def test_emulated_stats_and_max_steps_zero(emu_neb):
    model = _cpu_model()
    x0, x1, Z, cell, batch = _two_lattice_bands()
    st = {}
    images, e = neb_device(model, Z, x0, x1, cell, n_images=4, batch=batch, max_steps=3, fmax=1e-6, skin=0.5, stats=st, device="cpu")
    assert images.shape == (4, len(Z), 3) and images.dtype == torch.float32 and e.shape == (2, 6) and e.dtype == torch.float32
    for k, shape, dtype in (("energy", (4, 2, 4), torch.float32), ("fmax", (4, 2), torch.float64), ("imax", (4, 2), torch.int32),
                            ("dt", (4, 2), torch.float64), ("alpha", (4, 2), torch.float64), ("n_pos", (4, 2), torch.int32),
                            ("converged", (2,), torch.bool), ("steps", (2,), torch.int32)):
        assert st[k].shape == shape and st[k].dtype == dtype, k
    assert st["steps"].tolist() == [3, 3] and st["builds"] + st["reuses"] == 4
    assert torch.equal(st["energy"][-1], e[:, 1:-1])
    assert ((st["imax"] >= 1) & (st["imax"] <= 4)).all()
    assert torch.equal(st["imax"][-1].long(), e[:, 1:-1].argmax(1) + 1)
    # max_steps = 0: the linear interpolation (of the re-expressed final configuration: the same up to rounding), untouched
    st0 = {}
    p0, e0 = neb_device(model, Z, x0, x1, cell, n_images=4, batch=batch, max_steps=0, stats=st0, device="cpu")
    lin = x0[None] + (np.arange(1, 5) / 5.0)[:, None, None] * (x1 - x0)[None].astype(np.float64)
    assert float((p0.double() - torch.from_numpy(lin)).abs().max()) < 1e-6
    assert st0["steps"].tolist() == [0, 0] and st0["energy"].shape == (1, 2, 4) and torch.equal(e0[:, 0], e[:, 0])


def _bad_cases():
    x0 = np.zeros((4, 3))
    x0[:, 0] = np.arange(4) * 1.5
    x1 = x0 + 0.5
    return [
        dict(fmax=0.0), dict(dt=0.0), dict(dt=0.5, dt_max=0.4), dict(max_step=0.0), dict(max_steps=-1),
        dict(n_images=0), dict(n_images=2.5), dict(spring_constant=0.0), dict(spring_constant=-1.0),
        dict(spring_constant=float("nan")), dict(spring_constant=float("inf")), dict(spring_constant=[0.1, 0.1]),
        dict(initial=x0[:3]), dict(final=x1.reshape(3, 4)), dict(images=np.zeros((4, 4, 3))),
        dict(initial=np.where(np.arange(12).reshape(4, 3) == 5, np.nan, x0)), dict(final=x1 + np.inf),
        dict(images=np.full((5, 4, 3), np.nan)),
        dict(final=x0.copy()),                                                # initial and final coincide
        dict(final=x0 + 10.0 * np.array([1.0, 0.0, 0.0])),                    # ... once re-expressed in the cell
        dict(images=np.stack([x0 + 0.1 * k for k in (1, 2, 2, 3, 4)])),       # two consecutive images coincide
        dict(images=np.stack([x0] + [x0 + 0.1 * k for k in (2, 3, 4, 5)])),   # the first image is the initial one
        dict(batch=[0, 0, 1, 0]), dict(batch=[0, 0, 2, 2]), dict(cell=np.zeros((2, 3, 3)) + np.eye(3)),
        dict(cell=np.diag([10.0, 10.0, 0.0])), dict(cell=np.full((3, 3), np.nan)),
    ]


@pytest.mark.parametrize("bad", _bad_cases())
def test_validation_errors(bad):
    x0 = np.zeros((4, 3))
    x0[:, 0] = np.arange(4) * 1.5
    args = dict(initial=x0, final=x0 + 0.5, cell=10.0 * np.eye(3))
    args.update(bad)
    with pytest.raises(ValueError):
        neb_device(None, [8, 1, 1, 8], args.pop("initial"), args.pop("final"), args.pop("cell"), device="cpu", **args)


# ---------------------------------------------------------------------------------------------------------------------
# kernel level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _gpu_layout(sizes, K, seed):
    rng = np.random.default_rng(seed)
    bands = [np.cumsum(rng.normal(0.0, 0.3, (K + 2, n, 3)), 0) + 20.0 * rng.normal(size=(1, 1, 3)) for n in sizes]
    return [t.to(DEV) for t in band_major(bands, K)]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,K", [([200_000], 5), ([1 + (53 * b) % 900 for b in range(300)], 4)], ids=["B1-1e6", "B300"])
def test_reduce_matches_float64_and_is_deterministic(sizes, K):
    pos, initial, final, image, image_ptr, band_ptr = _gpu_layout(sizes, K, len(sizes))
    force = torch.randn(pos.shape, generator=torch.Generator().manual_seed(2)).to(DEV)
    got = ops.neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K)
    ref = ref_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K)
    n_per_image = pos.size(0) / (len(sizes) * K)
    assert np.abs(_np(got) - ref).max() <= 1e-12 * np.abs(ref).max() * max(1.0, n_per_image) ** 0.5
    assert torch.equal(got, ops.neb_reduce(pos, force, initial, final, image, image_ptr, band_ptr, K))


@pytest.mark.gpu
def test_empty_launches_are_no_ops():
    z3, zi = torch.zeros(0, 3, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV)
    one = torch.zeros(1, dtype=torch.int32, device=DEV)
    assert ops.neb_reduce(z3, z3.clone(), z3.clone(), z3.clone(), zi, one, one, 3).shape == (0, 5)
    d0 = torch.zeros(0, dtype=torch.float64, device=DEV)
    coef = torch.zeros(0, 2, dtype=torch.float64, device=DEV)
    ops.neb_step(torch.zeros(0, 5, dtype=torch.float64, device=DEV), torch.zeros(0, device=DEV), torch.zeros(0, 2, device=DEV), d0,
                 True, coef, zi.clone())
    ops.neb_project(z3, z3.clone(), z3.clone(), z3.clone(), zi, one, one, 3, coef)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("climb", [False, True], ids=["plain", "climb"])
def test_step_matches_float64_in_every_branch(climb):
    bands, E = _random_bands(2)
    K = 5
    reps = 40                                          # many bands per pattern, random sums
    rng = np.random.default_rng(3)
    E = np.tile(E, (reps, 1)).astype(np.float32)
    B = len(E)
    sums = np.abs(rng.normal(size=(B * K, 5)))
    sums[:, 2] = rng.normal(size=B * K)
    sums[:, 3:] = rng.normal(size=(B * K, 2))
    sums[4 * K::5 * K, :] = 0.0                        # T = 0 in image 0 of every fifth band
    springs = rng.uniform(0.05, 2.0, B)
    coef = torch.full((B * K, 2), -7.0, dtype=torch.float64, device=DEV)
    imax = torch.zeros(B, dtype=torch.int32, device=DEV)
    energy, end_energy = torch.from_numpy(E[:, 1:-1].reshape(-1).copy()).to(DEV), torch.from_numpy(E[:, [0, -1]].copy()).to(DEV)
    ops.neb_step(torch.from_numpy(sums).to(DEV), energy, end_energy, torch.from_numpy(springs).to(DEV), climb, coef, imax)
    branches = set()
    ref_c, ref_i = ref_step(sums, energy, end_energy, springs, climb, branches)
    assert len(branches) == 6
    assert np.array_equal(_np(imax), ref_i)
    assert np.allclose(_np(coef), ref_c, rtol=1e-12, atol=1e-300)


@pytest.mark.gpu
def test_project_matches_torch_float64():
    sizes, K = [5000, 1, 20_001, 333], 3
    pos, initial, final, image, image_ptr, band_ptr = _gpu_layout(sizes, K, 7)
    gen = torch.Generator().manual_seed(4)
    force = torch.randn(pos.shape, generator=gen).to(DEV)
    coef = torch.randn(len(sizes) * K, 2, generator=gen, dtype=torch.float64).to(DEV)
    got = force.clone()
    ops.neb_project(got, pos, initial, final, image, image_ptr, band_ptr, K, coef)
    x, prev, nxt = (torch.from_numpy(a).to(DEV) for a in _neighbours(pos, initial, final, image, image_ptr, band_ptr, K))
    c = coef[image.long()]
    ref = force.double() + c[:, :1] * (nxt - x) + c[:, 1:] * (x - prev)
    assert float((got.double() - ref).abs().max()) <= 6e-8 * float(ref.abs().max())


# ---------------------------------------------------------------------------------------------------------------------
# model level (GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mueller_brown_bands_find_the_saddle_alone_and_together():
    a, c = _mb_endpoints()
    shifted = a + np.array([[0.0, 0.0, 0.3]])                   # an endpoint off the z minimum: a different band
    ends = [(a, c, 0.5), (c, a, 0.5), (a, c, 1.5), (shifted, c, 0.8)]
    x0 = np.concatenate([e[0] for e in ends])
    x1 = np.concatenate([e[1] for e in ends])
    springs = [e[2] for e in ends]
    kw = dict(MB_KW)
    kw.pop("spring_constant")
    st = {}
    images, energies = neb_device(MuellerBrown(), [1] * 4, x0, x1, None, batch=np.arange(4), spring_constant=springs, stats=st,
                                  device=DEV, **kw)
    print("Mueller-Brown (B200): steps", st["steps"].tolist())
    for b, (p, q, k) in enumerate(ends):
        sb = {}
        ib, eb = neb_device(MuellerBrown(), [1], p, q, None, spring_constant=k, stats=sb, device=DEV, **kw)
        assert int(sb["steps"][0]) == int(st["steps"][b])
        assert float((ib[:, 0] - images[:, b]).abs().max()) < 1e-6 and float((eb[0] - energies[b]).abs().max()) < 1e-6
        _check_mb_saddle(ib, eb, sb, kw["fmax"])


def _water_bands(seeds, rattle=0.05):
    """Periodic 192-atom C1 water boxes: the box rattled with two seeds gives the endpoints of one band."""
    x0, x1, Zs, cells = [], [], [], []
    for s in seeds:
        p, z, c = synthetic.water_box(4, seed=s)
        x0.append(p + np.random.default_rng(100 + s).normal(0.0, rattle, p.shape).astype(np.float32))
        x1.append(p + np.random.default_rng(200 + s).normal(0.0, rattle, p.shape).astype(np.float32))
        Zs.append(z)
        cells.append(c)
    return (np.concatenate(x0), np.concatenate(x1), np.concatenate(Zs), np.stack(cells),
            np.repeat(np.arange(len(seeds)), [len(z) for z in Zs]))


@pytest.mark.gpu
def test_driver_matches_host_neb_and_fire():
    model = _water_model()
    x0, x1, Z, cell, batch = _water_bands((1, 2))
    for climb in (False, True):
        check_against_host_neb(model, x0, x1, Z, cell, batch, DEV, 3, [0.1, 0.5], climb, 15, fmax=1e-6)


@pytest.mark.gpu
def test_a_lone_band_matches_the_batch_and_cuda_graph_matches_eager():
    model = _water_model()
    x0, x1, Z, cell, batch = _water_bands((3, 4, 5))
    kw = dict(n_images=3, climb=True, fmax=1e-6, max_steps=10, device=DEV)
    ib, eb = neb_device(model, Z, x0, x1, cell, batch=batch, **kw)
    sl = batch == 1
    i1, e1 = neb_device(model, Z[sl], x0[sl], x1[sl], cell[1], **kw)
    assert float((i1 - ib[:, torch.from_numpy(sl).to(DEV)]).abs().max()) < 1e-5
    assert float((e1[0] - eb[1]).abs().max()) < 1e-5 * max(1.0, float(eb.abs().max()))
    runs = {}
    for cg in (False, True):
        st = {}
        runs[cg] = neb_device(model, Z, x0, x1, cell, batch=batch, skin=0.8, cuda_graph=cg, stats=st, **dict(kw, max_steps=30)) + (st,)
    (p0, e0, s0), (p1, e1_, s1) = runs[False], runs[True]
    assert s1["builds"] == s0["builds"] and s1["reuses"] > 0
    assert float((p1 - p0).abs().max()) < 1e-5
    assert float((e1_ - e0).abs().max()) < 1e-5 * max(1.0, float(e0.abs().max()))


@pytest.mark.gpu
def test_a_band_that_starts_converged_is_returned_unchanged():
    model = _water_model()
    x0, x1, Z, cell, batch = _water_bands((6, 7))
    kw = dict(n_images=3, batch=batch, climb=True, device=DEV)
    st0 = {}
    p0, _ = neb_device(model, Z, x0, x1, cell, max_steps=0, stats=st0, **kw)
    f0 = _np(st0["fmax"][0])
    k = int(np.argmin(f0))
    fmax = float(f0[k]) * 1.01
    assert f0[1 - k] > fmax
    st = {}
    p, _ = neb_device(model, Z, x0, x1, cell, fmax=fmax, max_steps=20, stats=st, **kw)
    sl = torch.from_numpy(batch == k).to(DEV)
    assert torch.equal(p[:, sl], p0[:, sl])
    assert int(st["steps"][k]) == 0 and int(st["steps"][1 - k]) == 20 and bool(st["converged"][k])


@pytest.mark.gpu
def test_climbing_image_between_relaxed_boxes_is_a_stationary_point():
    model = _water_model()
    x0, x1, Z, cell, _ = _water_bands((8,), rattle=0.15)
    # relax both endpoints together, as two replicas
    pos = np.concatenate([x0, x1])
    rb = np.repeat([0, 1], len(Z))
    st_r0 = {}
    fire_relax_device(model, np.concatenate([Z, Z]), pos, np.stack([cell[0], cell[0]]), max_steps=0, batch=rb, stats=st_r0, device=DEV)
    st_r = {}
    p, _, _ = fire_relax_device(model, np.concatenate([Z, Z]), pos, np.stack([cell[0], cell[0]]), fmax=0.1 * float(st_r0["fmax"][0].min()),
                                max_steps=3000, batch=rb, skin=0.5, stats=st_r, device=DEV)
    assert bool(st_r["converged"].all())
    a, b = _np(p[: len(Z)]), _np(p[len(Z):])
    kw = dict(n_images=3, climb=True, device=DEV, skin=0.5)
    st0 = {}
    neb_device(model, Z, a, b, cell[0], max_steps=0, stats=st0, **kw)
    fmax = 0.2 * float(st0["fmax"][0, 0])
    st = {}
    # 779 steps on a B200; the budget leaves room for the order of reductions to change the trajectory
    images, energies = neb_device(model, Z, a, b, cell[0], fmax=fmax, max_steps=3000, stats=st, **kw)
    print(f"CI-NEB between relaxed boxes: fmax {fmax:.3e}, steps {st['steps'].tolist()}, builds {st['builds']} reuses {st['reuses']}, "
          f"endpoint relaxation steps {st_r['steps'].tolist()}")
    assert bool(st["converged"][0])
    im = int(st["imax"][-1, 0])
    out = model.energy_forces_virial(H.Data(pos=images[im - 1], atomic_number=torch.from_numpy(Z).to(DEV),
                                            cell=torch.from_numpy(cell[0]).reshape(1, 3, 3).to(DEV)))
    f = _np(out["forces"]).astype(np.float64)
    assert np.sqrt((f * f).sum(1).max()) < fmax * 1.01
    # the highest interior image (this random-weight model's relaxed boxes need not lie below the path between them)
    e = _np(energies)[0]
    assert e[im] == e[1:-1].max()
