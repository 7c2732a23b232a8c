"""The boundary between ``ops`` and the C ABI: how device pointers cross ctypes (``_lib.P``), how each launch is counted
and timed for ``bench.py`` (``ops.LAUNCHES`` / ``ops.TIMERS``), and that the wrappers with checks of their own refuse bad
arguments before anything is launched."""
import ctypes
import re
from types import SimpleNamespace

import pytest
import torch

from hermnet_b200 import _lib, ops, tileplan
from tests.util import edge_inputs, frozen_model, lattice_system

DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------------------------------
# pointer conversion (CPU)
# ---------------------------------------------------------------------------------------------------------------------
class _FarPointer:
    def data_ptr(self):
        return 2 ** 40 + 16


def test_pointer_argtype_converts_tensors_and_passes_none_and_void_pointers():
    assert _lib.P.from_param(None) is None
    t = torch.zeros(4)
    assert _lib.P.from_param(t).value == t.data_ptr()
    far = _lib.P.from_param(_FarPointer())
    assert isinstance(far, ctypes.c_void_p) and far.value == 2 ** 40 + 16        # no truncation to a 32-bit C int
    vp = ctypes.c_void_p(1234)
    assert _lib.P.from_param(vp) is vp


@pytest.mark.parametrize("bad", [1.5, "0x1000"])
def test_pointer_argtype_rejects_other_objects(bad):
    with pytest.raises(TypeError):
        _lib.P.from_param(bad)


# ---------------------------------------------------------------------------------------------------------------------
# launch and timer accounting (GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _accounting(fn):
    """``(launches added, {timer name: entries})`` of one call of ``fn`` with the timers on."""
    ops.TIMERS = {}
    n0 = ops.LAUNCHES["n"]
    try:
        fn()
        torch.cuda.synchronize()
        return ops.LAUNCHES["n"] - n0, {k: len(v) for k, v in ops.TIMERS.items()}
    finally:
        ops.TIMERS = None


def _cluster(n, spacing):
    pos = torch.arange(n, dtype=torch.float32).view(n, 1).repeat(1, 3) * spacing
    return pos.to(DEV), torch.tensor([0, n], dtype=torch.int32, device=DEV)


@pytest.mark.gpu
def test_plain_wrapper_is_one_timed_launch():
    X = torch.randn(5, 8, device=DEV)
    idx = torch.tensor([4, 0, 2], dtype=torch.int32, device=DEV)
    assert _accounting(lambda: ops.gather_rows(X, idx)) == (1, {"gather_rows": 1})


@pytest.mark.gpu
def test_graph_builders_are_counted_untimed():
    pos, gptr = _cluster(6, 1.0)
    assert _accounting(lambda: ops.radius_graph(pos, None, gptr, 1.9)) == (7, {})
    far, gptr = _cluster(3, 10.0)
    assert _accounting(lambda: ops.radius_graph(far, None, gptr, 1.9)) == (6, {})        # no edges: no fill launch
    keys = torch.tensor([2, 0, 1, 0, 2], dtype=torch.int32, device=DEV)
    assert _accounting(lambda: ops.sort_by_key(keys, 3)) == (1, {})


@pytest.mark.gpu
def test_triplet_kernels_are_neither_counted_nor_timed():
    pos, gptr = _cluster(6, 1.0)
    rowptr, col, _ = ops.radius_graph(pos, None, gptr, 2.5)
    out = {}
    assert _accounting(lambda: out.setdefault("t", ops.triplets(rowptr, col))) == (0, {})
    trip_ptr, e1, e2 = out["t"]
    assert e1.numel() > 0
    m_vec = torch.randn(col.numel(), 3, 4, device=DEV)
    assert _accounting(lambda: ops.triplet_dots(m_vec, trip_ptr, e1, e2)) == (0, {})


@pytest.mark.gpu
def test_shared_timer_windows():
    x = torch.randn(7, 64, device=DEV)
    assert _accounting(lambda: ops.layernorm_fwd(x, 1e-5)) == (1, {"node_elementwise": 1})
    v12 = torch.randn(7, 3, 128, device=DEV)
    vdot, xcat = torch.empty(7, 64, device=DEV), torch.empty(7, 128, device=DEV)
    assert _accounting(lambda: ops.node_mid(v12, vdot, xcat)) == (1, {"node_elementwise": 1})
    W1, b1 = torch.randn(32, 64, device=DEV), torch.randn(32, device=DEV)
    W2, b2 = torch.randn(32, device=DEV), torch.randn(1, device=DEV)
    assert _accounting(lambda: ops.readout_fwd(x, W1, b1, W2, b2)) == (1, {"readout": 1})
    geom = torch.rand(9, 4, device=DEV) + 1.0
    assert _accounting(lambda: ops.tc_basis_index(geom, 0.2, 20)) == (1, {"tc_plan": 1})


@pytest.mark.gpu
def test_tc_plan_sort_is_one_counted_tc_plan_window():
    E, K = 40, 20
    in_ptr = torch.tensor([0, 15, E], dtype=torch.int32, device=DEV)
    kc = (torch.arange(E, dtype=torch.int32, device=DEV) * 7) % K
    sub = torch.zeros(E, dtype=torch.int32, device=DEV)
    assert _accounting(lambda: ops.tc_plan_sort(in_ptr, None, kc, sub, 2, 1, K)) == (1, {"tc_plan": 1})


@pytest.mark.gpu
def test_fire_reduce_counts_two_kernels():
    n = 10
    force, vel = torch.randn(n, 3, device=DEV), torch.randn(n, 3, device=DEV)
    replica = torch.zeros(n, dtype=torch.int32, device=DEV)
    replica_ptr = torch.tensor([0, n], dtype=torch.int32, device=DEV)
    assert _accounting(lambda: ops.opt_fire_reduce(force, vel, None, replica, replica_ptr)) == (2, {"opt_fire_reduce": 1})


@pytest.mark.gpu
def test_gemm_timer_name_keyed_on_shape_when_asked():
    a = torch.randn(16, 32, device=DEV)
    w_hi, w_lo = ops.split_tf32(torch.randn(64, 32, device=DEV))
    assert _accounting(lambda: ops.gemm_tf32x3_ex(a, w_hi, w_lo, None)) == (1, {"gemm_tf32x3": 1})
    ops.GEMM_SHAPES = True
    try:
        assert _accounting(lambda: ops.gemm_tf32x3_ex(a, w_hi, w_lo, None)) == (1, {"gemm_tf32x3[16x32->64,mode0]": 1})
    finally:
        ops.GEMM_SHAPES = False


@pytest.mark.gpu
def test_tensor_core_edge_kernels_share_the_painn_edge_timers():
    pos, Z, cell = lattice_system(6, [1, 8], 5)
    pos, Z, cell = pos.to(DEV), Z.to(DEV), cell.to(DEV)
    model = frozen_model("HVNet", ["H", "O"], 128, 20, DEV)
    g = model.build_graph(pos, Z, cell)
    p, geom, xh, vec, Wt, bias, off, g_dx, g_dvec = edge_inputs(model, g, pos, cell)
    dst, src = tileplan.plans_of(g, geom, p.inv_rc, p.num_rbf, want_src=True)
    dst.update_windows(geom, p.inv_rc, p.num_rbf)
    src.update_windows(geom, p.inv_rc, p.num_rbf)
    wsplit, wscale = ops.tc_split_weights(Wt)
    assert _accounting(lambda: ops.tc_edge_fwd(p, dst, xh, vec, geom, wsplit, wscale, bias, off, p.n_rows)) == \
        (1, {"painn_edge_fwd": 1})
    assert _accounting(lambda: ops.tc_edge_bwd_dst(p, dst, xh, vec, geom, wsplit, wscale, bias, off, g_dx, g_dvec)) == \
        (1, {"painn_edge_bwd_dst": 1})
    assert _accounting(lambda: ops.tc_edge_bwd_src(p, src, xh, vec, geom, wsplit, wscale, bias, off, g_dx, g_dvec)) == \
        (1, {"painn_edge_bwd_src": 1})


# ---------------------------------------------------------------------------------------------------------------------
# rejection before launch (GPU): wrappers whose checks go beyond device, layout and dtype
# ---------------------------------------------------------------------------------------------------------------------
def _f(*shape, dtype=torch.float32):
    return torch.zeros(shape, dtype=dtype, device=DEV)


def _i(*shape, dtype=torch.int32):
    return torch.zeros(shape, dtype=dtype, device=DEV)


def _edge_virial_atom(bad):
    E = 6
    g = SimpleNamespace(n_edges=E, n_atoms=4)
    geom = {"dtype": _f(E, 4, dtype=torch.float64), "shape": _f(E + 1, 4)}[bad]
    ops.edge_virial_atom(geom, _f(E, 4), g)


def _painn_edge_bwd_w(bad):
    E, F, K = 6, 64, 16
    p = ops.EdgeParams(4, 4, 1, F, K, 5, 0.2, -10.0, 0, 1)
    p.live = {"dtype": _i(E, dtype=torch.uint8), "live": _i(E), "live_len": _i(E + 1, dtype=torch.uint8)}[bad]
    xh = _f(4, 3 * F, dtype=torch.float64 if bad == "dtype" else torch.float32)
    ops.painn_edge_bwd_w(p, xh, _f(4, 3, F), _f(E, 4), None, _f(K), _f(4, F), _f(4, 3, F))


def _tc_tile_windows(bad):
    E = 6
    live = {"live": _i(E), "live_len": _i(E + 1, dtype=torch.uint8)}[bad]
    ops.tc_tile_windows(None, _f(E, 4), 0.2, 16, live)


def _halo_pack(bad):
    F, n = 32, 4
    x = _f(n, F, dtype=torch.float64 if bad == "dtype" else torch.float32)
    base = _i(2, dtype=torch.int32 if bad == "base" else torch.int64)
    ops.halo_pack(x, _f(n, 3 * F), _i(n), _i(n), _i(n), base)


def _md_langevin_baoa(bad):
    n, G = 5, 2
    pos = _f(n, 3, dtype=torch.float64 if bad == "dtype" else torch.float32)
    vel = _f(n, 2) if bad == "shape" else _f(n, 3)
    kT = _f(G + 1) if bad == "shape2" else _f(G)
    seed = _i(G, dtype=torch.int32 if bad == "dtype2" else torch.int64)
    ops.md_langevin_baoa(pos, vel, _f(n, 3), _f(n), _i(n), _i(G + 1), kT, seed, _i(1, dtype=torch.int64), 0.9, 0.1, 1.0)


def _md_kick(bad):
    n = 5
    vel = _f(n, 3, dtype=torch.float64 if bad == "dtype" else torch.float32)
    step = _i(2 if bad == "shape" else 1, dtype=torch.int64)
    ops.md_kick(vel, _f(n, 3), _f(n), 0.5, _f(n), step)


def _md_scr_barostat(bad):
    G = 3
    cell = _f(G, 3, 3, dtype=torch.float64 if bad == "dtype" else torch.float32)
    virial = _f(G, 3, 2) if bad == "shape" else _f(G, 3, 3)
    ops.md_scr_barostat(cell, _f(G), virial, _f(G), _f(G), _f(G), _i(G, dtype=torch.int64), _i(1, dtype=torch.int64), 1.0, 100.0,
                        _f(G), _f(G))


def _md_affine_scale(bad):
    n = 5
    replica = _i(n, dtype=torch.int64 if bad == "dtype" else torch.int32)
    vel = _f(n, 2) if bad == "shape" else _f(n, 3)
    ops.md_affine_scale(_f(n, 3), vel, replica, _f(1))


def _opt_fire_reduce(bad):
    n, G = 5, 2
    A = {"dtype": _f(G, 3, 3), "shape": _f(G, 3, 2, dtype=torch.float64)}[bad]
    ops.opt_fire_reduce(_f(n, 3), _f(n, 3), A, _i(n), _i(G + 1))


def _opt_fire_step(bad):
    G = 2
    d = lambda *s: _f(*s, dtype=torch.float64)
    dt = _f(G) if bad == "dtype" else d(G)
    coef = d(G, 2) if bad == "shape" else d(G, 3)
    virial = None if bad == "missing" else _f(G, 3, 3)
    ops.opt_fire_step(d(G, 4), virial, _f(G, 3, 3), d(G, 3, 3), d(G, 3, 3), d(G, 3, 3), d(G, 3, 3), d(G), d(G), dt, d(G),
                      _i(G), _i(G), _i(G), 0.05, 1.0, 0.2, True, coef, d(G), _i(1))


def _opt_fire_update(bad):
    n, G = 5, 2
    d = lambda *s: _f(*s, dtype=torch.float64)
    coef = _f(G, 3) if bad == "dtype" else d(G, 3)
    x = None if bad == "missing" else _f(n, 3)
    ops.opt_fire_update(x, _f(n, 3), _f(n, 3), _f(n, 3), d(G, 3, 3), d(G, 3, 3), _i(n), _i(G), coef)


def _gemm_tf32x3_ex(bad):
    M, K, N = 16, 32, 64
    a = _f(M, K, dtype=torch.float64 if bad == "dtype" else torch.float32)
    out = _f(N, M).t() if bad == "layout" else None
    ops.gemm_tf32x3_ex(a, _f(N, K), _f(N, K), None, out)


REJECT = [
    ("edge_virial_atom", _edge_virial_atom, "dtype", RuntimeError),
    ("edge_virial_atom", _edge_virial_atom, "shape", RuntimeError),
    ("painn_edge_bwd_w", _painn_edge_bwd_w, "dtype", RuntimeError),
    ("painn_edge_bwd_w", _painn_edge_bwd_w, "live", TypeError),
    ("painn_edge_bwd_w", _painn_edge_bwd_w, "live_len", TypeError),
    ("tc_tile_windows", _tc_tile_windows, "live", TypeError),
    ("tc_tile_windows", _tc_tile_windows, "live_len", TypeError),
    ("halo_pack", _halo_pack, "dtype", RuntimeError),
    ("halo_pack", _halo_pack, "base", TypeError),
    ("md_langevin_baoa", _md_langevin_baoa, "dtype", RuntimeError),
    ("md_langevin_baoa", _md_langevin_baoa, "dtype2", RuntimeError),
    ("md_langevin_baoa", _md_langevin_baoa, "shape", RuntimeError),
    ("md_langevin_baoa", _md_langevin_baoa, "shape2", RuntimeError),
    ("md_kick", _md_kick, "dtype", RuntimeError),
    ("md_kick", _md_kick, "shape", RuntimeError),
    ("md_scr_barostat", _md_scr_barostat, "dtype", RuntimeError),
    ("md_scr_barostat", _md_scr_barostat, "shape", RuntimeError),
    ("md_affine_scale", _md_affine_scale, "dtype", RuntimeError),
    ("md_affine_scale", _md_affine_scale, "shape", RuntimeError),
    ("opt_fire_reduce", _opt_fire_reduce, "dtype", RuntimeError),
    ("opt_fire_reduce", _opt_fire_reduce, "shape", RuntimeError),
    ("opt_fire_step", _opt_fire_step, "dtype", RuntimeError),
    ("opt_fire_step", _opt_fire_step, "shape", RuntimeError),
    ("opt_fire_step", _opt_fire_step, "missing", RuntimeError),
    ("opt_fire_update", _opt_fire_update, "dtype", RuntimeError),
    ("opt_fire_update", _opt_fire_update, "missing", RuntimeError),
    ("gemm_tf32x3_ex", _gemm_tf32x3_ex, "dtype", RuntimeError),
    ("gemm_tf32x3_ex", _gemm_tf32x3_ex, "layout", RuntimeError),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,call,bad,exc", REJECT, ids=[f"{r[0]}-{r[2]}" for r in REJECT])
def test_wrapper_rejects_bad_argument_before_launch(name, call, bad, exc):
    n0 = ops.LAUNCHES["n"]
    with pytest.raises(exc, match=re.escape(f"hermnet_b200.{name}:")) as info:
        call(bad)
    assert type(info.value) is exc
    assert ops.LAUNCHES["n"] == n0
