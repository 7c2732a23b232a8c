"""The C-ABI shared library loads and exports every symbol ``include/hermnet_b200.h`` declares (no compute calls,
so no GPU is needed), and the ctypes table in ``hermnet_b200/_lib.py`` covers exactly the same set."""
import ctypes
import os
import re

from hermnet_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "hermnet_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hn_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    syms = declared_symbols()
    for must in ("hn_radius_graph_count", "hn_radius_graph_fill", "hn_triplets_count", "hn_triplets_fill",
                 "hn_edge_geom_fwd", "hn_edge_geom_bwd", "hn_painn_edge_fwd", "hn_painn_edge_bwd_dst",
                 "hn_painn_edge_bwd_src", "hn_painn_edge_bwd_w", "hn_gather_rows", "hn_segment_sum"):
        assert must in syms


def test_library_builds_and_exports_every_declared_symbol():
    path = build.build()
    lib = ctypes.CDLL(path)
    for name in declared_symbols():
        assert hasattr(lib, name), f"{name} declared in include/hermnet_b200.h but not exported by {path}"


def test_ctypes_table_matches_header():
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    lib = _lib.load()
    assert lib.hn_abi_version() == 2
    assert lib.hn_painn_edge_num_slices(128, 0) == 1 and lib.hn_painn_edge_num_slices(256, 0) == 2
    assert lib.hn_painn_edge_num_slices(96, 0) == 3 and lib.hn_painn_edge_num_slices(100, 1) == 0
    assert lib.hn_painn_edge_num_slices(128, 1) == lib.hn_painn_edge_num_slices(128, 1) >= 1 and lib.hn_segment_sum_workspace_bytes(2, 1) > 0
    assert lib.hn_radius_graph_workspace_bytes(1000, 1) > 0


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "hermnet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)
