"""The C-ABI library loads on a CPU-only machine and exports every symbol the public header declares; the
layout table it reports matches the Python-side statement of the reference's state_dict contract."""
import ctypes
import os
import re

import pytest

from dynaboa_b200 import _lib, build, layout

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    build.build()
    return _lib.load()


def header_symbols():
    src = open(os.path.join(REPO, 'include', 'dynaboa_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(dboa_[a-z0-9_]+)\s*\(', src)))


def test_header_symbols_exported(lib):
    syms = header_symbols()
    assert len(syms) >= 35
    for s in syms:
        assert hasattr(lib, s), f'{s} declared in include/dynaboa_b200.h but not exported'
    assert set(syms) == set(_lib.SIGNATURES), 'ctypes signature table out of sync with the header'


def test_version_and_counters(lib):
    assert b'sm_100a' in lib.dboa_version()
    assert lib.dboa_launch_count() >= 0


def test_layout_matches_reference_contract(lib):
    from dynaboa_b200.hmr import ArenaLayout
    lay = ArenaLayout()
    ref = layout.param_shapes()
    assert lay.n == 169 and lay.names == list(ref.keys())
    assert [tuple(s) for s in lay.shapes] == [tuple(v) for v in ref.values()]
    assert sum(int(__import__('numpy').prod(s)) for s in lay.shapes) == layout.num_params() == 26977501
    # views must not overlap and must stay inside the arena
    spans = sorted((o, o + 1 + sum((s - 1) * st for s, st in zip(sh, stv))) for o, sh, stv in zip(lay.offsets, lay.shapes, lay.strides))
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 <= b0
    assert spans[-1][1] <= lay.floats


def test_size_queries(lib):
    assert lib.dboa_hmr_tape_floats(1) > 20_000_000 and lib.dboa_hmr_tape_floats(0) < 0
    assert lib.dboa_hmr_scratch_floats(2) > 0
    assert lib.dboa_smpl_tape_floats(2) == 2 * (8 * 20670 + 648)      # 7 blend-shape row splits + posed vertices, chain state


def test_argument_errors_do_not_need_a_gpu(lib):
    assert lib.dboa_rot6d_fwd(None, None, 4, None) == -1
    assert lib.dboa_sgd_update(None, None, None, 0.1, 8, None) == -1
    off, nd = ctypes.c_longlong(), ctypes.c_int()
    shp, st = (ctypes.c_longlong * 4)(), (ctypes.c_longlong * 4)()
    assert lib.dboa_hmr_param_info(999, None, 0, ctypes.byref(off), ctypes.byref(nd), shp, st) == -1
    plan = (ctypes.c_longlong * 5)()
    for kernel in (-1, 3):
        assert lib.dboa_last_wide_plan(kernel, plan) == -1
        assert lib.dboa_set_split_limits(kernel, -1, -1, -1) == -1
    assert lib.dboa_last_wide_plan(0, None) == -1
    for kernel in (0, 1, 2):
        assert lib.dboa_last_wide_plan(kernel, plan) == 0
        assert lib.dboa_set_split_limits(kernel, -1, -1, -1) == 0      # restore the defaults: changes nothing here


def test_tensor_map_cache_keeps_held_pointers_across_evictions(lib):
    """Host logic of the TMA tensor-map cache (csrc/conv_wide.cu: MapCache): a launch looks up to six maps up before it
    dereferences them, and an eviction between two of those lookups must not free the earlier ones.  Round 2 shipped for a while
    with a cache that freed everything at 4096 entries -- one core dump in five GPU suite runs.  The self test inserts far past the
    bound while holding the last `window` pointers and checks the bytes a freed chunk would lose to the allocator."""
    assert lib.dboa_selftest_map_cache(64, 5000, 6) == 0
    assert lib.dboa_selftest_map_cache(6, 5000, 6) == 0           # eviction every seven insertions, six pointers held
    assert lib.dboa_selftest_map_cache(1, 1000, 1) == 0
    assert lib.dboa_selftest_map_cache(4, 100, 6) == -1           # more pointers held than one generation guarantees: rejected
    assert lib.dboa_selftest_map_cache(0, 10, 1) == -1
