"""Host-side contract of the batched C entry points, each test named after the entry point it covers.

- A refusal sets its own error text: topay_last_error() is thread-local and never cleared, so an entry point that
  returned TOPAY_ERR_NOT_READY without text would report whatever an earlier, unrelated failure left behind.
- In/out arrays the header promises to leave alone come back unchanged: pc of a visible segment
  (topay_field_line_visible) and grad of the nearest-cell kinds (topay_rogfield_query).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PRIMED = "int_K must be in [1, 32]"


def _d(a, t=C.c_double):
    return a.ctypes.data_as(C.POINTER(t))


def _prime(field_h):
    """Leaves a known text behind: topay_solver_create refuses int_K = 99 before it looks at the field."""
    from topay_b200 import _lib
    from topay_b200.field import robot_params_default
    from topay_b200.optimizer import opt_params_default
    l = _lib.lib()
    o = opt_params_default()
    o.int_K = 99
    rp = robot_params_default()
    h = C.c_void_p()
    assert l.topay_solver_create(C.byref(o), C.byref(rp), field_h, 4, 8, C.byref(h)) == _lib.ERR_TOO_LARGE
    assert l.topay_last_error().decode() == PRIMED


def _unbuilt_calls():
    """(entry point, call(l, h)) for every field entry point that refuses a field that was never rebuilt."""
    import torch
    from topay_b200.field import robot_params_default
    n = 4
    p2 = np.linspace(-1.0, 1.0, 2 * n).reshape(n, 2)
    p3 = np.linspace(-1.0, 1.0, 3 * n).reshape(n, 3) + [0.0, 0.0, 1.0]
    q3 = p3 + [0.5, 0.3, 0.0]
    p2r = p2[::-1].copy()
    idx = np.full((n, 2), 10, dtype=np.int32)
    states = np.zeros((n, 10))
    dist, grad, val = np.empty(n), np.empty((n, 3)), np.empty(n)
    flag = np.empty(n, dtype=np.int8)
    pc = np.zeros((n, 3))
    paths = np.array([[0.0, 0.0, 0.5], [1.0, 0.0, 0.5], [0.0, 0.2, 0.5], [1.0, 0.2, 0.5]])
    off = np.array([0, 2, 4], dtype=np.int32)
    pairs = np.array([0, 1], dtype=np.int32)
    rp = robot_params_default()
    tp = torch.from_numpy(p3).cuda()
    td = torch.empty(n, dtype=torch.float64, device="cuda")
    tg = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    i8 = C.c_int8
    return [
        ("topay_field_query3d", lambda l, h: l.topay_field_query3d(h, _d(p3), n, _d(dist), _d(grad))),
        ("topay_field_query2d", lambda l, h: l.topay_field_query2d(h, _d(p2), n, 0, _d(dist), _d(grad))),
        ("topay_field_distance3d", lambda l, h: l.topay_field_distance3d(h, _d(p3), n, _d(dist))),
        ("topay_field_distance2d", lambda l, h: l.topay_field_distance2d(h, _d(p2), n, _d(dist))),
        ("topay_field_is_collision2d", lambda l, h: l.topay_field_is_collision2d(h, _d(p2), n, 0.1, _d(flag, i8))),
        ("topay_field_is_collision3d", lambda l, h: l.topay_field_is_collision3d(h, _d(p3), n, 0.1, _d(flag, i8))),
        ("topay_field_is_line_collision_grid2d",
         lambda l, h: l.topay_field_is_line_collision_grid2d(h, _d(p2), _d(p2r), n, 0.0, _d(flag, i8))),
        ("topay_field_dist_coarse2d", lambda l, h: l.topay_field_dist_coarse2d(h, _d(p2), n, 0, _d(val))),
        ("topay_field_dist_coarse2i", lambda l, h: l.topay_field_dist_coarse2i(h, _d(idx, C.c_int32), n, 0, _d(val))),
        ("topay_field_whole_body_collision",
         lambda l, h: l.topay_field_whole_body_collision(h, C.byref(rp), _d(states), n, _d(flag, i8))),
        ("topay_field_line_visible",
         lambda l, h: l.topay_field_line_visible(h, _d(p3), _d(q3), n, 0.1, 0, _d(flag, i8), _d(pc))),
        ("topay_field_same_topo_paths",
         lambda l, h: l.topay_field_same_topo_paths(h, _d(paths), _d(off, C.c_int32), 2, _d(pairs, C.c_int32), 1,
                                                    0.1, 0, _d(flag, i8))),
        ("topay_field_query3d_dev",
         lambda l, h: l.topay_field_query3d_dev(h, C.c_void_p(tp.data_ptr()), n, C.c_void_p(td.data_ptr()),
                                                C.c_void_p(tg.data_ptr()))),
    ]


def test_unbuilt_field_refusals_set_their_own_text():
    """Every field entry point that refuses a never-rebuilt field returns ERR_NOT_READY and replaces the error text
    an earlier failure left behind."""
    from topay_b200 import _lib
    from topay_b200.field import GridMap
    l = _lib.lib()
    gm = GridMap()
    calls = _unbuilt_calls()
    assert len(calls) == 13
    stale = []
    for name, call in calls:
        _prime(gm.h)
        rc = call(l, gm.h)
        assert rc == _lib.ERR_NOT_READY, (name, rc)
        if l.topay_last_error().decode() == PRIMED:
            stale.append(name)
    assert not stale, f"refused with the stale text {PRIMED!r}: {stale}"
    gm.close()


def test_topay_field_line_visible_keeps_pc_of_visible_segments():
    """topay_field_line_visible: pc rows of visible segments come back exactly as passed in; blocked segments get
    their collision point."""
    from topay_b200.field import GridMap
    gm = GridMap()
    wall = np.array([[x, y, z] for x in (0.0, 0.05) for y in np.arange(-2.0, 2.0, 0.05) for z in (0.05, 0.5)])
    gm.rasterize(wall)
    gm.updateESDF()
    n = 64
    y = np.linspace(-6.0, 6.0, n)
    p1 = np.stack([np.full(n, -1.5), y, np.full(n, 0.5)], axis=1)
    p2 = np.stack([np.full(n, 1.5), y, np.full(n, 0.5)], axis=1)
    sentinel = 1000.0 + np.arange(3 * n, dtype=np.float64).reshape(n, 3) * 0.25
    vis, pc = gm.lineVisib(p1, p2, 0.1, pc=sentinel)
    assert vis.any() and not vis.all()
    assert np.array_equal(pc[vis], sentinel[vis])
    assert not np.any(pc[~vis] == sentinel[~vis])
    gm.close()


@pytest.mark.parametrize("kind", [3, 4, 5], ids=["Q_CELL", "Q_CELL_FLAT", "Q_CELL_CRITICAL"])
def test_topay_rogfield_query_cell_kinds_leave_grad(kind):
    """topay_rogfield_query: the nearest-cell kinds write dist only; a sentinel grad comes back unchanged and dist
    equals the query made without grad."""
    import topay_b200 as tp
    from topay_b200 import _lib
    from topay_b200.rog import ESDFMap
    m = ESDFMap(tp.rog_desc(half_prob_map_size_i=(30, 22, 9), prob_resolution=0.1, esdf_resolution=0.1,
                            local_update_box=(5.0, 3.0, 1.5), map_sliding_en=True))
    rng = np.random.default_rng(3)
    m.updateGridCounter(rng.uniform(-1, 1, (300, 3)) * [2.5, 1.8, 0.6], 1, 3)
    m.updateESDF3D((0.0, 0.0, 0.0))
    pos = np.ascontiguousarray(rng.uniform(-1, 1, (200, 3)) * [2.0, 1.5, 0.5])
    sentinel = -7.0 - np.arange(3 * len(pos), dtype=np.float64).reshape(-1, 3)
    grad = sentinel.copy()
    dist = np.empty(len(pos))
    l = _lib.lib()
    _lib.check(l.topay_rogfield_query(m.h, kind, _d(pos), len(pos), _d(dist), _d(grad)), "topay_rogfield_query")
    assert np.array_equal(grad, sentinel)
    assert np.array_equal(dist, m._query(kind, pos, want_grad=False))
    m.close()
