"""The size limits of the kernel routes, read from the library's own predicates (no GPU needed).

Every route has a size limit past which a call takes another route: the one-CTA tile kernel and the persistent
planner kernel (vhp_sweep_tile_supported / vhp_planner_supported: the fp64 tile state of an 8-warp CTA in 227 KB of
shared memory, for the planner with its 544 bytes of static shared memory on top), the direct window / range-merge /
cover route (vhp_sweep_window_supported) and the direct view merge (vhp_sweep_merge_view_supported, 16 bytes more).
tests/test_gpu_limits.py runs each route at its edge and one past it on a B200, at the shapes pinned here.  The edges
are found by bisection over the predicates, so that the GPU tests follow the layout; this file pins where they fall
today so that a change of the tile layout is noticed."""
import ctypes as C

import pytest

MAX_SIDE = 16384  # check_grid_dtype: the largest side of any grid

RECHECK = ("the tile layout moved a route's size limit: re-check tests/test_gpu_limits.py on a GPU (it runs every "
           "route at its edge and one past it), then update this table")

# (predicate, the other sizes) -> the largest accepted nx (tile / planner) or radius (window / view merge)
TILE_EDGES = {1: 9632, 32: 9632, 33: 9632, 40: 9632, 64: 9632, 65: 9600, 1000: 9472, 4096: 9088, 8192: 8544,
              16384: 7584}
PLANNER_EDGES = {1: 9600, 32: 9600, 33: 9568, 40: 9568, 64: 9568, 65: 9568, 1000: 9440, 4096: 9056, 8192: 8512,
                 16384: 7552}
WINDOW_EDGES = {(16384, 16384): 4223, (12000, 12000): 4223, (16384, 40): 4815}
VIEW_EDGES = {(16384, 16384): 4223, (12000, 12000): 4223, (16384, 40): 4799}


def predicates():
    """tile, grid, window, view, planner: the library's exported C++ predicates (through their mangled names)"""
    import visibility_heuristic_path_planner_b200 as vhp
    lib = vhp.load_library()

    def fn(name, nargs):
        f = getattr(lib, name)
        f.restype = C.c_bool
        f.argtypes = [C.c_int] * nargs
        return lambda *a: bool(f(*a))
    return dict(tile=fn("_Z24vhp_sweep_tile_supportedii", 2), grid=fn("_Z24vhp_sweep_grid_supportedii", 2),
                window=fn("_Z26vhp_sweep_window_supportediii", 3),
                view=fn("_Z30vhp_sweep_merge_view_supportediii", 3),
                planner=fn("_Z21vhp_planner_supportedii", 2))


def last_accepted(pred, lo, hi):
    """the largest v in [lo, hi] with pred(v), for a pred that holds on [lo, edge] and fails above; lo must pass"""
    assert pred(lo), f"the predicate refuses its lower bound {lo}"
    if pred(hi):
        return hi
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if pred(mid):
            lo = mid
        else:
            hi = mid
    return lo


def tile_edge(p, ny):
    """largest nx the one-CTA tile kernel takes at this ny"""
    return last_accepted(lambda nx: p["tile"](nx, ny), 1, MAX_SIDE)


def planner_edge(p, ny):
    return last_accepted(lambda nx: p["planner"](nx, ny), 1, MAX_SIDE)


def window_edge(p, nx, ny):
    """largest radius the direct window / range-merge / cover route takes on an nx x ny map"""
    return last_accepted(lambda r: p["window"](nx, ny, r), 0, MAX_SIDE)


def view_edge(p, nx, ny):
    return last_accepted(lambda r: p["view"](nx, ny, r), 0, MAX_SIDE)


@pytest.fixture(scope="module")
def preds():
    return predicates()


@pytest.mark.parametrize("ny", sorted(TILE_EDGES))
def test_tile_and_planner_width_edges(preds, ny):
    got = tile_edge(preds, ny)
    assert got == TILE_EDGES[ny], f"{RECHECK}: tile kernel edge at ny = {ny} is nx = {got}, was {TILE_EDGES[ny]}"
    assert preds["tile"](got, ny) and not preds["tile"](got + 1, ny)
    pl = planner_edge(preds, ny)
    assert pl == PLANNER_EDGES[ny], f"{RECHECK}: planner kernel edge at ny = {ny} is nx = {pl}, was {PLANNER_EDGES[ny]}"
    assert pl < got  # the planner kernel's static shared memory comes on top of the tile state


@pytest.mark.parametrize("shape", sorted(WINDOW_EDGES))
def test_window_and_view_merge_radius_edges(preds, shape):
    w, v = window_edge(preds, *shape), view_edge(preds, *shape)
    assert w == WINDOW_EDGES[shape], f"{RECHECK}: direct window edge on {shape} is R = {w}, was {WINDOW_EDGES[shape]}"
    assert v == VIEW_EDGES[shape], f"{RECHECK}: direct view-merge edge on {shape} is R = {v}, was {VIEW_EDGES[shape]}"
    assert v <= w  # the view merge needs the window layout plus its tail


def test_view_merge_falls_back_while_the_range_merge_is_direct(preds):
    """on 16384 x 40 the radii 4800..4815 take the direct route for windows and range merges, the fallback for views"""
    for r in range(4800, 4816):
        assert preds["window"](16384, 40, r) and not preds["view"](16384, 40, r), (RECHECK, r)


def test_grid_route_takes_every_shape_up_to_the_maximum(preds):
    """Grid mode is the fallback of every route, so it must take every shape up to 16384 in both directions.  Its
    shared memory grows with nx and with ny, so the rows and columns through 16384 x 16384 bound every shape; the
    small sides are run as well."""
    grid = preds["grid"]
    for n in range(1, MAX_SIDE + 1):
        assert grid(n, MAX_SIDE) and grid(MAX_SIDE, n) and grid(n, 1) and grid(1, n), n
    for s in (1, 40, 1000, MAX_SIDE):
        assert not grid(MAX_SIDE + 1, s) and not grid(s, MAX_SIDE + 1)
        assert not preds["tile"](MAX_SIDE + 1, s) and not preds["tile"](s, MAX_SIDE + 1)
        assert not preds["window"](MAX_SIDE + 1, s, 0) and not preds["window"](s, MAX_SIDE + 1, 0)


def test_bisection_finds_the_edge():
    assert last_accepted(lambda v: v <= 9632, 1, MAX_SIDE) == 9632
    assert last_accepted(lambda v: v <= 1, 1, MAX_SIDE) == 1
    assert last_accepted(lambda v: True, 0, MAX_SIDE) == MAX_SIDE
