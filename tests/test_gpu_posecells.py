"""GPU parity of the pose-cell path against the oracle and the reference-generated fixtures.

Every call goes through the C ABI (ctypes -> libpyratslam_b200.so).  Bars (SURVEY.md section 8d):
arg-max cell bit-exact at every step; activities  max|gpu - ref| / max|ref|  <= 1e-5 in float32 and
<= 1e-12 in float64.
"""
import math

import numpy as np
import pytest
import torch

from oracle import drivers as odrv
from oracle import posecells as opc

pytestmark = pytest.mark.gpu

RTOL = {np.float32: 1e-5, np.float64: 1e-12}
PATHS = ["auto", "generic", "resident", "tiled", "cluster", "pair"]


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _make(shape, dtype, path, **kw):
    from pyratslam_b200 import PoseCellNetwork
    net = PoseCellNetwork(shape, dtype=dtype, **kw)
    _force(net._ens, path)
    return net


def _force(ens, path):
    if path == "auto":
        return
    try:
        ens.force_path(path)
    except ValueError as e:
        pytest.skip(str(e))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name,shape,inject", [
    ("simulate_50x50x10.npz", (50, 50, 10), None),
    ("ros_21x21x36.npz", (21, 21, 36), None),
    ("ros_21x21x36_dies.npz", (21, 21, 36), None),
    ("odd_9x8x7.npz", (9, 8, 7), (4, 3, 2)),
    ("odd_17x23x11.npz", (17, 23, 11), (16, 0, 10)),
])
def test_golden_trajectories(golden, name, shape, inject, dtype, path):
    g = golden(name)
    net = _make(shape, dtype, path)
    net.inject(1, tuple(s // 2 for s in shape) if inject is None else inject)
    worst = 0.0
    for s, v in enumerate(g["odom"]):
        got = net.update(v)
        assert tuple(got) == tuple(g["argmax"][s]), (name, s, got, g["argmax"][s])
        key = "state_%03d" % s
        if key in g.files:
            ref = g[key]
            if ref.max() == 0:
                assert net.posecells.max() == 0
            else:
                worst = max(worst, _rel(net.posecells, ref))
    assert worst <= RTOL[dtype], worst


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_simulate_driver(golden, dtype):
    from pyratslam_b200 import simulate
    trace = simulate.main(steps=40, verbose=False, dtype=dtype)
    assert [tuple(t) for t in trace] == [tuple(t) for t in golden("simulate_50x50x10.npz")["argmax"].tolist()]


def test_keyerror_and_radius(golden):
    for v, expect in golden("keyerror.npz")["cases"]:
        net = _make((21, 21, 36), np.float32, "auto")
        net.inject(1, (10, 10, 18))
        if expect:
            before = net.posecells
            with pytest.raises(KeyError):
                net.update((v, 0.0))
            assert np.array_equal(net.posecells, before)   # raised before the device state was touched
        else:
            net.update((v, 0.0))
    net = _make((9, 8, 7), np.float32, "auto")
    net.inject(1, (4, 3, 2))
    with pytest.raises(ValueError):
        net.update((1.32, 0.0))    # 6.6 cells: 3 + 7 > 8


def test_device_error_flags_for_ensembles():
    from pyratslam_b200 import PoseCellEnsemble
    ens = PoseCellEnsemble((21, 21, 36), 3)
    ens.inject(1, (10, 10, 18))
    with pytest.raises(KeyError):
        ens.update(np.array([[0.03, 0.0], [0.1, 0.0], [0.02, 0.0]]))     # network 1 hits the LUT hole
    with pytest.raises(ValueError):
        ens.update(np.array([[0.03, 0.0], [0.02, 0.0], [4.0, 0.0]]))     # 20 cells > 21 - 3


def test_inject_argmax_ties_and_roundtrip():
    net = _make((9, 8, 7), np.float32, "auto")
    assert net.get_pc_max() == (0, 0, 0)                 # all-zero grid -> first cell
    rng = np.random.default_rng(0)
    st = rng.uniform(0, 1, (9, 8, 7))
    st[5, 2, 3] = 2.0
    st[2, 7, 6] = 2.0                                    # equal maxima: the lower flat index wins
    net.posecells = st
    assert np.allclose(net.posecells, st.astype(np.float32))
    assert net.get_pc_max() == (2, 7, 6)
    net.inject(0.5, (5, 2, 3))
    assert net.get_pc_max() == (5, 2, 3)
    net.inject(1.0, (-1, -1, -1))                        # numpy-style negative indices
    assert net.posecells[8, 7, 6] == pytest.approx(st[8, 7, 6] + 1.0, rel=1e-6)
    with pytest.raises(IndexError):
        net.inject(1.0, (9, 0, 0))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_path_integration_alone(dtype):
    shape = (17, 23, 11)
    ref = opc.PoseCellNetwork(shape)
    rng = np.random.default_rng(3)
    st = rng.uniform(0, 1, shape)
    ref.posecells = st.copy()
    net = _make(shape, dtype, "auto")
    net.posecells = st
    for v in [(0.37, 0.21), (-0.8, -0.4)]:
        ref.path_integration(*v)
        net.path_integration(*v)
    assert _rel(net.posecells, ref.posecells) <= (2e-6 if dtype == np.float32 else 1e-12)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("path", PATHS)
def test_ensemble_against_oracle(dtype, path):
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 12, 25
    rng = np.random.default_rng(3)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    ref_amax, ref_states = opc.run_ensemble(shape, gis, odom)
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis, dtype=dtype)
    _force(ens, path)
    ens.inject(1.0, tuple(s // 2 for s in shape))
    # half the steps one at a time through the host entry, the rest as one multi-step run
    got = [ens.update(odom[t]) for t in range(10)]
    got = np.concatenate([np.stack(got), ens.run(odom[10:])])
    assert np.array_equal(got, ref_amax)
    assert _rel(ens.posecells, ref_states) <= RTOL[dtype]


def test_overlapped_host_stepping_matches_blocking_calls():
    """update_submit / update_result (one step in flight) return exactly what consecutive update() calls return."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 300, 9
    rng = np.random.default_rng(5)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    a = PoseCellEnsemble(shape, B, global_inhibition=gis)
    b = PoseCellEnsemble(shape, B, global_inhibition=gis)
    for e in (a, b):
        e.inject(1.0, (10, 10, 18))
    want = np.stack([a.update(odom[t]) for t in range(T)])
    got = np.stack(list(b.update_stream(odom[t] for t in range(T))))
    assert np.array_equal(got, want) and torch.equal(a.state, b.state)
    with pytest.raises(RuntimeError):
        b.update_result()
    b.update_submit(odom[0])
    b.update_submit(odom[1])
    with pytest.raises(RuntimeError):
        b.update_submit(odom[2])
    b.update_result(), b.update_result()


def test_large_grid_one_step_against_oracle():
    """BASELINE config 3 at full size (256x256x72): two steps against the scipy oracle (a few seconds)."""
    shape = (256, 256, 72)
    ref = opc.PoseCellNetwork(shape)
    net = _make(shape, np.float32, "auto")
    for n in (ref, net):
        n.inject(1.0, (128, 128, 36))
        n.inject(0.5, (3, 250, 70))      # a second packet across the periodic boundary
    for v in [(0.21, 0.03), (0.12, -0.04)]:
        want = tuple(ref.update(v))
        assert tuple(net.update(v)) == want
    assert _rel(net.posecells, ref.posecells) <= 1e-5


@pytest.mark.parametrize("shape", [(33, 35, 9), (70, 40, 19), (128, 64, 8), (36, 36, 3), (72, 100, 9), (65, 66, 20),
                                   (96, 64, 23)])
@pytest.mark.parametrize("path", ["tiled", "cluster"])
def test_tiled_path_shapes_against_oracle(shape, path):
    """The large-grid kernels (and the cluster kernel, where it applies) on shapes that exercise their edges: X*Y
    not a multiple of 4 (scalar accesses), ragged tiles and segments in x and y, theta counts that are not a
    multiple of the chunk, tiles that wrap on every side.  Two packets (one across the periodic corner) and an
    exact tie for the maximum."""
    ref = opc.PoseCellNetwork(shape)
    net = _make(shape, np.float32, path)
    assert net.path == path
    X, Y, Th = shape
    for n in (ref, net):
        n.inject(1.0, (X // 2, Y // 2, Th // 2))
        n.inject(0.75, (X - 1, 0, Th - 1))
    # the last two steps move by 7 / 11 cells: integer origins far beyond the 3-cell halo of a tile
    for v in [(0.21, 0.03), (0.12, -0.04), (0.0, 0.0), (0.33, 0.0), (1.41, 0.02), (2.21, -0.03)]:
        if 3 + np.ceil(abs(v[0]) / 0.2) > min(X, Y):
            continue
        assert tuple(net.update(v)) == tuple(ref.update(v)), v
        assert _rel(net.posecells, ref.posecells) <= 1e-5
    # equal maxima: the lowest flat index must win; then an all-zero grid reports cell (0, 0, 0)
    st = np.zeros(shape)
    st[X - 2, 3, 1] = st[1, Y - 1, 1] = 1.0       # translated copies: bit-identical responses
    ref.posecells = st.copy()
    net.posecells = st
    got, want = net.update((0.0, 0.0)), ref.update((0.0, 0.0))
    assert tuple(got) == tuple(want)
    pc = net.posecells
    assert np.array_equal(pc[X - 2, 3], pc[1, Y - 1]) and pc[tuple(got)] == pc.max()   # an exact tie, lowest index won
    if Th >= 7:
        assert tuple(got)[:2] == (1, Y - 1)
    gi0 = ref.global_inhibition
    ref.global_inhibition = net.global_inhibition = 50.0
    assert tuple(net.update((0.0, 0.0))) == tuple(ref.update((0.0, 0.0))) == (0, 0, 0)
    assert net.posecells.max() == 0
    ref.global_inhibition = net.global_inhibition = gi0


@pytest.mark.parametrize("shape,B", [((21, 21, 36), 1), ((21, 21, 36), 5), ((50, 50, 10), 3), ((9, 8, 7), 2),
                                     ((17, 23, 12), 1), ((30, 24, 16), 2), ((12, 40, 27), 1)])
def test_cluster_path_against_oracle(shape, B):
    """One network per thread-block cluster: cluster sizes 2..8, 1..9 planes per CTA, ragged segments, small
    ensembles with per-network inhibition and odometry (including a network that dies and a theta shift)."""
    from pyratslam_b200 import PoseCellEnsemble
    T = 8
    rng = np.random.default_rng(sum(shape) + B)
    gis = np.linspace(0.08, 0.22, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.3, 0.3, (T, B))], axis=-1)
    odom[3] = 0.0
    ref_amax, ref_states = opc.run_ensemble(shape, gis, odom)
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis)
    _force(ens, "cluster")
    assert ens.path == "cluster"
    ens.inject(1.0, tuple(s // 2 for s in shape))
    got = [ens.update(odom[t]) for t in range(4)]
    got = np.concatenate([np.stack(got), ens.run(odom[4:])])
    assert np.array_equal(got, ref_amax)
    assert _rel(ens.posecells, ref_states) <= 1e-5


def test_translation_equivariance_large():
    """Size-independent property: the update commutes with a cyclic shift of the grid in x and y
    (not in theta: the heading decides which way a plane moves)."""
    shape = (64, 48, 36)
    rng = np.random.default_rng(9)
    st = np.zeros(shape)
    st[10:14, 20:23, 5:9] = rng.uniform(0.5, 1.0, (4, 3, 4))
    a = _make(shape, np.float32, "auto")
    b = _make(shape, np.float32, "auto")
    a.posecells = st
    b.posecells = np.roll(st, (17, -9), axis=(0, 1))
    for v in [(0.21, 0.05), (0.12, -0.05), (0.33, 0.0)]:
        ma, mb = a.update(v), b.update(v)
        assert ((ma[0] + 17) % 64, (ma[1] - 9) % 48, ma[2]) == tuple(mb)
    assert _rel(np.roll(a.posecells, (17, -9), axis=(0, 1)), b.posecells) <= 2e-6


def test_full_size_ensemble_replicas_and_samples():
    """BASELINE config 4 at full size: 4096 networks; a sample is checked against the oracle and
    identical networks must produce identical bits."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 4096, 6
    rng = np.random.default_rng(3)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    gis[1000], odom[:, 1000] = gis[7], odom[:, 7]        # network 1000 is a replica of network 7
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis)
    ens.inject(1.0, (10, 10, 18))
    got = ens.run(odom)
    pick = [0, 7, 1000, 2047, 4095]
    ref_amax, ref_states = opc.run_ensemble(shape, gis[pick], odom[:, pick])
    assert np.array_equal(got[:, pick], ref_amax)
    st = ens.state
    assert torch.equal(st[7], st[1000])
    pc = ens.posecells
    assert _rel(pc[pick], ref_states) <= 1e-5


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_active_cells_sparse_readback(dtype):
    """The device-side compaction returns exactly nonzero(pc > thr) in C order (simulate.py:60-62)."""
    net = _make((50, 50, 10), dtype, "auto")
    net.inject(1, (25, 25, 5))
    for v in [(3.0, 0.0), (3.0, 0.0), (3.0, math.pi / 4)]:
        net.update(v)
    pc = net.posecells
    for thr in (0.002, 0.0, 0.05, 10.0):
        idx, val = net.active_cells(thr)
        ref = np.stack(np.nonzero(pc > thr), axis=-1)
        assert np.array_equal(idx, ref)
        assert np.array_equal(val, pc[pc > thr])
    idx, val = net.active_cells(0.0, max_cells=5)      # truncated output keeps the first cells
    assert np.array_equal(idx, np.stack(np.nonzero(pc > 0), axis=-1)[:5])


def test_single_call_update_checks_match_numpy():
    """prs_pc_update_host's host-side checks (C doubles) against the numpy expressions of the reference
    (posecell_network.py:249,252-267): same accept / KeyError decision for odometry on and around the LUT hole."""
    from pyratslam_b200 import PoseCellNetwork
    shape = (21, 21, 36)
    net = PoseCellNetwork(shape)
    net.inject(1, (10, 10, 18))
    e = net._ens
    rng = np.random.default_rng(12)
    cand = np.concatenate([np.array([0.1, 0.5, 0.9, 0.3, 0.7, 0.1 + 1e-17, 0.1 - 1e-16, 0.5000000000000001]),
                           np.round(rng.uniform(0, 1.5, 40), 1), rng.uniform(0, 1.5, 40)])
    n_key = 0
    for v in cand:
        vt = v / e.pc_vtrans_scale
        ex = vt * e._cos
        want_key = bool(((((ex - np.around(ex)) * 10).astype(np.int64)) >= 5).any())
        n_key += want_key
        if want_key:
            before = net.posecells
            with pytest.raises(KeyError):
                net.update((float(v), 0.0))
            assert np.array_equal(net.posecells, before)
        else:
            net.update((float(v), 0.0))
    assert n_key >= 3
    assert net.get_pc_max() == net.max_pc


def test_segmented_pair_kernel_50x50x10_ensemble():
    """simulate.py's grid (50, 50, 10) as an ensemble on the fused, segmented pair kernel (k_pc_pair_seg): per-network
    inhibition and odometry, a network that dies, theta shifts in both directions, single steps and a multi-step run."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (50, 50, 10), 7, 14
    rng = np.random.default_rng(50)
    gis = np.linspace(0.05, 0.27, B)              # the last one is above max(kernel_3d): that network dies
    odom = np.stack([rng.uniform(0, 0.6, (T, B)), rng.uniform(-0.7, 0.7, (T, B))], axis=-1)
    odom[5] = 0.0
    ref_amax, ref_states = opc.run_ensemble(shape, gis, odom)
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis)
    _force(ens, "pair")
    assert ens.path == "pair"
    ens.inject(1.0, (25, 25, 5))
    ens.inject(0.6, (49, 0, 9))                   # a second packet across the periodic corner
    ref2 = []
    for b in range(B):                            # the oracle ensemble starts from one packet: redo it with two
        n = opc.PoseCellNetwork(shape, global_inhibition=float(gis[b]))
        n.inject(1.0, (25, 25, 5))
        n.inject(0.6, (49, 0, 9))
        ref2.append(n)
    got = [ens.update(odom[t]) for t in range(6)]
    got = np.concatenate([np.stack(got), ens.run(odom[6:])])
    want = np.stack([[n.update(odom[t, b]) for b, n in enumerate(ref2)] for t in range(T)])
    assert np.array_equal(got, want)
    states = np.stack([n.posecells for n in ref2])
    assert _rel(ens.posecells, states) <= 1e-5
    assert states[-1].max() == 0 and ens.posecells[-1].max() == 0


# ------------------------------------------------------------------ active-set (sparsity-aware) path, posecell_active.cu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("name,shape,inject", [
    ("simulate_50x50x10.npz", (50, 50, 10), None),
    ("ros_21x21x36.npz", (21, 21, 36), None),
    ("ros_21x21x36_dies.npz", (21, 21, 36), None),
    ("odd_9x8x7.npz", (9, 8, 7), (4, 3, 2)),
    ("odd_17x23x11.npz", (17, 23, 11), (16, 0, 10)),
])
def test_active_set_golden_trajectories(golden, name, shape, inject, dtype, mode):
    """The reference's own trajectories through the active-set kernels (scan every update / list carried over)."""
    g = golden(name)
    net = _make(shape, dtype, "auto", active_set=mode)
    net.inject(1, tuple(s // 2 for s in shape) if inject is None else inject)
    worst = 0.0
    for s, v in enumerate(g["odom"]):
        got = net.update(v)
        assert tuple(got) == tuple(g["argmax"][s]), (name, s, got, g["argmax"][s])
        key = "state_%03d" % s
        if key in g.files:
            ref = g[key]
            if ref.max() == 0:
                assert net.posecells.max() == 0
            else:
                worst = max(worst, _rel(net.posecells, ref))
    assert worst <= RTOL[dtype], worst


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("mode", [1, 2])
def test_active_set_ensemble_against_oracle(dtype, mode):
    """An ensemble whose networks are in every regime at once: compact packets (active-set kernel), a dense random state
    and a negative global inhibition (flagged, updated by the dense kernels in the same call), a dead network, two packets
    across the periodic border, an injection between updates (invalidates the carried list)."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 9, 14
    rng = np.random.default_rng(11)
    gis = np.linspace(0.05, 0.25, B)
    gis[5] = -0.01                                   # zero cells do not stay zero: dense from the first update on
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    init = np.zeros((B,) + shape)
    init[:, 10, 10, 18] = 1.0
    init[2] = rng.uniform(0, 1, shape)               # dense state: falls back for one update, compact afterwards
    init[3] = 0.0                                    # dead from the start
    init[4, 0, 20, 35] = 0.7                         # second packet, wraps in all three axes
    refs = [opc.PoseCellNetwork(shape, global_inhibition=float(g)) for g in gis]
    for r, s in zip(refs, init):
        r.posecells = s.copy()
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis, dtype=dtype, active_set=mode)
    ens.posecells = init
    for t in range(T):
        if t == 6:                                   # view-template style injection in the middle of a run
            for r in refs:
                r.inject(0.3, (3, 17, 5))
            ens.inject(0.3, (3, 17, 5))
        want = np.array([r.update(tuple(odom[t, b])) for b, r in enumerate(refs)])
        got = ens.update(odom[t])
        assert np.array_equal(got, want), t
        assert _rel(ens.posecells, np.stack([r.posecells for r in refs])) <= RTOL[dtype], t
    got = ens.run(odom[:5])                          # multi-step entry
    want = np.array([[r.update(tuple(odom[t, b])) for b, r in enumerate(refs)] for t in range(5)])
    assert np.array_equal(got, want)
    assert _rel(ens.posecells, np.stack([r.posecells for r in refs])) <= RTOL[dtype]


def test_active_set_matches_dense_kernels_on_a_large_ensemble():
    """600 networks of the ROS grid, 30 updates: same arg-max trace as the fused dense kernel; with mode 2 a torch write to
    the state followed by invalidate_active() is picked up.  The states of two float32 implementations are compared at 1e-4
    of the peak: a few parameter regimes amplify any rounding difference by ~1.3x per update (bench_tools/error_growth.py:
    the float64 build drifts from 1e-16 to 1e-13 against the oracle over these 30 updates, the fused dense kernel reaches
    2.7e-5 and the active-set kernels 4e-6 on network 373), everywhere else they agree to 1e-6."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 600, 30
    rng = np.random.default_rng(12)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    dense = PoseCellEnsemble(shape, B, global_inhibition=gis)
    act = {m: PoseCellEnsemble(shape, B, global_inhibition=gis, active_set=m) for m in (1, 2)}
    for e in [dense] + list(act.values()):
        e.inject(1.0, (10, 10, 18))
    want = dense.run(odom)
    for m, e in act.items():
        assert np.array_equal(e.run(odom), want), m
        assert _rel(e.posecells, dense.posecells) <= 1e-4, m
    for e in [dense] + list(act.values()):
        e.state[:, 7, 3, 4] += 0.25                  # behind the library's back
    act[2].invalidate_active()
    want = dense.run(odom[:4])
    for m, e in act.items():
        assert np.array_equal(e.run(odom[:4]), want), m
        assert _rel(e.posecells, dense.posecells) <= 1e-4, m


def test_active_set_large_grid_against_oracle():
    """BASELINE config 3 (256x256x72) through the active-set kernels: two packets, one across the periodic border."""
    shape = (256, 256, 72)
    ref = opc.PoseCellNetwork(shape)
    nets = [_make(shape, np.float32, "auto", active_set=m) for m in (1, 2)]
    for n in [ref] + nets:
        n.inject(1.0, (128, 128, 36))
        n.inject(0.5, (3, 250, 70))
    for v in [(0.21, 0.03), (0.12, -0.04), (2.93, 0.3)]:
        want = tuple(ref.update(v))
        for n in nets:
            assert tuple(n.update(v)) == want
    for n in nets:
        assert _rel(n.posecells, ref.posecells) <= 1e-5


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape,B", [((5, 6, 4), 3), ((3, 3, 3), 2), ((7, 9, 5), 4), ((21, 21, 36), 7), ((50, 50, 10), 3),
                                     ((64, 33, 17), 2), ((70, 40, 19), 2), ((130, 65, 9), 1), ((256, 12, 72), 1)])
def test_active_set_random_states_match_the_generic_kernels(shape, B, dtype):
    """Random sparse states -- several packets, packets across the periodic border, single cells, negative cells, shifts of
    many cells -- on shapes that exercise every corner of the set arithmetic (axes shorter than the 7-tap reach, axes longer
    than 64 cells, odd strides): the active-set kernels run the taps in the generic kernels' order, so the two agree to
    rounding of the one sum whose order differs (the total)."""
    from pyratslam_b200 import PoseCellEnsemble
    X, Y, Th = shape
    rng = np.random.default_rng(X * 1000 + Y * 10 + Th)
    T = 6
    init = np.zeros((B,) + shape)
    for b in range(B):
        for _ in range(int(rng.integers(1, 4))):          # packets
            c = [int(rng.integers(0, n)) for n in shape]
            for _ in range(int(rng.integers(1, 12))):
                d = [int(rng.integers(-1, 2)) for _ in range(3)]
                init[b, (c[0] + d[0]) % X, (c[1] + d[1]) % Y, (c[2] + d[2]) % Th] += rng.uniform(0.05, 1.0)
        if b % 3 == 2:
            init[b, int(rng.integers(0, X)), int(rng.integers(0, Y)), int(rng.integers(0, Th))] = -0.3
    vmax = 0.2 * (min(X, Y) - 3) * 0.999                  # 3 + ceil(|vtrans| / 0.2) <= min(X, Y)
    odom = np.stack([rng.uniform(-vmax, vmax, (T, B)), rng.uniform(-0.5, 0.5, (T, B))], axis=-1)
    gis = rng.uniform(0.0, 0.05, B)                        # low inhibition: the packets survive and grow
    want = PoseCellEnsemble(shape, B, global_inhibition=gis, dtype=dtype)
    want.force_path("generic")
    got = {m: PoseCellEnsemble(shape, B, global_inhibition=gis, dtype=dtype, active_set=m) for m in (1, 2)}
    for e in [want] + list(got.values()):
        e.posecells = init
    tol = 2e-6 if dtype == np.float32 else 1e-13
    for t in range(T):
        try:
            ref = want.update(odom[t])
        except KeyError:                                   # the LUT hole of the reference: the same for every path
            for e in got.values():
                with pytest.raises(KeyError):
                    e.update(odom[t])
            continue
        ws = want.posecells
        for m, e in got.items():
            assert np.array_equal(e.update(odom[t]), ref), (m, t)
            assert _rel(e.posecells, ws) <= tol, (m, t, _rel(e.posecells, ws))


@pytest.mark.parametrize("shape,B", [((21, 21, 36), 5), ((50, 50, 10), 3)])
def test_active_set_fallback_behind_a_conditional_graph_node(shape, B):
    """prs_pc_step replays the active-set update as a graph whose dense fall-back is the body of a conditional node that the
    kernel raises when it flags a network.  Network 1 has a negative inhibition (dense on every update: the body runs),
    in a second ensemble nothing is ever flagged (the body never runs); both against the dense kernels, update by update."""
    from pyratslam_b200 import PoseCellEnsemble
    rng = np.random.default_rng(21)
    T = 7
    odom = torch.from_numpy(np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)).cuda()
    for neg in (True, False):
        gis = np.linspace(0.05, 0.2, B)
        if neg:
            gis[1] = -0.02
        want = PoseCellEnsemble(shape, B, global_inhibition=gis)
        got = PoseCellEnsemble(shape, B, global_inhibition=gis, active_set=2)
        for e in (want, got):
            e.inject(1.0, tuple(s // 2 for s in shape))
        for t in range(T):                               # the third call on captures the graph
            want.update_async(odom[t])
            got.update_async(odom[t])
            torch.cuda.synchronize()
            assert torch.equal(got._argmax, want._argmax), (neg, t)
            assert _rel(got.posecells, want.posecells) <= 1e-5, (neg, t)
            assert int(got._err.abs().sum().item()) == 0


def test_active_set_lists_follow_the_state_tensor():
    """One plan, two state tensors through the C ABI (prs_pc_step): the carried list of non-zero cells (mode 2) describes
    the tensor of the previous call; a call with another tensor must start from a scan of that tensor."""
    from pyratslam_b200 import PoseCellEnsemble, _native as nat
    shape, B = (21, 21, 36), 3
    gis = np.array([0.05, 0.1, 0.2])
    act = PoseCellEnsemble(shape, B, global_inhibition=gis, active_set=2)
    ref = [PoseCellEnsemble(shape, B, global_inhibition=gis) for _ in range(2)]
    states = [act.state, torch.zeros_like(act.state)]
    for st, r, loc in ((states[0], ref[0], (10, 10, 18)), (states[1], ref[1], (3, 17, 30))):
        r.inject(1.0, loc)
        st.copy_(r.state)
    act.invalidate_active()
    rng = np.random.default_rng(8)
    L = nat.lib()
    for t in range(8):
        od = torch.from_numpy(np.stack([rng.uniform(0, 0.3, B), rng.uniform(-0.1, 0.1, B)], axis=-1)).cuda()
        w = t % 2 if t < 6 else 1                     # alternate the tensors, then stay on one
        nat.check(L.prs_pc_step(act._h, states[w].data_ptr(), od.data_ptr(), act._gi.data_ptr(), act._argmax.data_ptr(),
                                act._total.data_ptr(), act._err.data_ptr(), nat.stream_ptr()), "prs_pc_step")
        ref[w].update_async(od)
        torch.cuda.synchronize()
        assert torch.equal(act._argmax, ref[w]._argmax), t
        assert float((states[w] - ref[w].state).abs().max() / ref[w].state.abs().max()) <= 1e-5, t


@pytest.mark.parametrize("B", [160, 300, 512])
def test_overlapping_launches_equal_serialised_launches(B):
    """Consecutive updates of an ensemble overlap on the device (programmatic dependent launch + one sequence number per
    network, posecell_resident.cu): 120 back-to-back updates of one ensemble -- and of two ensembles interleaved on one
    stream -- give bit for bit the states and arg-max cells of the same updates with a device synchronisation between
    them; so does the zero-copy host API (update_stream) against blocking update() calls."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, T = (21, 21, 36), 120
    rng = np.random.default_rng(B)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    od = torch.from_numpy(odom).cuda()
    ens = [PoseCellEnsemble(shape, B, global_inhibition=gis) for _ in range(5)]
    for e in ens:
        assert e.path == "resident"
        e.inject(1.0, (10, 10, 18))
    a, b1, b2, c, d = ens
    amax_a, amax_b = [], []
    for t in range(T):                                   # serialised
        a.update_async(od[t])
        torch.cuda.synchronize()
        amax_a.append(a._argmax.clone())
    for t in range(T):                                   # overlapping, two ensembles interleaved
        b1.update_async(od[t])
        b2.update_async(od[t])
        if t % 7 == 0:
            amax_b.append((t, b1._argmax.clone()))       # a stream-ordered read between two launches
    torch.cuda.synchronize()
    assert torch.equal(b1.state, a.state) and torch.equal(b2.state, a.state)
    assert torch.equal(b1._argmax, a._argmax) and torch.equal(b2._argmax, a._argmax)
    for t, am in amax_b:
        assert torch.equal(am, amax_a[t]), t
    want = np.stack([c.update(odom[t]) for t in range(T)])               # blocking host calls
    got = np.stack(list(d.update_stream(odom[t] for t in range(T))))     # one step in flight
    assert np.array_equal(got, want) and torch.equal(c.state, d.state) and torch.equal(c.state, a.state)
    assert np.array_equal(want[-1], a._unravel(a._argmax.cpu().numpy()))
