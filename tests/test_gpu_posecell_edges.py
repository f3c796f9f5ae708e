"""Every pose-cell kernel family against the float64 oracle at the edges of its inputs.

One update per case, each case one network of an ensemble (hundreds of cases per launch, several networks per CTA on
the resident kernel): edge odometry from test_posecell_edge_cases.py (integer origins on a half, the F0 / F-1 switch,
theta origins on their boundary and far out, translations up to the radius bound and one past it, non-finite values)
on four kinds of start state -- a packet from a few realistic updates, two packets one of them across the periodic
corner, a dense random state, a packet x5 that is not normalised.  Checked per network: the state
(max|gpu - ref| / max|ref| <= 1e-5 in float32, 1e-12 in float64, SURVEY.md section 8d), the arg-max cell, ``total``
(the sum before normalisation) and the PRS_ERR_* bits.  Then zero and negative global inhibition, the OR of the error
bits over a multi-step run, short runs of edge odometry, and the ensemble replay with zero and negative inhibition.

The start states are float32 values and the inhibitions float32 numbers, so the oracle (computed once per module)
serves both dtypes exactly.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import posecells as opc
from test_posecell_edge_cases import NEG_GIS, edge_cases, one_step_suite, plan, start_states

pytestmark = pytest.mark.gpu

RTOL = {np.float32: 1e-5, np.float64: 1e-12}
FAMILIES = {
    (21, 21, 36): ["generic", "resident", "pair", "cluster", "active1", "active2"],
    (50, 50, 10): ["generic", "pair", "cluster", "tiled"],
    (17, 23, 11): ["generic", "cluster", "tiled"],
    (12, 10, 5): ["generic", "active1", "active2"],
}
COMBOS = [(s, f, d) for s, fams in FAMILIES.items() for f in fams for d in (np.float32, np.float64)]
COMBO_IDS = ["%dx%dx%d-%s-%s" % (s + (f, np.dtype(d).name)) for s, f, d in COMBOS]
def _ensemble(shape, family, dtype, B, gis):
    from pyratslam_b200 import PoseCellEnsemble
    active = {"active1": 1, "active2": 2}.get(family, 0)
    ens = PoseCellEnsemble(shape, B, global_inhibition=gis, dtype=dtype, active_set=active)
    if not active:
        try:
            ens.force_path(family)
        except ValueError as e:
            pytest.skip(str(e))
        assert ens.path == family
    return ens


def _check_network(got_state, got_total, got_amax, ref, tol):
    """None if the device's result for one network matches the oracle's, else what differs."""
    want, want_total, want_amax = ref
    top = np.abs(want).max()
    if top == 0:
        if np.abs(got_state).max() != 0:
            return "state should be zero"
    else:
        rel = np.abs(got_state - want).max() / top
        if not rel <= tol:
            return "state rel %.3g" % rel
    if not abs(got_total - want_total) <= tol * abs(want_total):
        return "total %r vs %r" % (got_total, want_total)
    if tuple(got_amax) != tuple(want_amax):
        flat = np.sort(want.ravel())
        if not (flat[-1] - flat[-2] <= 4 * tol * top and want[tuple(got_amax)] >= flat[-1] - tol * top):
            return "arg-max %s vs %s" % (tuple(got_amax), tuple(want_amax))
    return None


def _run_and_check(shape, family, dtype, kind):
    states, gis, odom, errs, refs, _ = one_step_suite(shape, kind)
    B = len(states)
    ens = _ensemble(shape, family, dtype, B, gis)
    ens.posecells = states
    ens.update_async(torch.from_numpy(odom).to(ens.device))
    torch.cuda.synchronize()
    err = ens._err.cpu().numpy()
    total = ens._total.cpu().numpy().astype(np.float64)
    amax = ens._unravel(ens._argmax.cpu().numpy())
    pc = ens.posecells
    bad = []
    for b in range(B):
        if err[b] != errs[b]:
            bad.append((b, tuple(odom[b]), gis[b], "err %d, expected %d" % (err[b], errs[b])))
        elif refs[b] is not None:
            why = _check_network(pc[b], total[b], amax[b], refs[b], RTOL[dtype])
            if why:
                bad.append((b, tuple(odom[b]), gis[b], why))
    assert not bad, "%d of %d networks differ from the oracle: %s" % (len(bad), B, bad[:6])
    return B


@pytest.mark.parametrize("shape,family,dtype", COMBOS, ids=COMBO_IDS)
def test_one_step_edges_against_oracle(shape, family, dtype):
    """Every edge row on two start states each, one launch; the networks the plan refuses carry exactly their bits."""
    B = _run_and_check(shape, family, dtype, "edges")
    assert B >= 150


@pytest.mark.parametrize("shape,family,dtype", COMBOS, ids=COMBO_IDS)
def test_zero_and_negative_inhibition_against_oracle(shape, family, dtype):
    """gi = -0.005, -0.0005, -0.0, 0.0 on packet starts.  The reference's two masked writes (posecell_network.py:339-340)
    leave a cell below a negative gi at -gi, not at 0: every cell outside the packet."""
    _run_and_check(shape, family, dtype, "inhibition")


@pytest.mark.parametrize("shape,family,dtype", COMBOS, ids=COMBO_IDS)
def test_run_ors_error_bits_over_steps(shape, family, dtype):
    """prs_pc_run: err[b] is the OR of network b's bits over the T updates, each bit raised at a different step."""
    from pyratslam_b200 import _native as nat
    rows = edge_cases(shape)
    by_err = {}
    for r in rows:
        by_err.setdefault(plan(shape, r[1], r[2])[4], []).append((r[1], r[2]))
    ok = [v for v in by_err[0] if abs(plan(shape, *v)[3]) <= 4]
    bad = [v for e, vs in sorted(by_err.items()) if e for v in vs]
    T, B = 4, 3 * len(bad)
    odom = np.empty((T, B, 2))
    want = np.zeros(B, dtype=np.int32)
    for b in range(B):
        for t in range(T):
            odom[t, b] = ok[(b + 5 * t) % len(ok)]
        if b < 2 * len(bad):                            # one error at step b % T; then, for b >= len(bad), a second one
            for k, t in enumerate((b % T, (b + 2) % T)[: 1 + b // len(bad)]):
                v = bad[(b + k * 7) % len(bad)]
                odom[t, b] = v
                want[b] |= plan(shape, *v)[4]
    ens = _ensemble(shape, family, dtype, B, np.full(B, 0.1))
    ens.inject(1.0, tuple(s // 2 for s in shape))
    od = torch.from_numpy(odom).to(ens.device)
    am = torch.empty((T, B), dtype=torch.int64, device=ens.device)
    tot = torch.empty((T, B), dtype=ens.torch_dtype, device=ens.device)
    nat.check(nat.lib().prs_pc_run(ens._h, ens.state.data_ptr(), od.data_ptr(), T, ens._gi.data_ptr(), am.data_ptr(),
                                   tot.data_ptr(), ens._err.data_ptr(), nat.stream_ptr()), "prs_pc_run")
    assert np.array_equal(ens._err.cpu().numpy(), want)
    assert len(set(want[: len(bad)].tolist())) >= 3                  # the first networks carry different bits


@functools.lru_cache(maxsize=None)
def _multi_step(shape, B, T):
    """Accepted edge odometry (|og| <= 4) for T updates of B networks from the packet starts, and the oracle's trace."""
    starts = start_states(shape)
    ok = [(r[1], r[2]) for r in edge_cases(shape) if plan(shape, r[1], r[2])[4] == 0 and abs(plan(shape, r[1], r[2])[3]) <= 4]
    odom = np.array([[ok[(7 * b + 3 * t) % len(ok)] for b in range(B)] for t in range(T)])
    gis = np.array([float(np.float32(g)) for g in np.linspace(0.0, 0.03, B)])
    init = np.stack([starts[(0, 1, 3)[b % 3]] for b in range(B)])
    trace = []
    nets = [opc.PoseCellNetwork(shape, global_inhibition=float(g)) for g in gis]
    for n, s in zip(nets, init):
        n.posecells = s.copy()
    for t in range(T):
        am = [n.update(tuple(odom[t, b])) for b, n in enumerate(nets)]
        trace.append([(n.posecells.copy(), n.last_total, a) for n, a in zip(nets, am)])
    return init, gis, odom, trace


@pytest.mark.parametrize("shape,family,dtype", [c for c in COMBOS if c[0] in ((21, 21, 36), (50, 50, 10))
                                                and c[1] in ("resident", "pair", "cluster", "tiled")],
                         ids=[i for c, i in zip(COMBOS, COMBO_IDS) if c[0] in ((21, 21, 36), (50, 50, 10))
                              and c[1] in ("resident", "pair", "cluster", "tiled")])
def test_ten_updates_of_edge_odometry_on_the_fused_kernels(shape, family, dtype):
    """Ten consecutive updates with edge odometry (translations up to the radius bound, theta origins up to 4, origins
    on halves): what one update leaves in the kernel's carried state must not leak into the next."""
    B, T = 24, 10
    init, gis, odom, trace = _multi_step(shape, B, T)
    ens = _ensemble(shape, family, dtype, B, gis)
    ens.posecells = init
    od = torch.from_numpy(odom).to(ens.device)
    for t in range(T):
        ens.update_async(od[t])
        torch.cuda.synchronize()
        pc = ens.posecells
        total = ens._total.cpu().numpy().astype(np.float64)
        amax = ens._unravel(ens._argmax.cpu().numpy())
        assert not ens._err.cpu().numpy().any(), t
        for b in range(B):
            why = _check_network(pc[b], total[b], amax[b], trace[t][b], RTOL[dtype] * (1 + t))
            assert why is None, (t, b, why)


def test_overlapping_launches_of_edge_odometry_equal_serialised_launches():
    """120 back-to-back updates of 300 networks with edge odometry on the resident kernel (overlapping launches) give bit
    for bit the states, arg-max cells and totals of the same updates with a device synchronisation between them."""
    from pyratslam_b200 import PoseCellEnsemble
    shape, B, T = (21, 21, 36), 300, 120
    ok = [(r[1], r[2]) for r in edge_cases(shape) if plan(shape, r[1], r[2])[4] == 0 and abs(plan(shape, r[1], r[2])[3]) <= 4]
    odom = np.array([[ok[(7 * b + 3 * t) % len(ok)] for b in range(B)] for t in range(T)])
    od = torch.from_numpy(odom).cuda()
    gis = np.linspace(0.0, 0.03, B)
    a, c = (PoseCellEnsemble(shape, B, global_inhibition=gis) for _ in range(2))
    for e in (a, c):
        assert e.path == "resident"
        e.posecells = np.stack([start_states(shape)[(0, 1, 3)[b % 3]] for b in range(B)])
    amax_a, tot_a = [], []
    for t in range(T):
        a.update_async(od[t])
        torch.cuda.synchronize()
        amax_a.append(a._argmax.clone())
        tot_a.append(a._total.clone())
    seen = []
    for t in range(T):
        c.update_async(od[t])
        if t % 11 == 0:
            seen.append((t, c._argmax.clone(), c._total.clone()))
    torch.cuda.synchronize()
    assert torch.equal(a.state, c.state) and torch.equal(a._argmax, c._argmax) and torch.equal(a._total, c._total)
    for t, am, tot in seen:
        assert torch.equal(am, amax_a[t]) and torch.equal(tot, tot_a[t]), t
    assert int((a.state.reshape(B, -1).amax(1) > 0).sum()) == B       # no network died: the comparison means something


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_ensemble_replay_with_zero_and_negative_inhibition(dtype):
    """replay_ensemble (frame graphs, ensemble graphs) with gi <= 0 against the oracle's replay loop with the agent's gi."""
    from test_gpu_ros_ensemble import _check_agent, _inputs, _oracle
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 30
    frames, odom = _inputs(T)
    gis = [float(np.float32(g)) for g in (-0.005, 0.0, -0.002, -0.0)]   # no DoG cell within 1e-4 of its peak of gi
    thresholds, energies = (45000, 30000, 45000, 60000), (None, 0.3, None, 0.02)
    out = replay_ensemble(frames, odom, match_threshold=list(thresholds), global_inhibition=gis,
                          inject_energy=list(energies), dtype=dtype)
    for b, (thr, g, en) in enumerate(zip(thresholds, gis, energies)):
        _check_agent(out, b, _oracle(T, thr, g, en), RTOL[dtype], "gi %r" % g)
