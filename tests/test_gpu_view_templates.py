"""GPU parity of the view-template matcher: template ids, create-vs-match decisions and scores are
bit-exact against the oracle / the reference-generated fixtures (integer arithmetic)."""
import numpy as np
import pytest
import torch

from oracle import view_templates as ovt
from synth import synth_frames

pytestmark = pytest.mark.gpu


def _vts(threshold=45000, **kw):
    from pyratslam_b200 import ViewTemplates
    return ViewTemplates((32, 96), (32, 96), 2, 2, 256, 256, threshold, **kw)


def test_golden_frame_sequence(golden):
    g = golden("view_templates.npz")
    vts = _vts()
    assert vts.shape == tuple(g["shape"]) and int(vts.mask.sum()) == int(g["mask_count"])
    T = int(g["n_frames"])
    frames = synth_frames(np.random.default_rng(int(g["frame_seed"])), T)
    for t in range(T):
        n0 = len(vts.templates)
        tm = vts.match(frames[t], t % 21, (2 * t) % 21, t % 36)
        assert tm.get_index() == g["index"][t], t
        assert (len(vts.templates) > n0) == bool(g["created"][t]), t
        assert (vts.last_score if vts.last_score is not None else -1) == g["best_score"][t], t
        assert len(vts.templates) == g["n_templates"][t]
    # stored templates are the sub-sampled frames, locations are what match() was given
    t3 = vts.templates[3]
    assert np.array_equal(t3.template, frames[3][vts.mask].reshape(32, 32))
    assert t3.location() == (3, 6, 3) and t3.get_index() == 3


def test_score_tables(golden):
    from pyratslam_b200 import ViewTemplate
    g = golden("view_templates.npz")
    lib, qs = g["lib_u8"], g["queries_u8"]
    vts = _vts()
    vts.load_library(lib)
    for qi, q in enumerate(qs):
        frame = np.zeros((256, 256), np.uint8)
        rows = np.arange(33, 96, 2)
        frame[np.ix_(rows, rows)] = q
        assert vts.scores(frame).tolist() == g["scores_u8"][qi].tolist()
        assert int(ViewTemplate(0, 0, 0, 0, lib[2]).match(q)) == g["scores_u8"][qi][2]
    vf = _vts()
    vf.load_library(lib.astype(np.float32))
    for qi, q in enumerate(qs):
        frame = np.zeros((256, 256), np.float32)
        frame[np.ix_(rows, rows)] = q
        assert vf.scores(frame).astype(np.float64).tolist() == g["scores_f64"][qi].tolist()


def test_threshold_is_strict(golden):
    g = golden("view_templates.npz")
    lib, qs = g["lib_u8"], g["queries_u8"]
    best = int(g["scores_u8"][3].min())
    rows = np.arange(33, 96, 2)
    f0 = np.zeros((256, 256), np.uint8)
    f1 = np.zeros((256, 256), np.uint8)
    f0[np.ix_(rows, rows)] = lib[int(g["scores_u8"][3].argmin())]
    f1[np.ix_(rows, rows)] = qs[3]
    out = []
    for thr in (best, best - 1):
        v = _vts(thr)
        out += [v.match(f0, 0, 0, 0).get_index(), v.match(f1, 0, 0, 0).get_index()]
    assert out == g["threshold_case"].tolist() == [0, 0, 0, 1]


def _sweep(lib_t, q_t, mode, want_scores=True):
    from pyratslam_b200 import _native as nat
    n = lib_t.shape[0]
    key = torch.zeros(1, dtype=torch.int64, device="cuda")
    if lib_t.dtype == torch.uint8:
        sc = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
        fn = nat.lib().prs_vt_sweep_u8
    else:
        sc = torch.zeros(max(n, 1), dtype=torch.float32, device="cuda")
        fn = nat.lib().prs_vt_sweep_f32
    nat.check(fn(lib_t.data_ptr() if n else None, n, q_t.data_ptr(), mode, 0, key.data_ptr(),
                 sc.data_ptr() if want_scores else None, None))
    torch.cuda.synchronize()
    return int(key.item()) & ((1 << 64) - 1), sc[:n].cpu().numpy()


@pytest.mark.parametrize("mode", ["ref", "circular"])
@pytest.mark.parametrize("n", [0, 1, 2, 3, 5, 64, 1001])
def test_ragged_library_sizes_u8(mode, n):
    rng = np.random.default_rng(100 + n)
    lib = rng.integers(0, 256, (n, 32, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (32, 32), dtype=np.uint8)
    if n > 3:
        lib[n - 1] = lib[2]                    # a tie: the lower index must win
        q = lib[2].copy()
    key, sc = _sweep(torch.from_numpy(lib).cuda(), torch.from_numpy(q).cuda(), 0 if mode == "ref" else 1)
    if n == 0:
        assert key == (1 << 64) - 1
        return
    ref = ovt.library_scores(lib, q, mode=mode)
    assert sc.view(np.uint32).astype(np.int64).tolist() == ref.astype(np.int64).tolist()
    assert key == (int(ref.min()) << 32) | int(np.argmin(ref))


def _sweep_packed(lib, q, mode, want_scores=True):
    """Pack a row-major uint8 library and sweep it through the bit-sliced kernels (C ABI)."""
    from pyratslam_b200 import _native as nat
    n = lib.shape[0]
    L = nat.lib()
    packed = torch.zeros(int(L.prs_vt_packed_bytes(max(n, 1))), dtype=torch.uint8, device="cuda")
    lib_t = torch.from_numpy(lib).cuda() if not isinstance(lib, torch.Tensor) else lib
    q_t = torch.from_numpy(q).cuda()
    nat.check(L.prs_vt_pack_u8(lib_t.data_ptr() if n else None, n, packed.data_ptr(), 0, None))
    key = torch.zeros(1, dtype=torch.int64, device="cuda")
    sc = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
    scratch = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    nat.check(L.prs_vt_sweep_packed_u8(packed.data_ptr() if n else None, n, q_t.data_ptr(), mode, 0, key.data_ptr(),
                                       sc.data_ptr() if want_scores else None, scratch.data_ptr(), None))
    torch.cuda.synchronize()
    return int(key.item()) & ((1 << 64) - 1), sc[:n].cpu().numpy().view(np.uint32).astype(np.int64), packed


@pytest.mark.parametrize("mode", ["ref", "circular"])
@pytest.mark.parametrize("n", [0, 1, 2, 31, 32, 33, 64, 1001, 2077])
def test_packed_library_matches_oracle(mode, n):
    rng = np.random.default_rng(200 + n)
    lib = rng.integers(0, 256, (n, 32, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (32, 32), dtype=np.uint8)
    if n > 3:
        lib[n - 1] = lib[2]                    # a tie: the lower index must win
        q = np.roll(lib[2], 3, axis=0)
        lib[0][5:9] = 0                        # extremes of the byte range
        lib[1][5:9] = 255
    key, sc, packed = _sweep_packed(lib, q, 0 if mode == "ref" else 1)
    if n == 0:
        assert key == (1 << 64) - 1
        return
    ref = ovt.library_scores(lib, q, mode=mode)
    assert sc.tolist() == ref.astype(np.int64).tolist()
    assert key == (int(ref.min()) << 32) | int(np.argmin(ref))
    # the packed layout round-trips
    from pyratslam_b200 import _native as nat
    out = torch.zeros((32, 32), dtype=torch.uint8, device="cuda")
    for i in sorted({0, n // 2, n - 1}):
        nat.check(nat.lib().prs_vt_unpack_u8(packed.data_ptr(), i, out.data_ptr(), None))
        assert np.array_equal(out.cpu().numpy(), lib[i])


def test_packed_equals_bytewise_kernel():
    """The two uint8 kernels (byte-wise SWAR and bit-sliced) agree on a 20 000-template library."""
    rng = np.random.default_rng(77)
    lib = rng.integers(0, 256, (20000, 32, 32), dtype=np.uint8)
    q = np.clip(lib[12345].astype(np.int16) - 3, 0, 255).astype(np.uint8)
    for mode in (0, 1):
        k1, s1 = _sweep(torch.from_numpy(lib).cuda(), torch.from_numpy(q).cuda(), mode)
        k2, s2, _ = _sweep_packed(lib, q, mode)
        assert k1 == k2 and s1.view(np.uint32).astype(np.int64).tolist() == s2.tolist()
    assert k2 & 0xFFFFFFFF == 12345


@pytest.mark.parametrize("mode", ["ref", "circular"])
def test_float32_library(mode):
    rng = np.random.default_rng(5)
    lib = rng.integers(0, 256, (777, 32, 32)).astype(np.float32)      # integer-valued: sums are exact
    q = np.roll(lib[400], 5 if mode == "ref" else 13, axis=0) + 0.0
    lib[600] = lib[400]
    key, sc = _sweep(torch.from_numpy(lib).cuda(), torch.from_numpy(q).cuda(), 0 if mode == "ref" else 1)
    ref = ovt.library_scores(lib, q, mode=mode)
    assert np.array_equal(sc, ref)
    j = int(np.argmin(ref))
    assert j == 400 and key & 0xFFFFFFFF == 400
    assert np.array([key >> 32], dtype=np.uint32).view(np.float32)[0] == ref[j]
    # non-integer data: same selection, scores within float32 summation error
    libr = rng.uniform(0, 255, (300, 32, 32)).astype(np.float32)
    qr = (libr[123] + rng.normal(0, 2, (32, 32))).astype(np.float32)
    key, sc = _sweep(torch.from_numpy(libr).cuda(), torch.from_numpy(qr).cuda(), 0 if mode == "ref" else 1)
    ref = ovt.library_scores(libr.astype(np.float64), qr.astype(np.float64), mode=mode)
    assert key & 0xFFFFFFFF == int(np.argmin(ref)) == 123
    assert np.abs(sc - ref).max() <= 1e-5 * ref.max()
    # ragged library sizes: the key is the oracle's arg-min and the smallest of the returned scores
    for n in (1, 31, 33, 2077):
        libn = rng.uniform(0, 255, (n, 32, 32)).astype(np.float32)
        qn = rng.uniform(0, 255, (32, 32)).astype(np.float32)
        key, sc = _sweep(torch.from_numpy(libn).cuda(), torch.from_numpy(qn).cuda(), 0 if mode == "ref" else 1)
        ref = ovt.library_scores(libn.astype(np.float64), qn.astype(np.float64), mode=mode)
        assert np.abs(sc - ref).max() <= 1e-4 * ref.max(), n
        assert key & 0xFFFFFFFF == int(np.argmin(ref)), n
        assert np.array([key >> 32], dtype=np.uint32).view(np.float32)[0] == sc.min(), n


def test_extract_matches_mask():
    rng = np.random.default_rng(1)
    frame = rng.integers(0, 256, (256, 256), dtype=np.uint8)
    vts = _vts()
    tm = vts.match(frame, 1, 2, 3)
    assert np.array_equal(tm.template, frame[vts.mask].reshape(32, 32))
    # torch frames already on the device take the same path
    tm2 = vts.match(torch.from_numpy(frame).cuda(), 1, 2, 3)
    assert tm2.get_index() == 0 and vts.last_score == 0


def test_million_template_library_properties():
    """BASELINE config 5 at full size (2^20 templates, 1 GiB): a planted darker, row-shifted copy is found;
    the key equals min/argmin of the per-template scores; a 4096-template slice equals the oracle."""
    n = 1 << 20
    g = torch.Generator(device="cuda").manual_seed(4)
    lib = torch.randint(0, 256, (n, 32, 32), dtype=torch.uint8, device="cuda", generator=g)
    target = 777_777
    src = lib[target].cpu().numpy()
    q = np.roll(np.clip(src.astype(np.int16) - 2, 0, 255).astype(np.uint8), -4, axis=0)
    key, sc = _sweep(lib, torch.from_numpy(q).cuda(), 0)
    sc = sc.view(np.uint32).astype(np.int64)
    assert key & 0xFFFFFFFF == target == int(np.argmin(sc)) and key >> 32 == int(sc.min())
    key_p, sc_p, _ = _sweep_packed(lib, q, 0)          # the bit-sliced layout the product streams
    assert key_p == key and np.array_equal(sc_p, sc)
    lo = 500_000
    ref = ovt.library_scores(lib[lo:lo + 4096].cpu().numpy(), q)
    assert sc[lo:lo + 4096].tolist() == ref.astype(np.int64).tolist()
    # circular mode finds any rotation exactly
    qc = np.roll(src, 19, axis=0)
    key, _ = _sweep(lib, torch.from_numpy(qc).cuda(), 1, want_scores=False)
    assert key == target                       # score 0, index target


def test_replay_loop_matches_reference_fixture(golden):
    from pyratslam_b200 import ros_simulate
    g = golden("replay_ros.npz")
    T = int(g["n_frames"])
    frames = synth_frames(np.random.default_rng(int(g["frame_seed"])), T)
    for dtype, fused, piped, native in ((np.float32, False, False, False), (np.float64, False, False, False),
                                        (np.float32, True, False, False), (np.float64, True, False, False),
                                        (np.float32, True, True, False), (np.float64, True, True, False),
                                        (np.float32, False, False, True), (np.float64, False, False, True)):
        rec = ros_simulate.replay(frames, g["odom"], fused=fused, pipelined=piped, native=native, dtype=dtype)
        assert np.array_equal(rec["template"], g["template"])
        assert np.array_equal(rec["created"], g["created"])
        assert np.array_equal(rec["argmax"], g["argmax"])
        assert np.array_equal(rec["n_exp"], g["n_exp"])
        assert np.allclose(rec["em_xy"][-1], g["em_xy"][-1], rtol=0, atol=0)
        fs = rec["node"].pcn.posecells
        assert np.abs(fs - g["final_state"]).max() / g["final_state"].max() <= (1e-5 if dtype == np.float32 else 1e-12)
        # the library holds the sub-sampled frames and the locations the reference would have stored
        node = rec["node"]
        first_created = int(np.flatnonzero(g["created"])[3])
        tm = node.vts.templates[int(g["template"][first_created])]
        assert np.array_equal(tm.template, frames[first_created][node.vts.mask].reshape(32, 32))
        assert tm.location() == tuple(g["argmax"][first_created])


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_other_template_shapes(dtype):
    """A configuration away from the reference's 32x32: (x_range, y_range) = ((20, 100), (40, 88)), step 2 -> 40x24."""
    from pyratslam_b200 import ViewTemplates
    args = ((20, 100), (40, 88), 2, 2, 128, 128, 30000 if dtype == np.uint8 else 9000.0)
    ref = ovt.ViewTemplates(*args)
    got = ViewTemplates(*args)
    assert got.shape == ref.shape == (40, 24) and np.array_equal(got.mask, ref.mask)
    rng = np.random.default_rng(8)
    frames = []
    for t in range(14):
        if t % 3 == 2:
            f = np.clip(frames[rng.integers(0, t)].astype(np.int16) - rng.integers(0, 3, (128, 128)), 0, 255)
        else:
            f = rng.integers(0, 256, (128, 128))
        frames.append(f.astype(dtype))
    for t, f in enumerate(frames):
        a = ref.match(f, t, 0, 0)
        b = got.match(f, t, 0, 0)
        assert a.get_index() == b.get_index() and len(ref.templates) == len(got.templates), t
    assert 3 < len(got.templates) < 14
    assert np.array_equal(got.templates[1].template, ref.templates[1].template)
    q = frames[5][ref.mask].reshape(ref.shape)
    assert float(got.templates[0].match(q)) == float(ref.templates[0].match(q))


def test_replay_with_template_injection():
    """SURVEY 8f row 2: the match -> pose-cell injection the reference left commented out (ros_simulate.py:106-108),
    against the oracle's replay with the same coupling; both the three-call and the fused loop."""
    from oracle import drivers as odrv
    from pyratslam_b200 import ros_simulate
    T = 20
    frames = synth_frames(np.random.default_rng(77), T)
    rng = np.random.default_rng(78)
    odom = np.stack([rng.uniform(0, 3.0, T), rng.uniform(-1, 1, T)], axis=1)
    odom[7] = 0.0
    ref = odrv.replay_run(frames, odom, inject_energy=0.02)
    for fused in (False, True):
        rec = ros_simulate.replay(frames, odom, fused=fused, inject_energy=0.02)
        assert np.array_equal(rec["template"], ref["template"]) and np.array_equal(rec["created"], ref["created"])
        assert np.array_equal(rec["argmax"], ref["argmax"])
        fs = rec["node"].pcn.posecells
        assert np.abs(fs - ref["final_state"]).max() / ref["final_state"].max() <= 1e-5


@pytest.mark.parametrize("compression", ["none", "bz2"])
def test_replay_from_rosbag(golden, tmp_path, compression):
    """SURVEY 8f row 1: the reference fixture's run written as a ROS1 bag (one Odometry + one Image per step),
    read back and replayed -- same decisions as the array replay; the recorded output topics match too."""
    from pyratslam_b200 import ros_simulate, rosbag_io as rb
    g = golden("replay_ros.npz")
    T = int(g["n_frames"])
    frames = synth_frames(np.random.default_rng(int(g["frame_seed"])), T)
    path = str(tmp_path / "run.bag")
    rb.write_run(path, frames, g["odom"], compression=compression, chunk_threshold=1 << 20)
    for fused in (False, True):
        out_path = str(tmp_path / ("out%d.bag" % fused))
        rec = ros_simulate.replay_bag(path, fused=fused, record=out_path)
        assert np.array_equal(rec["template"], g["template"]) and np.array_equal(rec["created"], g["created"])
        assert np.array_equal(rec["argmax"], g["argmax"]) and np.array_equal(rec["n_exp"], g["n_exp"])
        assert np.array_equal(rec["em_xy"][-1], g["em_xy"][-1])
        out = rb.BagReader(out_path)
        idx = [rb.decode_int32(m.data) for m in out.messages([rb.MATCH_TOPIC])]
        assert idx == g["template"].tolist()
        poses = [rb.decode_pose2d(m.data) for m in out.messages([rb.EM_TOPIC])]
        moved = (np.abs(g["odom"]) > 0.001).any(axis=1)
        assert len(poses) == int(moved.sum()) and poses[-1][:2] == tuple(g["em_xy"][-1])
    # messages that do not alternate: two twists before a frame, a frame without a twist
    ev = rb.read_events(path)[:40]
    ev = [ev[0], ev[2]] + ev[1:2] + ev[3:]
    a = ros_simulate.replay_events(ev, fused=False)
    b = ros_simulate.replay_events(ev, fused=True)
    for k in ("template", "created", "argmax", "n_exp", "em_xy"):
        assert np.array_equal(a[k], b[k]), k


def test_big_library_sweeps_back_to_back():
    """Six queries enqueued back to back, without a synchronisation, each with its own key and score buffers, against
    libraries big enough that every warp of the uint8 ring sweep refills its ring across groups (more than 94 720
    templates) and the float32 pair sweep wraps its three-slot ring (more than 7 104).  The bit-sliced sweeps equal
    the byte-wise kernel bit for bit; the float32 sweep of integer-valued profiles (exact sums) equals
    prs_vt_sweep_any_f32."""
    from pyratslam_b200 import _native as nat
    L = nat.lib()
    st = nat.stream_ptr()
    g = torch.Generator(device="cuda").manual_seed(12)
    n = (1 << 17) + 77
    lib = torch.randint(0, 256, (n, 32, 32), dtype=torch.uint8, device="cuda", generator=g)
    packed = torch.zeros(int(L.prs_vt_packed_bytes(n)), dtype=torch.uint8, device="cuda")
    nat.check(L.prs_vt_pack_u8(lib.data_ptr(), n, packed.data_ptr(), 0, st))
    nf = (1 << 17) + 5
    libf = torch.randint(0, 256, (nf, 32, 32), dtype=torch.float32, device="cuda", generator=g)

    def rand_u8():
        return torch.randint(0, 256, (32, 32), dtype=torch.uint8, device="cuda", generator=g)
    # (kind, mode, query, index of the planted template or None)
    sweeps = [("u8", 0, (lib[n - 3].to(torch.int16) - 2).clamp(0, 255).to(torch.uint8), n - 3),
              ("u8", 0, rand_u8(), None),
              ("u8", 1, torch.roll(lib[70000], 5, 0), 70000),
              ("u8", 1, rand_u8(), None),
              ("f32", 0, torch.roll(libf[nf - 1], 3, 0), nf - 1),
              ("f32", 0, rand_u8().to(torch.float32), None)]
    keys = torch.zeros(len(sweeps), dtype=torch.int64, device="cuda")
    scores, scratch = [], [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in sweeps]
    for i, (kind, mode, q, _) in enumerate(sweeps):
        if kind == "u8":
            scores.append(torch.zeros(n, dtype=torch.int32, device="cuda"))
            nat.check(L.prs_vt_sweep_packed_u8(packed.data_ptr(), n, q.data_ptr(), mode, 0, keys[i:].data_ptr(),
                                               scores[i].data_ptr(), scratch[i].data_ptr(), st))
        else:
            scores.append(torch.zeros(nf, dtype=torch.float32, device="cuda"))
            nat.check(L.prs_vt_sweep_f32(libf.data_ptr(), nf, q.data_ptr(), mode, 0, keys[i:].data_ptr(),
                                         scores[i].data_ptr(), st))
    torch.cuda.synchronize()
    for i, (kind, mode, q, planted) in enumerate(sweeps):
        want_key = torch.zeros(1, dtype=torch.int64, device="cuda")
        if kind == "u8":
            want = torch.zeros(n, dtype=torch.int32, device="cuda")
            nat.check(L.prs_vt_sweep_u8(lib.data_ptr(), n, q.data_ptr(), mode, 0, want_key.data_ptr(), want.data_ptr(),
                                        st))
        else:
            want = torch.zeros(nf, dtype=torch.float32, device="cuda")
            nat.check(L.prs_vt_sweep_any_f32(libf.data_ptr(), nf, q.data_ptr(), 32, 32, 8, 0, want_key.data_ptr(),
                                             want.data_ptr(), st))
        torch.cuda.synchronize()
        assert int(keys[i]) == int(want_key[0]), i
        assert torch.equal(scores[i].view(torch.int32), want.view(torch.int32)), i
        if planted is not None:
            assert int(keys[i]) & 0xFFFFFFFF == planted, i


def test_native_replay_matches_frame_by_frame():
    """prs_replay_run (the loop on the C side, zero-copy frame chain, small-library sweep) against the three
    reference-shaped calls per frame: identical records, library contents and experience map."""
    from pyratslam_b200 import ros_simulate
    T = 150
    frames = synth_frames(np.random.default_rng(5), T)
    rng = np.random.default_rng(6)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    odom[7] = (0.0005, -0.0002)          # below the 0.001 gate: no pose-cell update for this frame
    odom[8] = (0.0, 0.0)
    a = ros_simulate.replay(frames, odom)
    for n_plans in (1, 3):
        node = ros_simulate.RatslamRos()
        res = node.replay_native(frames, odom, n_plans=n_plans)
        assert res["template_index"].tolist() == a["template"].tolist()
        assert (res["created"] != 0).tolist() == a["created"].tolist()
        assert len(node.em.experiences) == len(a["node"].em.experiences)
        assert node.em.get_points() == a["node"].em.get_points()
        assert len(node.vts.templates) == a["n_templates"]
        i = int(np.flatnonzero(a["created"])[-1])
        tm, tr = node.vts.templates[int(a["template"][i])], a["node"].vts.templates[int(a["template"][i])]
        assert np.array_equal(tm.template, tr.template) and tm.location() == tr.location()
        assert node.pcn.get_pc_max() == a["node"].pcn.get_pc_max()
    b = ros_simulate.replay(frames, odom, native=True)
    for k in ("template", "created", "argmax", "n_exp", "em_xy"):
        assert np.array_equal(a[k], b[k]), k
    with pytest.raises(KeyError):       # vtrans = 0.1 after the /10 scaling: the reference's LUT hole
        bad = odom.copy()
        bad[20] = (1.0, 0.0)
        ros_simulate.replay(frames[:30], bad[:30], native=True)


def test_sharded_batch_matches_per_query():
    """ShardedViewTemplates.match_keys (one reduction and one read-back per batch) against match_key per query and the
    oracle, on a single rank (the multi-rank path runs in tests/multigpu_check.py)."""
    from pyratslam_b200 import ShardedViewTemplates
    rng = np.random.default_rng(21)
    n = 3001
    lib = rng.integers(0, 256, (n, 32, 32), dtype=np.uint8)
    qs = np.stack([np.clip(lib[1234].astype(np.int16) - 2, 0, 255).astype(np.uint8),
                   np.roll(lib[77], 3, axis=0), rng.integers(0, 256, (32, 32), dtype=np.uint8)])
    for mode in ("ref", "circular"):
        svt = ShardedViewTemplates(lib, 100, match_threshold=45000, mode=mode)      # base index 100: global indices
        got = svt.match_keys(torch.from_numpy(qs).cuda())
        assert got == [svt.match_key(torch.from_numpy(q).cuda()) for q in qs]
        for (score, idx), q in zip(got, qs):
            ref = ovt.library_scores(lib, q, mode=mode)
            assert (score, idx) == (int(ref.min()), 100 + int(np.argmin(ref)))
    svf = ShardedViewTemplates(lib.astype(np.float32), 0, match_threshold=9000.0)
    gotf = svf.match_keys(torch.from_numpy(qs.astype(np.float32)).cuda())
    assert [i for _, i in gotf] == [int(np.argmin(ovt.library_scores(lib.astype(np.float64), q.astype(np.float64)))) for q in qs]


def test_fused_frames_after_unfused_calls():
    """ADVICE r1: the frame plans cache the arg-max and the library size on the device.  A pose-cell update, an inject
    or a template append made OUTSIDE the plan (lone odometry message, vis_callback) between two fused frames must be
    seen by the next fused frame -- also when that frame's own twist is below the 0.001 gate (no update of its own).
    Reference for every step: the three reference-shaped calls on a second node."""
    from pyratslam_b200 import ros_simulate
    T = 14
    frames = synth_frames(np.random.default_rng(5), T)
    rng = np.random.default_rng(6)
    odom = np.stack([rng.uniform(0.5, 3.0, T), rng.uniform(-1, 1, T)], axis=1)
    a, b = ros_simulate.RatslamRos(), ros_simulate.RatslamRos()
    still = (0.0, 0.0)

    def plain(node, twist, im):
        if twist is not None:
            node.odom_callback(twist)
            node.spin_once()
        return node.vis_callback(im), tuple(int(c) for c in node.pcn.get_pc_max())

    for t in range(T):
        tw = (float(odom[t, 0]), float(odom[t, 1]))
        kind = t % 4
        if kind == 0:      # fused frame with its own update
            got = a.fused_frame(tw, frames[t]), tuple(int(c) for c in a.pcn.max_pc)
            want = plain(b, tw, frames[t])
        elif kind == 1:    # odom(moving) alone, then odom(sub-threshold) + image as ONE fused frame: the stale-cache case
            for node in (a, b):
                node.odom_callback(tw)
                node.spin_once()
            got = a.fused_frame(still, frames[t]), tuple(int(c) for c in a.pcn.max_pc)
            want = plain(b, None, frames[t])
        elif kind == 2:    # a template appended outside the plan, then a fused frame that must not overwrite its slot
            ra, rb_ = a.vis_callback(frames[t]), b.vis_callback(frames[t])
            assert ra == rb_
            got = a.fused_frame(tw, frames[(t + 5) % T]), tuple(int(c) for c in a.pcn.max_pc)
            want = plain(b, tw, frames[(t + 5) % T])
        else:              # inject outside the plan, then an image-only fused frame
            for node in (a, b):
                node.pcn.inject(0.5, (3, 4, 5))
            got = a.fused_frame(None, frames[t]), tuple(int(c) for c in a.pcn.max_pc)
            want = plain(b, None, frames[t])
        assert got == want, (t, kind, got, want)
    assert len(a.vts.templates) == len(b.vts.templates)
    for i in range(len(b.vts.templates)):
        assert np.array_equal(a.vts.templates[i].template, b.vts.templates[i].template), i
        assert a.vts.templates[i].location() == b.vts.templates[i].location(), i


def test_sharded_match_decides_on_device_single_rank():
    """ShardedViewTemplates.match through the fused exchange kernel (csrc/sharded.cu) on one rank: create-or-match,
    strict threshold, appends slot by slot (capacity growth included) -- against the oracle's ViewTemplates loop."""
    from pyratslam_b200 import ShardedViewTemplates
    rng = np.random.default_rng(33)
    for dtype, thr in ((np.uint8, 45000), (np.float32, 30000.0)):
        lib = rng.integers(0, 256, (40, 32, 32)).astype(dtype)
        svt = ShardedViewTemplates(lib[:0], 0, match_threshold=thr, capacity=32)
        assert svt.exchange == "fused"
        ref_lib = []
        for i in range(80):
            if i % 3 == 2 and ref_lib:
                src = ref_lib[int(rng.integers(0, len(ref_lib)))]
                q = np.clip(src.astype(np.int16) - rng.integers(0, 3, src.shape), 0, 255).astype(dtype)
            else:
                q = rng.integers(0, 256, (32, 32)).astype(dtype)
            if ref_lib:
                sc = ovt.library_scores(np.stack(ref_lib), q)
                j = int(np.argmin(sc))
                want = (len(ref_lib), True) if sc[j] > thr else (j, False)
            else:
                want = (0, True)
            if want[1]:
                ref_lib.append(q)
            assert svt.match(torch.from_numpy(q).cuda()) == want, (dtype, i)
        assert svt.n_total == len(ref_lib) > 32
        # threshold equality is a match (strict '>')
        q = ref_lib[3]
        s0 = int(ovt.library_scores(np.stack(ref_lib), q).min()) if dtype == np.uint8 else 0.0
        svt.match_threshold = s0
        assert svt.match(torch.from_numpy(q).cuda())[1] is False
        svt.close()


def test_two_streams_sweep_concurrently():
    """The packed sweeps read the query planes from ONE constant buffer per device; sweeps issued on two streams must
    not see each other's query (they are event-ordered on the device, csrc/view_templates.cu VtqScope)."""
    from pyratslam_b200 import _native as nat
    rng = np.random.default_rng(9)
    n = 20000
    lib = rng.integers(0, 256, (n, 32, 32), dtype=np.uint8)
    L = nat.lib()
    dlib = torch.from_numpy(lib).cuda()
    packed = torch.zeros(int(L.prs_vt_packed_bytes(n)), dtype=torch.uint8, device="cuda")
    nat.check(L.prs_vt_pack_u8(dlib.data_ptr(), n, packed.data_ptr(), 0, nat.stream_ptr()))
    qa = np.clip(lib[111].astype(np.int16) - 1, 0, 255).astype(np.uint8)
    qb = np.clip(lib[19000].astype(np.int16) - 1, 0, 255).astype(np.uint8)
    want = {}
    for name, q in (("a", qa), ("b", qb)):
        sc = ovt.library_scores(lib, q)
        want[name] = (int(sc.min()) << 32) | int(np.argmin(sc))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    qd = [torch.from_numpy(qa).cuda(), torch.from_numpy(qb).cuda()]
    keys = [torch.zeros(64, dtype=torch.int64, device="cuda") for _ in range(2)]
    scratch = [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    for it in range(64):
        for s in range(2):
            with torch.cuda.stream(streams[s]):
                nat.check(L.prs_vt_sweep_packed_u8(packed.data_ptr(), n, qd[s].data_ptr(), 0, 0,
                                                   keys[s][it:].data_ptr(), None, scratch[s].data_ptr(),
                                                   ctypes_stream(streams[s])))
    torch.cuda.synchronize()
    assert set(keys[0].tolist()) == {want["a"]} and set(keys[1].tolist()) == {want["b"]}


def ctypes_stream(s):
    import ctypes
    return ctypes.c_void_p(s.cuda_stream)


def test_replay_with_experience_links():
    """SURVEY 8f row 3 in the loop: every odometry update tagged with the latest template match, revisits close loops.
    Plain, fused and native replays build the same graph as the oracle's replay with the specification map."""
    from oracle import drivers as odrv
    from pyratslam_b200 import ros_simulate
    T = 72
    frames = synth_frames(np.random.default_rng(7), T)
    frames[36:] = frames[:36]                      # the second half revisits the first
    odom = np.zeros((T, 2))                        # rotate on the spot by one theta cell per step (vrot = angular.z / 10):
    odom[:, 1] = 2 * np.pi / 36 * 10 * 0.999       # after 36 steps the pose cells revisit as well
    ref = odrv.replay_run(frames, odom, experience_links=True)
    assert ref["em"].n_loop_closures > 20 and len(ref["em"].experiences) < T - 20
    ref["em"].iterate(5)
    for kw in ({}, {"fused": True}, {"native": True}):
        rec = ros_simulate.replay(frames, odom, experience_links=True, **kw)
        em = rec["node"].em
        assert np.array_equal(rec["template"], ref["template"]), kw
        assert em.n_loop_closures == ref["em"].n_loop_closures and len(em.experiences) == len(ref["em"].experiences), kw
        assert em.links == [(l.exp_from, l.exp_to, l.d, l.heading_rad, l.facing_rad) for l in ref["em"].links], kw
        em.iterate(5)
        assert em.get_poses() == ref["em"].get_poses(), kw


def test_smaller_frames_that_cover_the_mask():
    """ADVICE r1: the reference scenario publishes 128x128 frames against the 256x256 mask; every selected pixel (rows /
    columns 33..95) lies inside such a frame, and the reference's numpy accepted it.  Same templates and decisions as the
    padded 256x256 frame; a frame that does not cover the selection is numpy's IndexError."""
    rng = np.random.default_rng(4)
    a, b = _vts(), _vts()
    for i in range(6):
        small = rng.integers(0, 256, (128, 128), dtype=np.uint8)
        if i == 4:
            small = np.clip(first.astype(np.int16) - 1, 0, 255).astype(np.uint8)     # a revisit
        if i == 0:
            first = small
        big = np.zeros((256, 256), np.uint8)
        big[:128, :128] = small
        ta, tb = a.match(small, 1, 2, 3), b.match(big, 1, 2, 3)
        assert ta.get_index() == tb.get_index() and a.last_score == b.last_score
    assert len(a.templates) == len(b.templates) == 5
    assert np.array_equal(a.templates[2].template, b.templates[2].template)
    with pytest.raises(IndexError):
        a.match(np.zeros((90, 128), np.uint8), 0, 0, 0)
