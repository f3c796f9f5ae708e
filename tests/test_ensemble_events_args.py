"""Message-stream ensemble replay without CUDA: the tick compaction, the validation of streams and parameters, the
bag helpers iter_events / write_events, the message-loop specification against replay_run on alternating streams,
and the CLI's --all-messages."""
import numpy as np
import pytest

from event_oracle import replay_events_run
from pyratslam_b200 import ros_ensemble
from pyratslam_b200 import rosbag_io as rb
from pyratslam_b200.ros_ensemble import event_streams, event_ticks, replay_ensemble_events


def _img(v):
    return np.full((256, 256), v, np.uint8)


def _odom(x, z=0.0):
    return ("odom", (0, 0), (x, z))


def _image(v):
    return ("image", (0, 0), _img(v))


def _ticks(events):
    fr, od, mv, im = event_ticks(events)
    return [int(f[0, 0]) for f in fr], od.tolist(), mv.tolist(), im.tolist()


def test_odometry_odometry_image():
    fr, od, mv, im = _ticks([_odom(1.5), _odom(2.0, 0.5), _image(7)])
    assert fr == [7] and mv == [1, 1] and im == [False, True] and od == [[1.5, 0.0], [2.0, 0.5]]


def test_image_image_and_leading_image():
    fr, od, mv, im = _ticks([_image(1), _image(2), _odom(2.0), _image(3)])
    assert fr == [1, 2, 3] and mv == [0, 0, 1] and im == [True, True, True] and od[2] == [2.0, 0.0]


def test_gated_out_twists_make_no_tick():
    fr, od, mv, im = _ticks([_odom(0.0005, -0.0002), _odom(0.0), _odom(0.0), _image(4), _odom(1e-4)])
    assert fr == [4] and mv == [0] and im == [True] and od == [[0.0, 0.0]]     # the image's own, image-only tick


def test_trailing_odometry():
    fr, od, mv, im = _ticks([_odom(1.0), _image(1), _odom(2.0), _odom(0.0), _odom(0.0, -3.0)])
    assert fr == [1] and mv == [1, 1, 1] and im == [True, False, False] and od[1:] == [[2.0, 0.0], [0.0, -3.0]]


def test_empty_streams():
    fr, od, mv, im = event_ticks([])
    assert fr.shape == (0, 256, 256) and od.shape == (0, 2) and len(mv) == len(im) == 0
    fr, od, mv, im = event_ticks([_odom(0.0), _odom(0.0001)])
    assert fr.shape == (0, 256, 256) and len(mv) == 0


def test_stream_validation():
    for bad in ([("laser", (0, 0), 1)], [_image(1)[:2]], [("image", (0, 0), np.zeros((128, 256), np.uint8))],
                [("image", (0, 0), np.zeros((256, 256), np.int16))], [("odom", (0, 0), ("a", 1))],
                [("odom", (0, 0), (1.0,))], "odom", 5):
        with pytest.raises(ValueError):
            event_ticks(bad)
    s = [_odom(1.0), _image(1)]
    assert len(event_streams(s, 1)) == 1 and len(event_streams([s, [], s], 3)) == 3
    for bad, R in (([s, s], 3), (s, 2), ([s], 2), ("xy", 2)):
        with pytest.raises(ValueError):
            event_streams(bad, R)


def test_replay_ensemble_events_validation():
    s = [_odom(1.0), _image(1)]
    for kw in ({"experience_map": True}, {"experience_map": "host"}, {"mode": "circular"},
               {"match_threshold": [1, 2], "global_inhibition": [0.1, 0.2, 0.3]}, {"inject_energy": -1.0},
               {"recording": 1}, {"n_agents": 2, "recording": [0, 2]}):
        with pytest.raises(ValueError):
            replay_ensemble_events(s, **kw)
    with pytest.raises(ValueError):
        replay_ensemble_events([s, s], recording=[0, 2])
    with pytest.raises(ValueError):
        replay_ensemble_events([("image", (0, 0), np.zeros((8, 8), np.uint8))])


def _stream(rng, n_img, per_image, trailing=2):
    """Images with 0..per_image twists before each (some below the gate) and odometry after the last."""
    ev, ns = [], 0
    for i in range(n_img):
        for _ in range(int(rng.integers(0, per_image + 1))):
            ns += 1000
            tw = (float(rng.uniform(0, 3)), float(rng.uniform(-1, 1))) if rng.random() > 0.15 else (0.0, 0.0)
            ev.append(("odom", (ns // 10 ** 9, ns % 10 ** 9), tw))
        ns += 1000
        ev.append(("image", (ns // 10 ** 9, ns % 10 ** 9), rng.integers(0, 256, (256, 256), dtype=np.uint8)))
    for _ in range(trailing):
        ns += 1000
        ev.append(("odom", (ns // 10 ** 9, ns % 10 ** 9), (float(rng.uniform(0, 3)), 0.25)))
    return ev


def _same_events(a, b):
    assert len(a) == len(b)
    for (ka, sa, pa), (kb, sb, pb) in zip(a, b):
        assert ka == kb and tuple(sa) == tuple(sb)
        if ka == "image":
            assert np.array_equal(pa, pb)
        else:
            assert tuple(pa) == tuple(pb)


def test_write_events_round_trip(tmp_path):
    ev = _stream(np.random.default_rng(1), 9, 3)
    path = str(tmp_path / "ev.bag")
    rb.write_events(path, ev)
    _same_events(rb.read_events(path), ev)
    rb.write_events(path, [])
    assert rb.read_events(path) == []
    with pytest.raises(ValueError):
        rb.write_events(str(tmp_path / "bad.bag"), [("laser", (0, 0), 1)])


@pytest.mark.parametrize("chunk", [1, 2, 4, 9, 50])
def test_iter_events_pieces_concatenate_to_read_events(tmp_path, chunk):
    ev = _stream(np.random.default_rng(2), 9, 3)
    path = str(tmp_path / "ev.bag")
    rb.write_events(path, ev)
    pieces = list(rb.iter_events(path, chunk))
    assert all(sum(k == "image" for k, _, _ in p) <= chunk for p in pieces)
    assert all(sum(k == "image" for k, _, _ in p) == chunk for p in pieces[:-1])
    _same_events([e for p in pieces for e in p], rb.read_events(path))
    with pytest.raises(ValueError):
        next(rb.iter_events(path, 0))


def test_specification_equals_replay_run_on_alternating_streams(tmp_path):
    from oracle import drivers as odrv
    from synth import synth_frames
    rng = np.random.default_rng(4)
    T = 10
    frames = synth_frames(rng, T)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    odom[4] = (0.0, 0.0)
    path = str(tmp_path / "run.bag")
    rb.write_run(path, frames, odom)
    events = rb.read_events(path)
    f, o, _ = rb.events_to_arrays(events)
    for links, energy in ((False, None), (True, 0.3)):
        want = odrv.replay_run(f, o, inject_energy=energy, experience_links=links)
        got = replay_events_run(events, inject_energy=energy, experience_links=links)
        for k in ("template", "created", "argmax", "n_exp", "em_xy"):
            assert np.array_equal(got[k], want[k]), (links, k)
        assert got["n_templates"] == want["n_templates"]
        assert np.array_equal(got["final_state"], want["final_state"])


def test_cli_all_messages(monkeypatch, capsys):
    calls = []

    def fake(bags, chunk, image_topic, odom_topic, recording, **kw):
        calls.append((list(bags), chunk, recording, kw["n_agents"], kw["experience_map"], kw["experience_links"]))
        B = kw["n_agents"]
        return (np.arange(B), np.zeros(B, np.int64), np.array([7] * len(bags)), [(1, 2, 3)] * B, np.full(B, 5),
                np.full(B, 2))
    monkeypatch.setattr(ros_ensemble, "_replay_all_messages", fake)
    ros_ensemble.main(["a.bag", "--all-messages", "--match-threshold", "1,2"])
    ros_ensemble.main(["a.bag", "b.bag", "--all-messages", "--chunk", "16", "--experience-links"])
    assert calls == [(["a.bag"], None, [0, 0], 2, "device", False), (["a.bag", "b.bag"], 16, [0, 1], 2, "device", True)]
    lines = capsys.readouterr().out.splitlines()
    assert len(lines) == 4
    assert lines[1].startswith("agent 1  match_threshold 2 ") and lines[1].endswith(
        "created 0/7  final arg-max (1, 2, 3)  experiences 5")
    assert lines[3].startswith("bag b.bag  agent 1 ") and lines[3].endswith("experiences 5  loop closures 2")
    for bad in ("0", "x"):
        with pytest.raises(SystemExit):
            ros_ensemble.main(["a.bag", "--all-messages", "--chunk", bad])
