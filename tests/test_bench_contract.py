"""bench.py's command line.  The reference arm (`--impl reference`) needs no GPU: it runs here on a tiny budget (the
bounded-sample path) and its JSON line is checked against the contract; ranks > 0 of a torchrun launch must exit 0 without
output.  Arguments bench.py cannot honour are refused, and `--dump-outputs` writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", env.get("WORLD_SIZE", "1"),
                           "--steps", "1", "--warmup", "0", "--ref-budget-seconds", "1"], capture_output=True, text=True, timeout=900,
                          env=env, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "frames/sec SegNet(T)+ORB" and line["unit"] == "frames/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["steps"] == 1 and line["warmup"] == 0
    assert abs(line["ms_per_step"] * line["value"] - 1e3) < 1e-6 * 1e3
    assert line["config"]["workload"].startswith("Bayesian SegNet Basic T=6 + ORB(2000) x2")
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "T=2 of 6 samples" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29999"})
    assert r.returncode == 0 and r.stdout.strip() == "", (r.stdout[-500:], r.stderr[-500:])


def test_arguments_that_cannot_be_honoured_are_refused():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr[-500:])


def _fake_record(n_left, n_right, h=352, w=1024, cap=None):
    from sivo_b200 import record
    from sivo_b200.orb import KP_DTYPE
    rng = np.random.default_rng(7)
    cap = cap or max(n_left, n_right)
    mk = lambda n: np.array([tuple(rng.normal(size=5).astype(np.float32)) + (int(rng.integers(0, 8)), -1) for _ in range(n)], KP_DTYPE)
    buf = np.zeros(record.record_bytes(h * w, cap), np.uint8)
    record.pack_host(buf, h * w, cap, 5, rng.integers(0, 15, (h, w), dtype=np.uint8), rng.random((h, w)), rng.random((h, w)),
                     mk(n_left), rng.integers(0, 256, (n_left, 32), dtype=np.uint8), mk(n_right),
                     rng.integers(0, 256, (n_right, 32), dtype=np.uint8))
    return record.unpack(buf, h, w, cap)


def _load(out):
    got = {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    return got


def test_dump_outputs_writes_every_result_as_float(tmp_path):
    import bench
    rec = _fake_record(1200, 900)
    conf, ent = np.random.default_rng(1).random((2, 352, 1024))
    bench.dump_outputs(str(tmp_path / "out"), rec, conf, ent)
    got = _load(tmp_path / "out")
    assert sorted(got) == sorted(["classes", "confidence", "entropy", "record_confidence", "record_entropy", "keypoints_left",
                                  "descriptors_left", "keypoints_right", "descriptors_right"])
    assert np.array_equal(got["classes"], rec["classes"]) and np.array_equal(got["confidence"], conf) and np.array_equal(got["entropy"], ent)
    assert got["confidence"].dtype == np.float64 and np.array_equal(got["record_entropy"], rec["entropy"])
    for side in ("left", "right"):
        kp = rec["kp_" + side]
        assert got["keypoints_" + side].shape == (len(kp), 7) and got["descriptors_" + side].shape == (len(kp), 32)
        assert np.array_equal(got["keypoints_" + side][:, 0], kp["x"]) and np.array_equal(got["keypoints_" + side][:, 5], kp["octave"])
        assert np.array_equal(got["descriptors_" + side], rec["desc_" + side])
    assert sum(os.path.getsize(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")) < bench.DUMP_BYTES


def test_dump_outputs_samples_keypoints_to_stay_within_the_budget(tmp_path, monkeypatch):
    import bench
    rec = _fake_record(3000, 2500)
    maps = 352 * 1024 * (4 + 8 + 8 + 4 + 4)
    monkeypatch.setattr(bench, "DUMP_BYTES", maps + 2 * 1000 * 4 * (7 + 32))  # room for 1000 keypoints per image
    conf, ent = np.zeros((2, 352, 1024))
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), rec, conf, ent)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in a)  # a fixed sample
    assert sum(v.nbytes for v in a.values()) <= bench.DUMP_BYTES
    for side in ("left", "right"):
        kp, desc = rec["kp_" + side], rec["desc_" + side]
        assert len(a["keypoints_" + side]) == 1000 and len(np.unique(kp["x"])) == len(kp)
        # the kept rows are distinct rows of the record, in record order, the same rows for keypoints and descriptors
        idx = [int(np.flatnonzero(kp["x"] == x)[0]) for x in a["keypoints_" + side][:, 0]]
        assert idx == sorted(set(idx)) and len(idx) == 1000
        assert np.array_equal(a["keypoints_" + side][:, 4], kp["response"][idx])
        assert np.array_equal(a["descriptors_" + side], desc[idx])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs against a separate computation of the frame its last timed step ran: the same seeded model and
    frame through segmentImage and the synchronous extractor calls (both bit-identical to the device forms the bench times)."""
    import bench
    from sivo_b200 import BayesianSegNet, BayesianSegNetParams, ORBextractor
    steps, warmup = 3, 2
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
                        "--sustain-seconds", "0", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    got = _load(out)
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= bench.DUMP_BYTES
    # bench.py runs device_step 8 x 3 times to set up (8 input frames, 3 records), then warmup, then the timed steps; SegNet's
    # frame counter advances once per run
    i = warmup + steps - 1
    left, gl, gr = bench.frames(1, start=i % 8)[0]
    _, proto, model, _ = bench.model_files("basic", 6, str(tmp_path / "models"))
    seg = BayesianSegNet(BayesianSegNetParams(proto, model), seed=1234)
    seg.set_frame(8 * 3 + i)
    cls, conf, ent = seg.segmentImage(left)
    assert np.array_equal(got["classes"], cls) and np.array_equal(got["confidence"], conf) and np.array_equal(got["entropy"], ent)
    assert np.array_equal(got["record_confidence"], conf.astype(np.float32)) and np.array_equal(got["record_entropy"], ent.astype(np.float32))
    for side, gray in (("left", gl), ("right", gr)):
        kps, desc = ORBextractor(2000, 1.2, 8, 20, 7)(gray, None)
        assert len(kps) > 1000
        assert np.array_equal(got["keypoints_" + side], np.stack([kps[f].astype(np.float32) for f in kps.dtype.names], axis=1))
        assert np.array_equal(got["descriptors_" + side], desc)
