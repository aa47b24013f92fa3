"""bench.py contract: the reference arm (the oracle port timed on host cores) prints ONE JSON line with the keys a
reader of the result needs, honours --steps/--warmup, and needs no GPU; --dump-outputs writes what the timed path
computed in its last step."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                                   "--warmup", "0"], cwd=ROOT, text=True, stderr=subprocess.DEVNULL, timeout=600)
    lines = [l for l in out.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "audio_seconds_per_second" and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1 and d["scaling"] == "weak"
    assert d["value"] > 0 and abs(d["value"] - 8.0 / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]   # 2 x 4 s per step
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_dump_outputs_writes_float_arrays(tmp_path):
    """bench.dump_outputs: one DIR/<name>.npy per tensor, floats as float32, integer codes as exact float64, size bound."""
    import numpy as np
    import torch
    import bench
    codes = torch.arange(12, dtype=torch.int64).reshape(1, 3, 4) * 97
    y = torch.randn(2, 1, 30, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "out"), {"y": y, "codes_r": codes})
    a, b = np.load(tmp_path / "out" / "y.npy"), np.load(tmp_path / "out" / "codes_r.npy")
    assert a.dtype == np.float32 and np.array_equal(a, y.float().numpy())
    assert b.dtype == np.float64 and np.array_equal(b, codes.numpy())
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"y": y}, limit_bytes=100)
    assert not (tmp_path / "big").exists()


def test_dump_outputs_rejects_other_arms():
    for extra in (["--impl", "reference"], ["--workload", "vq"], ["--steps", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "unused"] + extra, cwd=ROOT,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 2 and "usage" in r.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(built_lib, tmp_path):
    """The dump holds codec.forward's outputs for the input of the last timed step (batch (steps - 1) % 4 of the seeded
    rotation), and the run is deterministic: a second forward in this process gives the same bits."""
    import numpy as np
    import torch
    import facodec_b200 as fb
    from facodec_b200 import synth
    subprocess.check_call([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                           "--no-library-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT, stdout=subprocess.DEVNULL,
                          timeout=1200)
    got = {n: np.load(tmp_path / (n + ".npy")) for n in ("y", "codes_p", "codes_c", "codes_r", "timbre")}
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    sds = synth.synth_state_dicts(0)
    model = fb.build_model()
    for k in ("encoder", "quantizer", "decoder"):
        model[k].load_state_dict(sds[k])
        model[k].eval()
    x = synth.synth_waves(128, 96000, seed=114514)[32:64].contiguous().cuda()
    y, codes, timbre = fb.Codec(model).forward(x, n_c=2)
    want = dict(y=y, codes_p=codes[0], codes_c=codes[1], codes_r=codes[2], timbre=timbre)
    for n, t in want.items():
        assert got[n].shape == tuple(t.shape), n
        assert got[n].dtype == (np.float64 if n.startswith("codes") else np.float32), n
        assert np.array_equal(got[n], t.cpu().numpy().astype(got[n].dtype)), n
