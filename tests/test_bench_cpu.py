"""bench.py's output without a GPU: the stdout line of a full run and the --dump-outputs sample."""
import json
import os
import sys
import types

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_result_line_stays_short():
    """A full record of a 1-GPU run (every section) gives a stdout line under 4 KB with the headline's keys and the
    summary of the further workloads last."""
    full = json.load(open(os.path.join(ROOT, "profiles", "bench_lines", "r2_n1_full.json")))
    text = json.dumps(bench.result_line(full))
    assert len(text.encode()) < 4096
    line = json.loads(text)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "verified", "clocks"):
        assert line[k] == full[k], k
    for k in ("roofline", "cpu_baseline", "e2e"):
        assert line[k] and line[k].items() <= full[k].items(), k
    assert line["e2e"]["h2d_bytes_per_step"] == full["e2e"]["h2d_bytes_per_step"]
    assert list(line)[-1] == "summary"
    assert line["summary"]["gs_1024_its"] == full["configs"]["gs_1024"]["value"]
    assert line["summary"]["c5_gs_its"] == full["configs"]["config5"]["value"]


def _state(torch, batch, shape, loops, seed=0):
    g = torch.Generator().manual_seed(seed)
    holo = torch.rand((batch,) + shape, generator=g, dtype=torch.float64)
    frames = (torch.rand((batch,) + shape, generator=g) * 255).to(torch.uint8)
    errors = [np.linspace(1.0, 0.5, loops) + b for b in range(batch)]
    return {"res": types.SimpleNamespace(hologram=holo, errors=errors), "out": frames}


def test_dump_outputs_sample(tmp_path):
    torch = pytest.importorskip("torch")
    st = _state(torch, 3, (512, 512), 7)
    bench.dump_outputs(str(tmp_path / "a"), st)
    bench.dump_outputs(str(tmp_path / "b"), _state(torch, 3, (512, 512), 7))
    out = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("hologram", "frames", "errors")}
    assert (out["hologram"].dtype, out["frames"].dtype, out["errors"].dtype) == (np.float64, np.float32, np.float64)
    assert out["hologram"].shape == out["frames"].shape == (3, 1 << 16) and out["errors"].shape == (3, 7)
    idx = np.sort(np.random.default_rng(0).choice(512 * 512, size=1 << 16, replace=False))
    np.testing.assert_array_equal(out["hologram"][2], st["res"].hologram[2].reshape(-1).numpy()[idx])
    np.testing.assert_array_equal(out["frames"][1], st["out"][1].reshape(-1).numpy()[idx].astype(np.float32))
    for n in out:                                       # the same inputs give the same files
        np.testing.assert_array_equal(out[n], np.load(tmp_path / "b" / f"{n}.npy"))


def test_dump_outputs_bounded(tmp_path):
    torch = pytest.importorskip("torch")
    bench.dump_outputs(str(tmp_path), _state(torch, 2048, (64, 64), 100))
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    assert np.load(tmp_path / "hologram.npy").shape == (2048, 2048)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"],
                                  ["--workload", "slab", "--dump-outputs", "x"]])
def test_parse_rejects(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()
