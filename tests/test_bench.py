"""bench.py --dump-outputs: the byte budget and the fixed sample (CPU), and on the GPU the dump of a short run
against the CPU oracle on the inputs of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_budget_and_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    big = torch.arange(3000, dtype=torch.float32).reshape(30, 100)
    tensors = {"big": big, "small": torch.rand(2, 5), "loss": torch.tensor(1.5, dtype=torch.float64),
               "idx": torch.arange(5, dtype=torch.int32), "mask": torch.tensor([True, False])}
    written = bench.dump_outputs(tensors, str(tmp_path / "a"))
    bench.dump_outputs(tensors, str(tmp_path / "b"))
    got = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in tensors}
    assert sum(a.nbytes for a in got.values()) <= 4000
    for k in ("small", "loss", "idx", "mask"):        # within their share: whole, in their shape
        assert got[k].shape == tuple(tensors[k].shape) and np.array_equal(got[k], tensors[k].double().numpy())
    assert got["small"].dtype == np.float32 and got["mask"].dtype == np.float32
    assert got["loss"].dtype == np.float64 and got["idx"].dtype == np.float64
    n = got["big"].size                                # the rest of the budget, as a sample of the flat array
    assert got["big"].dtype == np.float32 and 0 < n < big.numel() and written["big"] == [[30, 100], n]
    idx = np.sort(np.random.default_rng(0).choice(big.numel(), n, replace=False))
    assert np.array_equal(got["big"], big.numpy().reshape(-1)[idx])
    for k in tensors:
        assert np.array_equal(got[k], np.load(str(tmp_path / "b" / (k + ".npy"))))


def test_result_tensors_flattens_tuples_and_names_the_rest():
    a, b, c = torch.zeros(2), torch.ones(3), torch.full((1,), 2.0)
    tensors, skipped = bench.result_tensors({"out": a, "keep": (b, c, None), "note": "text"})
    assert list(tensors) == ["out", "keep_0", "keep_1"] and skipped == ["keep_2", "note"]
    assert tensors["out"] is a and tensors["keep_0"] is b and tensors["keep_1"] is c


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """cfg1 for exactly 3 timed steps over the 3 input sets: the dump holds the results of set 2."""
    out = tmp_path / "out"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "3",
                          "--warmup", "1", "--no-cpu-baseline", "--e2e-steps", "1", "--dump-outputs", str(out)],
                         cwd=str(tmp_path), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["rounds_ms"]["n"] == 1 and line["gpu_launches"] == 2 * 3
    assert line["warmup"] == 3 + 3                     # at least 3 warm-up steps, then the untimed pass of 3
    assert sorted(os.listdir(str(out))) == ["corr.npy", "v_aligned.npy", "v_maps.npy", "x_aligned.npy"]
    d = bench.Cfg1().host_inputs(17 * 2)
    xa, va, vm = oracle.dfpn_align_tail(d["x_refs"], d["m_refs"], d["m_target"], d["flow"])
    for name, ref in (("x_aligned", xa), ("v_aligned", va), ("v_maps", vm)):
        assert np.array_equal(np.load(str(out / (name + ".npy"))), ref), name
    corr = np.load(str(out / "corr.npy"))
    ref = oracle.corr4d(d["feats_t"], d["v_t16"], d["feats_r"], d["v_r16"])
    assert corr.size == ref.size and np.abs(corr.reshape(-1) - ref.reshape(-1)).max() <= 2e-3
