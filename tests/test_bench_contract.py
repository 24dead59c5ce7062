"""bench.py contract pieces: the reference arm prints exactly one JSON line with the required keys (no GPU), and
``--dump-outputs`` writes the outputs of the last timed step (gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--workload", "C1"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("distill fwd+bwd") and d["higher_is_better"] is True
    # the arm times the UNMODIFIED reference (oracle/_ref, or the tree MAFED_REFERENCE names) at the full shard; where
    # neither is present it times the oracle restatement and must say so
    from oracle import ref_harness as R
    kind, what = ("reference", "unmodified reference") if R.available() else ("port", "reference files absent")
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "B=8 of 8 samples" in d["cpu_baseline"]["sample"] and what in d["cpu_baseline"]["sample"]
    assert d["steps"] == 1 and d["warmup"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] and "model" not in d["config"] and d["vs_baseline"] is None


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """``--dump-outputs``: the loss of the JSON line, the per-layer losses, the batch masks and a sample of every
    gradient, float32 / float64, under 64 MB, consistent with each other."""
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-c5",
                          "--no-other-workloads", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    a = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(a) == ["grad_row_index", "grad_row_sums", "grad_rows", "image_masks", "lang_masks", "layer_losses", "loss"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    L, B, T, D = d["config"]["layers_distilled"], d["config"]["per_gpu_batch"], d["config"]["T"], d["config"]["D"]
    n_vis = d["config"]["n_vis"]
    assert float(a["loss"]) == d["loss"]
    assert a["layer_losses"].shape == (L,) and np.isfinite(a["layer_losses"]).all() and (a["layer_losses"] > 0).all()
    # all-ones attention mask: every visual token is an image token, every text token a language token
    assert a["image_masks"].shape == a["lang_masks"].shape == (B, T)
    assert (a["image_masks"][:, :n_vis] == 1).all() and (a["image_masks"][:, n_vis:] == 0).all()
    assert (a["lang_masks"] == 1 - a["image_masks"]).all()
    rows, index, sums = a["grad_rows"], a["grad_row_index"].astype(np.int64), a["grad_row_sums"]
    assert rows.shape == (L, len(index), D) and sums.shape == (L, B, T)
    assert len(index) > 0 and (np.diff(index) > 0).all() and np.isfinite(rows).all() and np.abs(rows).max() > 0
    np.testing.assert_allclose(rows.astype(np.float64).sum(-1), sums.reshape(L, B * T)[:, index], rtol=1e-9, atol=1e-12)

    # ... and they are the step on bench's own seeded inputs: the oracle, run on them under bf16 autocast as the
    # reference runs it, within the bf16 tolerance
    import importlib.util

    import torch

    from oracle import distill_oracle as O
    keep = sys.dont_write_bytecode
    spec = importlib.util.spec_from_file_location("bench_inputs", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    sys.dont_write_bytecode = keep
    st, te, am = bench.make_device_inputs(d["config"]["id"], 0, torch.device("cuda", 0))
    cfg = O.OracleConfig(modality_strategy="balanced", layer_strategy="discounted", gamma=0.5, num_hidden_layers=L,
                         distillation_layer=None, loss="mse", num_vision_tokens=n_vis)
    ref = O.forward_backward(st, te, am, cfg, autocast_bf16=True)
    del st, te
    assert float(a["loss"]) == pytest.approx(float(ref["loss"]), rel=2e-3)
    np.testing.assert_allclose(a["layer_losses"], [float(ref["layer_losses"][l]) for l in range(L)], rtol=2e-3)
    idx = torch.from_numpy(index).cuda()
    for l in range(L):
        want = ref["grads"][l].reshape(B * T, D)[idx].double().cpu().numpy()
        assert np.linalg.norm(rows[l] - want) <= 2e-3 * np.linalg.norm(want), l


def test_non_rank0_reference_arm_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""
