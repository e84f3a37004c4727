"""The bench.py JSON contract, checked on the committed bench lines of the last round (profiles/) and on the
projection autograd node of the module (CPU, fp64) -- no GPU needed."""
import glob
import json
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = sorted(glob.glob(os.path.join(ROOT, "profiles", "r01e_bench_line*.json")) + glob.glob(os.path.join(ROOT, "profiles", "r02_bench_line*.json")))
LINES = [p for p in ALL if "reference_arm" not in p]
REF_LINES = [p for p in ALL if "reference_arm" in p]

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"]


@pytest.mark.parametrize("path", LINES, ids=[os.path.basename(p) for p in LINES])
def test_committed_bench_line_has_the_contract_fields(path):
    d = json.load(open(path))
    for key in REQUIRED:
        assert key in d, key
    assert d["metric"] == "cca_fwd_bwd_pixels_per_s" and d["unit"] == "pixels/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    assert "workload" in d["config"] and "model" not in d["config"]
    px = 8 * 97 * 97 * d["n_gpus"]
    assert abs(d["value"] - px / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]          # value is the whole-job aggregate
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    if os.path.basename(path).startswith("r02"):            # round 2: traffic parsed from the committed ncu summary, both ops reported
        assert r["traffic"] and r["traffic_source"].startswith("profiles/r02_tc_ncu_summary")
        assert r["op_fwd"]["frac"] > 0.38 and r["op_bwd"]["frac"] > 0.34 and r["other_dtype"]["dtype"] == "bf16"
        assert "module" in d and d["module"]["ms_per_step"] < 4.0
        if "error" not in (d.get("ccnet") or {"error": 1}):
            assert d["ccnet"]["train_images_per_s"] > 0 and d["ccnet"]["per_gpu_batch"] * d["n_gpus"] == 8
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 8 * 512 * 97 * 97 * 4 and e["d2h_bytes_per_step"] == 2 * e["h2d_bytes_per_step"]
    assert e["value"] < d["value"]                          # host copies + the module's projections are inside e2e
    assert d["gpu_launches"] > 0
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if d["n_gpus"] == 1 and d["cpu_baseline"] is not None:
        b = d["cpu_baseline"]
        assert b["kind"] in ("port", "reference") and b["cores"] >= 1 and b["value"] > 0 and b["sample"]


@pytest.mark.parametrize("path", REF_LINES, ids=[os.path.basename(p) for p in REF_LINES])
def test_committed_reference_arm_line(path):
    """`bench.py --impl reference`: same metric / unit / config as our arm, the CPU reference timed on the host cores."""
    d = json.load(open(path))
    same_round = [p for p in LINES if os.path.basename(p)[:3] == os.path.basename(path)[:3]]
    ours = json.load(open((same_round or LINES)[0]))
    assert d["impl"] == "reference" and d["metric"] == ours["metric"] and d["unit"] == ours["unit"]
    assert d["higher_is_better"] is True and d["config"]["workload"] == ours["config"]["workload"]
    b = d["cpu_baseline"]
    assert b["kind"] in ("port", "reference") and b["cores"] >= 1 and b["sample"] and b["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["value"] < 1e-2 * ours["value"]                # the point of the exercise


def test_qkv_projection_node_matches_the_three_convs():
    """ccnet_b200.module._QKVProject (one autograd node, GEMMs on the [pixels, C] view) == the reference's three
    nn.Conv2d 1x1 projections (functions.py:29,32,35), values and all gradients, in fp64 on the CPU."""
    from ccnet_b200.module import _QKVProject
    torch.manual_seed(0)
    x = torch.randn(2, 64, 5, 7, dtype=torch.float64).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    convs = [torch.nn.Conv2d(64, o, 1).double() for o in (8, 8, 64)]
    args = [t for c in convs for t in (c.weight, c.bias)]
    outs = _QKVProject.apply(x, *args)
    gs = [torch.randn_like(t) for t in outs]
    sum((o * g).sum() for o, g in zip(outs, gs)).backward()
    got = [x.grad.clone()] + [p.grad.clone() for p in args]
    x.grad = None
    for c in convs:
        c.zero_grad()
    refs = [c(x) for c in convs]
    sum((o * g).sum() for o, g in zip(refs, gs)).backward()
    want = [x.grad] + [p.grad for p in args]
    for o, r in zip(outs, refs):
        assert o.shape == r.shape and o.is_contiguous(memory_format=torch.channels_last)
        assert (o - r).abs().max().item() <= 1e-12
    for a, b in zip(got, want):
        assert a.shape == b.shape and (a - b).abs().max().item() <= 1e-10


def test_dump_outputs_writes_whole_or_fixed_samples_within_64mb(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files, small arrays whole in their NCHW shape, large ones as the documented
    seeded sample (same indices on every run), and the five op outputs of the flagship shape under 64 MB in all."""
    import numpy as np
    import bench
    B, C, H, W = (bench.CFG[n] for n in "BCHW")
    numels = [B * C * H * W, B * H * W, B * C // 8 * H * W, B * C // 8 * H * W, B * C * H * W]    # out, lse, dq, dk, dv
    assert sum(4 * min(n, bench.DUMP_MAX_ELEMS) for n in numels) <= 64 << 20
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 100)
    big = torch.randn(2, 8, 5, 6).contiguous(memory_format=torch.channels_last)
    small = torch.randn(2, 5, 6, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("big", "small")}
    assert all(v.dtype == np.float32 for v in got.values())
    assert got["small"].shape == (2, 5, 6) and np.array_equal(got["small"], small.float().numpy())
    idx = np.sort(np.random.default_rng(0).choice(big.numel(), 100, replace=False))
    assert np.array_equal(got["big"], big.contiguous().view(-1).numpy()[idx])
    assert all(np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy")) for n in got)
