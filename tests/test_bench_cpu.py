"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) must print ONE JSON line with the
B200 arm's metric / unit / config for the same workload, so that the driver can form the ratio of the two arms."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def _run(*extra):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", *extra],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_clip_workload_line():
    sys.path.insert(0, str(ROOT))
    import bench

    d = _run("--evals", "50", "--clips", "32")
    assert d["impl"] == "reference" and d["metric"] == "clips/sec" and d["unit"] == "clips/s" and d["higher_is_better"]
    assert d["config"] == bench.clip_config(50, 50, 32)          # identical to the B200 arm's config for these flags
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["e2e"] == {"value": d["value"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "sample" in d["cpu_baseline"] and d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_other_ranks_print_nothing(monkeypatch):
    import os

    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_budget_dtypes_and_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: small arrays whole with their shape, float32 unless float64; a large one as a sorted sample of its
    elements, the same sample on every run; the data never exceeds the budget"""
    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT))
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    arrays = {"image": (torch.arange(2 * 3 * 4) % 256).to(torch.uint8).reshape(2, 3, 4),
              "latents": torch.randn(2, 5).half(), "wave": torch.arange(5000, dtype=torch.float64)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert sorted(a) == ["image", "latents", "wave"]
    assert a["image"].dtype == np.float32 and np.array_equal(a["image"], arrays["image"].numpy())
    assert a["latents"].dtype == np.float32 and np.array_equal(a["latents"], arrays["latents"].float().numpy())
    w = a["wave"]
    assert w.dtype == np.float64 and w.ndim == 1 and 0 < w.size < 5000 and np.all(np.diff(w) > 0)   # distinct, in order
    assert sum(x.nbytes for x in a.values()) <= 4000
    for name, x in a.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{name}.npy"), x)


def test_workload_configs_and_eval_counts():
    """the img2img start-point arithmetic bench.py extrapolates with equals the reference's (riffusion_pipeline.py:358-396,
    SURVEY Appendix B: 38 evaluations at denoising 0.75, 50 at 1.0, 26 at 0.5) and the product scheduler's"""
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "riffusion-hobby_b200"))
    import bench
    from riffusion.scheduler_b200 import PNDMSchedulerB200

    assert [bench.n_evals_for(50, s) for s in (0.75, 1.0, 0.5)] == [38, 50, 26]
    sch = PNDMSchedulerB200()
    for steps, s in ((50, 0.75), (50, 1.0), (20, 0.7499999999999999), (8, 1.0)):
        sch.set_timesteps(steps)
        init = min(int(steps * s) + 1, steps)
        assert bench.n_evals_for(steps, s) == len(sch.timesteps[max(steps - init + 1, 0):])
    rt = bench.clip_config(50, 50, 16, "roundtrip")
    rf = bench.clip_config(50, 38, 1, "riffuse", 0.75)
    assert "configs[4]" in rt["workload"] and "configs[2]" in rf["workload"] and rt["clips_per_gpu"] == 16
