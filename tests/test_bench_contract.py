"""bench.py's output contract, exercised on CPU through the reference arm (the one arm that runs without a GPU):
exactly one JSON line on stdout with the keys the driver reads; the product arm refuses to run without CUDA."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=600, env=env)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--height", "64", "--width", "96", "--ref-batch", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_images_per_sec_480x640" and d["unit"] == "img/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"
    cb = d["cpu_baseline"]
    # "reference": the unmodified reference model was importable (oracle.ref_import); "port": its restatement
    from oracle import ref_import
    want = "reference" if ref_import.reference_src() is not None else "port"
    assert cb["kind"] == want and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_and_dump_outputs_of_the_reference_arm_are_refused():
    r = _run("--impl", "reference", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run("--impl", "reference", "--dump-outputs", "out")
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


def test_dump_outputs_reset_state_and_gradient_sample(tmp_path, monkeypatch):
    """--dump-outputs runs the timed step again from the seeded state: reset_state() must give exactly what a fresh
    model and a fresh Adam give, and the gradient sample must be a fixed one."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench

    def fresh():
        torch.manual_seed(0)
        return torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.BatchNorm1d(16), torch.nn.Linear(16, 4))

    x = torch.randn(5, 8)

    def step(model, opt):
        loss = model(x).square().mean()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss.item()

    model = fresh()
    opt = torch.optim.Adam(model.parameters(), 1e-2)
    state0 = {k: t.detach().clone() for k, t in model.state_dict().items()}
    for _ in range(3):
        step(model, opt)
    bench.reset_state(model, opt, state0)
    got = [step(model, opt), bench.grad_sample(model), step(model, opt)]
    ref_model = fresh()
    ref_opt = torch.optim.Adam(ref_model.parameters(), 1e-2)
    want = [step(ref_model, ref_opt), bench.grad_sample(ref_model), step(ref_model, ref_opt)]
    assert got[0] == want[0] and got[2] == want[2] and np.array_equal(got[1], want[1])
    for (k, a), b in zip(model.state_dict().items(), ref_model.state_dict().values()):
        assert torch.equal(a, b), k

    flat_g = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).numpy()
    assert np.array_equal(bench.grad_sample(model), flat_g)          # fewer elements than the sample: all of them
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 50)
    ga = bench.grad_sample(model)
    assert ga.dtype == np.float32 and ga.shape == (50,) and np.array_equal(ga, bench.grad_sample(model))
    assert np.isin(ga, flat_g).all()
    bench.dump_outputs(str(tmp_path / "d"), [got[0], got[2]], ga)
    loss = np.load(tmp_path / "d" / "loss.npy")
    assert loss.dtype == np.float64 and loss.tolist() == [got[0], got[2]]
    assert np.array_equal(np.load(tmp_path / "d" / "grads.npy"), ga)


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
