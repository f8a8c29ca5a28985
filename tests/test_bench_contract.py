"""CPU tier: the parts of bench.py's contract that do not need a GPU -- the reference arm (`--impl reference`: the
reference's CPU Dslash on the host cores, one JSON line with the agreed keys; under torchrun only rank 0 works) and the
rule that a torchrun rank never inherits an OpenMP thread binding (round 2 lost ~70 GPU-minutes to every rank's launch
thread being pinned to core 0)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env_extra=None):
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_PROC_BIND", "OMP_PLACES"):
        env.pop(k, None)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dim", "8", "8", "8", "8"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "wilson_dslash_gflops" and d["unit"] == "GFLOP/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and "sample" in cb
    assert cb["pinning"]["OMP_PROC_BIND"] == "close"  # the CPU arm pins its OpenMP threads


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dim", "8", "8", "8", "8", "--gpus", "2"],
             {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_torchrun_ranks_are_never_pinned():
    code = "import os, sys; sys.argv = ['bench.py', '--gpus', '2']; sys.path.insert(0, %r); import bench; " \
           "print(os.environ.get('OMP_PROC_BIND'), os.environ.get('OMP_PLACES'))" % ROOT
    for rank in ("0", "1"):
        env = dict(os.environ)
        env.pop("OMP_PROC_BIND", None)
        env.pop("OMP_PLACES", None)
        env.update({"RANK": rank, "WORLD_SIZE": "2", "LOCAL_RANK": rank})
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
        assert out.returncode == 0, out.stderr[-1000:]
        assert out.stdout.split() == ["None", "None"], out.stdout


def test_dump_outputs(tmp_path):
    """--dump-outputs: native buffers back in [site][spin][colour][re,im] order in the precision's real type, and above the
    byte budget the same seeded sample of sites at every call"""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from quda_b200 import fields as F
    Vh = 64
    host = [np.random.default_rng(i).random((Vh, 4, 3, 2)) for i in range(3)]
    for prec, dt in ((8, np.float64), (4, np.float32), (2, np.float32)):
        bufs = [torch.from_numpy(F.spinor_to_native(h, prec, rotate=False)) for h in host]
        bench.dump_outputs(str(tmp_path), "one", bufs[:1], prec, Vh, bench.DUMP_BYTES)
        one = np.load(tmp_path / "one.npy")
        assert one.dtype == dt and one.shape == (Vh, 4, 3, 2)
        assert np.array_equal(one, F.spinor_from_native(bufs[0].numpy(), Vh, prec, rotate=False))
        bench.dump_outputs(str(tmp_path), "all", bufs, prec, Vh, bench.DUMP_BYTES)
        assert np.load(tmp_path / "all.npy").shape == (3, Vh, 4, 3, 2)
        budget = 50 * 24 * np.dtype(dt).itemsize
        samples = []
        for _ in range(2):
            bench.dump_outputs(str(tmp_path), "sample", bufs, prec, Vh, budget)
            samples.append(np.load(tmp_path / "sample.npy"))
        assert samples[0].shape == (50, 4, 3, 2) and samples[0].nbytes <= budget
        assert np.array_equal(samples[0], samples[1])


def test_dump_outputs_and_steps_are_checked():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"], ["--op", "cg", "--dump-outputs", "d"]):
        r = _run(args)
        assert r.returncode == 2 and "error" in r.stderr, (args, r.stderr[-1000:])


def test_process_grid_defaults():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.process_grid(1) == [1, 1, 1, 1]
    assert bench.process_grid(2) == [1, 1, 1, 2]
    assert bench.process_grid(4) == [1, 1, 2, 2]
    assert bench.process_grid(8) == [1, 2, 2, 2]
