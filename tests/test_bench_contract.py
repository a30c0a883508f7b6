"""bench.py's command line on tiny workloads: the reference arm (the one arm that runs without a GPU) prints one JSON line
with the contract's keys and times as many steps as --steps asks, bad arguments are refused, and on a GPU --dump-outputs
writes what the last timed steps computed, the same arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_contract():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--log-n-msm", "12", "--log-n-ntt", "10"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-500:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "MSM/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "sample" in line["cpu_baseline"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["value"] > 0 and line["ntt"]["value"] > 0 and "workload" in line["config"]
    assert line["steps"] == 2 and line["ntt"]["steps"] == 2 and line["cpu_baseline"]["steps"] == 2


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_bad_arguments_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert p.returncode == 2 and "error" in p.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_are_the_last_steps_results(tmp_path):
    """--dump-outputs writes what the last timed step of the device-resident legs returned, as exact float64 halves of the u64
    limbs: the MSM equals the oracle's MSM of the same generated pairs, the sampled rows of the forward NTT equal the oracle's
    transform applied warmup + steps times to the generated input, and the inverse NTT's rows equal that input again.  2^17
    NTT rows exercise the seeded 2^16-row sample.  Two runs with the same arguments write the same arrays."""
    import torch

    import algebra_b200 as ab
    from algebra_b200 import _lib
    from oracle import coracle as C
    seed, log_msm, log_ntt, warmup, steps = 12345, 12, 17, 1, 2
    lines = []
    for run in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                            "--log-n-msm", str(log_msm), "--log-n-ntt", str(log_ntt), "--seed", str(seed), "--no-cpu-baseline",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-500:]
        lines.append(json.loads(p.stdout.strip().splitlines()[-1]))
    line = lines[0]
    assert line["steps"] == steps and line["e2e"]["steps"] == steps
    assert line["config"]["verified_vs_sum_identity"] is True and line["ntt"]["roundtrip_ok"] is True
    shapes = {"msm_affine": (24,), "ntt_fft": (1 << 16, 8), "ntt_ifft": (1 << 16, 8)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(k + ".npy" for k in shapes)
    got = {}
    for name, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float64 and a.shape == shape, name
        assert np.array_equal(a, b), name
        got[name] = a

    def halves(u64):
        return np.ascontiguousarray(u64, dtype=np.uint64).view(np.uint32).astype(np.float64)

    # the benchmark's inputs, generated again on the device with its seeds
    cv, L = ab.params.CURVES[0], _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    n, n_ntt = 1 << log_msm, 1 << log_ntt
    d_bases = torch.empty((n, 12), dtype=torch.int64, device="cuda")
    d_scal = torch.empty((n, 4), dtype=torch.int64, device="cuda")
    d_x = torch.empty((n_ntt, 4), dtype=torch.int64, device="cuda")
    _lib.check(L.b200_gen_bases_dev(cv.cid, seed, n, d_bases.data_ptr(), None, st))
    _lib.check(L.b200_gen_scalars_dev(cv.ntt_field_id, seed + 7777, n, d_scal.data_ptr(), st))
    _lib.check(L.b200_gen_scalars_dev(cv.ntt_field_id, seed + 99, n_ntt, d_x.data_ptr(), st))
    want_msm = C.msm_affine(0, d_bases.cpu().numpy().view(np.uint64), d_scal.cpu().numpy().view(np.uint64), threads=4)
    assert want_msm.any() and np.array_equal(got["msm_affine"], halves(want_msm))
    x0 = d_x.cpu().numpy().view(np.uint64)
    rows = np.sort(np.random.default_rng(seed).choice(n_ntt, size=1 << 16, replace=False))
    y = x0
    for _ in range(warmup + steps):
        y = C.fft(1, y, threads=4)
    assert np.array_equal(got["ntt_fft"], halves(y[rows]))
    assert np.array_equal(got["ntt_ifft"], halves(x0[rows]))
