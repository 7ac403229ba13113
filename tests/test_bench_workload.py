"""The bench's synthetic workload is the one BASELINE.json / SURVEY.md section 8(d) name -- FLUX.1-schnell 1024x1024,
dim 3072, 24 heads, mlp 12288, rank 32, 19 joint + 38 single blocks, 4096 image + 256 text tokens -- and its FLOP
bookkeeping matches SURVEY's figure (57 blocks x 113.25 M 4-bit params x 2 x tokens = 56.2 TFLOP per step); its command line
(CPU) and, on the GPU, the outputs it dumps for comparing two builds."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_layer_list_matches_flux_schnell():
    layers = bench.layer_list()
    assert len(layers) == 19 * 2 * 4 + 38 * 4 == 304
    params_per_block = sum(K * N for _, K, N in bench.BLOCK_LINEARS)
    assert params_per_block == 113_246_208                      # 113.25 M 4-bit parameters per block (SURVEY 8d)
    f_main, f_lr = bench.step_flops()
    tokens = bench.IMG_TOKENS + bench.TXT_TOKENS
    assert f_main == 2 * params_per_block * tokens * (19 + 38)
    assert abs(f_main / 1e12 - 56.2) < 0.1                      # SURVEY: 56.2 TFLOP / step
    assert abs(f_main * bench.STEPS_PER_IMAGE / 1e12 - 225) < 1  # 225 TFLOP / image
    assert f_lr < 0.03 * f_main                                 # low-rank branch ~2 % of the FLOPs at r = 32
    shapes = {(M, K, N) for _, M, K, N in layers}
    assert (4096, 3072, 3072) in shapes and (4352, 3072, 12288) in shapes and (256, 12288, 3072) in shapes


def test_gemm_bytes_formula_matches_survey_primary_shape():
    # SURVEY 8(d): (4096, 3072, 3072, r=32) INT4 -> 37.59 MB moved by the GEMM
    assert abs(bench.gemm_bytes(4096, 3072, 3072, 32, fp4=False) / 1e6 - 37.59) < 0.05


def test_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (CPU oracle arm): exactly one JSON line on stdout with the contract's keys."""
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert pr.returncode == 0, pr.stderr[-2000:]
    lines = [l for l in pr.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["metric"].startswith("FLUX.1-schnell") and "workload" in d["config"]


def test_steps_must_be_positive():
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert pr.returncode == 2 and "--steps" in pr.stderr and not pr.stdout.strip()


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """`--dump-outputs DIR`: the hidden states the timed path returned, float32, within 64 MB; `--steps` is the number of timed steps."""
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-secondary", "--no-legs", "--no-full",
                         "--skip-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert pr.returncode == 0, pr.stderr[-2000:]
    lines = [l for l in pr.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    assert [p.name for p in tmp_path.iterdir()] == ["hidden_states.npy"] and (tmp_path / "hidden_states.npy").stat().st_size <= 64 << 20
    y = np.load(tmp_path / "hidden_states.npy")
    assert y.dtype == np.float32 and y.shape == (bench.IMG_TOKENS + bench.TXT_TOKENS, bench.DIM)
    assert np.isfinite(y).all() and y.std() > 0


def test_host_threads_respects_the_cgroup_quota(monkeypatch):
    """The CPU arm's thread count is the affinity mask capped by the cgroup CPU quota (r01: 128 OpenMP threads behind a small quota made the
    same sample 16x slower on one box than on another)."""
    import builtins
    import io

    real_open = builtins.open

    def fake(quota_text):
        def _open(path, *a, **k):
            if path == "/sys/fs/cgroup/cpu.max":
                if quota_text is None:
                    raise OSError("no cgroup v2")
                return io.StringIO(quota_text)
            if str(path).startswith("/sys/fs/cgroup/cpu/"):
                raise OSError("no cgroup v1")
            return real_open(path, *a, **k)
        return _open

    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: set(range(128)), raising=False)
    monkeypatch.setattr(builtins, "open", fake("800000 100000"))
    assert bench.host_threads() == 8
    monkeypatch.setattr(builtins, "open", fake("250000 100000"))
    assert bench.host_threads() == 3          # 2.5 CPUs of quota -> 3 threads
    monkeypatch.setattr(builtins, "open", fake("max 100000"))
    assert bench.host_threads() == 128
    monkeypatch.setattr(builtins, "open", fake(None))
    assert bench.host_threads() == 128
