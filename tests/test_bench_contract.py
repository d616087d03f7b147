"""bench.py's reference arm (`--impl reference`) runs on host cores only, so its side of the
driver contract is checked here without a GPU: one JSON line on stdout with the agreed keys, and
under torchrun rank 0 alone prints while the other ranks exit 0 without work."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_CUDA = {"CUDA_VISIBLE_DEVICES": ""}          # a tuner child of the real library finds no device, GPU or not
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
            "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _check_line(out, n_gpus):
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["n_gpus"] == n_gpus and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"] == "groth16_prove_constraints_per_sec" and d["unit"] == "constraints/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_single_process():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--log-size", "10"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    _check_line(res.stdout, 1)


def test_reference_arm_under_torchrun_world2():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
           "--warmup", "1", "--log-size", "10"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    _check_line(res.stdout, 2)


DRY_RUN = '''
import importlib.util, sys
sys.path.insert(0, ROOT)
import torch
torch.cuda.set_device = lambda *a, **k: None
torch.cuda.synchronize = lambda *a, **k: None
_to = torch.Tensor.to
torch.Tensor.to = lambda self, *a, **k: self if (a and isinstance(a[0], str) and a[0].startswith("cuda")) else _to(self, *a, **k)
torch.Tensor.pin_memory = lambda self, *a, **k: self
import bellman_b200 as bb
bb.LIB_PATH, bb._lib = EMU_LIB, None          # the product sources on host fibers (tests/native)
import os
os.environ["LOCAL_RANK"] = "0"                # the emulation has one device: under torchrun every rank uses it
spec = importlib.util.spec_from_file_location("bench", ROOT + "/bench.py")
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)
sys.argv = ["bench.py", "--log-size", "8", "--steps", "2", "--warmup", "1", "--cpu-sample-log", "8", "--autotune-reps", "1", "--autotune", "2"] + EXTRA
bench.main()
'''


def test_own_arm_dry_run_on_the_emulated_device(tmp_path, emu_lib):
    """bench.py's default workload (prove: value leg, e2e leg, roofline, timeline, cpu_baseline) end
    to end with the CUDA library replaced by the host-fiber build of the same sources and torch.cuda
    stubbed: checks the script and the JSON contract, not the numbers."""
    script = tmp_path / "dry.py"
    dump = tmp_path / "outputs"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--dump-outputs', {str(dump)!r}]\n" + DRY_RUN)
    res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    need = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "timeline"}
    assert need <= set(d), need - set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["gpu_launches"] > 100
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
    assert len(d["timeline"]["device_ms_since_prove_start"]) == 8
    assert d["roofline"]["pairs_per_step"] > 0 and d["roofline"]["bucket_entries_per_step"] > d["roofline"]["pairs_per_step"]
    assert "workload" in d["config"] and "model" not in d["config"]
    at = d["autotune"]                                  # the MSM form was measured before the warm-up; every form eligible here
    assert len(at["ms"]) == len(at["forms"]) >= 2 and all(t > 0 for t in at["ms"]) and at["ms"][at["chosen"]] == min(at["ms"])
    import hashlib
    import numpy as np
    assert sorted(os.listdir(dump)) == ["proof.npy"]      # the last timed step's proof, byte values as float32
    proof = np.load(dump / "proof.npy")
    assert proof.dtype == np.float32 and proof.shape == (192,)
    assert hashlib.sha256(proof.astype(np.uint8).tobytes()).hexdigest() == d["proof_sha256"]


def test_tuner_child_mode_and_parent_fallback(tmp_path, emu_lib):
    """bench.py's sandboxed tuner: (1) child mode (--tune-child) builds the key and witness, tunes and prints its report --
    run here on the emulated device; (2) a parent whose child cannot run (the real library finds no CUDA device: none is
    made visible) records the error and measures the default form."""
    # (the unsharded tuner itself runs in the dry run above; here) the child of rank 1 of 2 -- the gate in front of the
    # collective tuner: that rank's key shard, no process group
    script = tmp_path / "child_shard.py"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--tune-child', '--shard-index', '1', '--shard-count', '2']\n" + DRY_RUN)
    env = dict(os.environ, WORLD_SIZE="2", RANK="1", LOCAL_RANK="0")
    res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert res.returncode == 0, res.stderr[-3000:]
    rep = json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])["tune_child"]
    assert all(t > 0 for t in rep["ms"]) and rep["name"]
    script = tmp_path / "parent.py"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--autotune', '1', '--no-cpu-baseline']\n" + DRY_RUN)
    res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, **NO_CUDA))
    assert res.returncode == 0, res.stderr[-3000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])
    at = d["autotune"]
    assert at["error"] and at["chosen"] == 0 and at["where"] == "child process" and "tuner process failed" in d["config"]["msm_form"]
    assert d["value"] > 0 and d["gpu_launches"] > 100


def test_own_arm_dry_run_two_ranks(tmp_path, emu_lib):
    """bench.py --gpus 2 under torchrun with gloo and the emulated device: the sharded step, the max over ranks, the gate in
    front of the collective tuner (the per-rank tuner children cannot run here -- no CUDA device is made visible -- so both
    ranks must stay on the default form and say why), the sharded proof == single-GPU proof check, one JSON line from rank 0."""
    script = tmp_path / "dry2.py"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--gpus', '2', '--autotune', '1', '--no-cpu-baseline']\n" + DRY_RUN)
    env = dict(os.environ, BB_BENCH_DIST_BACKEND="gloo", **NO_CUDA)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and d["scaling"] == "strong" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert "sharded proof == single-GPU proof" in d["proof_check"] and len(d["proof_sha256"]) == 64
    at = d["autotune"]
    assert at["chosen"] == 0 and at["error"] and "tuner process failed" in d["config"]["msm_form"]
    assert set(d["sharded_host_ms_per_step"]) >= {"queue_witness_msms", "all_gather"}


def test_msm_microbench_dry_run_on_the_emulated_device(tmp_path, emu_lib):
    """bench.py --workload msm (BASELINE configs[2] shape, here 2^10 points): both MSM forms are measured, the result
    is asserted against [sum k_i e_i]G inside the script"""
    script = tmp_path / "dry_msm.py"
    dump = tmp_path / "outputs"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--workload', 'msm', '--log-size', '10', '--dump-outputs', {str(dump)!r}]\n"
                      + DRY_RUN)
    res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.strip()][0])
    assert d["metric"] == "g1_msm_mpt_per_sec" and d["config"]["result_check"].endswith("equal")
    assert len(d["autotune"]["ms"]) == 2 and all(t > 0 for t in d["autotune"]["ms"])
    import numpy as np
    point = np.load(dump / "msm.npy")                     # the G1 point of the last timed step: 12 limbs, 96 bytes
    assert point.dtype == np.float32 and point.shape == (1, 96)
    assert point[0, :16].astype(np.uint8).tobytes().hex() == d["result_head"]


def test_reference_arm_sizes_its_pool_to_the_cpu_quota(monkeypatch):
    """host_cpu_info(): threads = min(affinity, ceil(cgroup quota)) -- the 1-GPU lease of round 1 reported 128
    cores under a 16-CPU quota (cpu.max = "1600000 100000"), and a 128-thread pool ran 3x slower than 16."""
    import builtins
    import importlib.util
    import io
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    real_open = builtins.open

    def fake_open(path, *a, **k):
        if path == "/sys/fs/cgroup/cpu.max":
            return io.StringIO(fake_open.content)
        return real_open(path, *a, **k)

    monkeypatch.setattr(builtins, "open", fake_open)
    monkeypatch.setattr(os, "sched_getaffinity", lambda pid: set(range(128)), raising=False)
    monkeypatch.delenv("BB_ORACLE_THREADS", raising=False)
    fake_open.content = "1600000 100000\n"
    info = bench.host_cpu_info()
    assert info["threads"] == 16 and info["cgroup_quota_cpus"] == 16.0 and info["affinity"] == 128
    fake_open.content = "max 100000\n"
    assert bench.host_cpu_info()["threads"] == 128
    fake_open.content = "250000 100000\n"
    assert bench.host_cpu_info()["threads"] == 3
    monkeypatch.setenv("BB_ORACLE_THREADS", "5")
    assert bench.host_cpu_info()["threads"] == 5


def test_ntt_microbench_dump_on_the_emulated_device(tmp_path, emu_lib):
    """bench.py --workload ntt --dump-outputs: the buffer after the last timed step's forward transform and after its
    inverse (here all 2^10 rows; a fixed sample of 2^16 rows at larger sizes), bytes as float32.  The forward rows must
    be the oracle's transform of the seed-41 input, the restored rows that input."""
    script = tmp_path / "dry_ntt.py"
    dump = tmp_path / "outputs"
    script.write_text(f"ROOT = {ROOT!r}\nEMU_LIB = {emu_lib!r}\nEXTRA = ['--workload', 'ntt', '--log-size', '10', '--dump-outputs', {str(dump)!r}]\n"
                      + DRY_RUN)
    res = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.strip()][0])
    assert d["metric"] == "fr_ntt_mpt_per_sec" and d["steps"] == 2 and d["config"]["round_trip_bit_exact"] is True
    import numpy as np
    import bellman_b200 as bb
    from oracle import o1
    n = 1 << 10
    saved = (bb.LIB_PATH, bb._lib)
    bb.LIB_PATH, bb._lib = emu_lib, None              # bench.py's input: the seed-41 scalars of the device generator
    try:
        w = bb.Worker(0)
        dv = w.device_alloc(n * 32)
        bb.synth_scalars_device(w, 41, n, dv)
        v = np.zeros((n, 4), np.uint64)
        w.download(dv, v)
        w.device_free(dv)
        w.close()
    finally:
        bb.LIB_PATH, bb._lib = saved
    assert sorted(os.listdir(dump)) == ["ntt.npy", "ntt_forward.npy"]

    def limbs(name):
        a = np.load(dump / name)
        assert a.dtype == np.float32 and a.shape == (n, 32) and a.max() <= 255 and np.array_equal(a, np.round(a))
        return a.astype(np.uint8).view(np.uint64)

    assert np.array_equal(limbs("ntt_forward.npy"), o1.fft(v, o1.FFT))
    assert np.array_equal(limbs("ntt.npy"), v)
