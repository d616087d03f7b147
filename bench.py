#!/usr/bin/env python
"""bench.py -- Groth16 prover throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W             # this back-end
    python bench.py --impl reference --gpus N --steps K ...   # restated bellman CPU path

A "step" is one create_proof of the synthetic 2^20-constraint MiMC-chain R1CS (BASELINE.json
configs[1]; SURVEY.md 8d) from "witness vectors complete" (prover.rs:217) to "192 proof
bytes written": 7 NTTs of 2^20, 6 G1 + 2 G2 MSMs, host finalisation.  `value` has the witness
already resident in HBM; `e2e` goes through the public call with pinned HOST buffers, copies
inside the timed region.  Other workloads (--workload msm | ntt) are the microbenches of
configs[2] and configs[3].

Before the warm-up the MSM form is chosen by measurement on the key about to be timed (DESIGN.md 4.3b): at N = 1 by
bb_groth16_autotune in a child process, at N > 1 by the collective tuner behind per-rank child probes; the timed steps
run the chosen form only and the line records every form's milliseconds under `autotune` (--autotune 0: default form).

--dump-outputs DIR writes what the last timed step returned (prove: the 192 proof bytes; msm: the point; ntt: the same
fixed sample of 2^16 rows of the buffer after the forward transform and after the inverse that restores it) as
DIR/<name>.npy, so that two builds can be compared output for output.

The oracle (oracle/) is used only by the cpu_baseline leg and by --impl reference.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FR_MODULUS = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
METRIC = "groth16_prove_constraints_per_sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="prove", choices=["prove", "msm", "ntt"])
    ap.add_argument("--log-size", type=int, default=None, help="log2 of constraints (prove) / points (msm, ntt)")
    ap.add_argument("--cpu-sample-log", type=int, default=17, help="log2 constraints of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-budget-s", type=float, default=None,
                    help="--impl reference: optional wall-clock bound of the proving loop; when given it overrides --steps / --warmup, "
                         "which shrink to fit it (the line reports what ran)")
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--precompute", type=int, default=None, help="force msm_precompute (0 = per-window bucket sets, 1 = window multiples + one bucket array "
                                                                   "per window, 2 = window multiples + ONE bucket array) instead of measuring")
    ap.add_argument("--autotune", type=int, default=1, help="1 = before the warm-up, time every MSM form on this key (bb_groth16_autotune; sharded: the whole "
                                                            "sharded proof, max over ranks) and run the fastest whose results are byte-identical; at N = 1 the tuner "
                                                            "runs in a child process (a form that faults there cannot take the measurement down with it); "
                                                            "2 = the same in this process; 0 = default form")
    ap.add_argument("--tune-child", action="store_true", help="internal: build the same key and witness, run the tuner, print its report, exit")
    ap.add_argument("--shard-index", type=int, default=0, help="internal (--tune-child): the key shard of the parent rank")
    ap.add_argument("--shard-count", type=int, default=1)
    ap.add_argument("--autotune-reps", type=int, default=3, help="timed proofs per MSM form in the tuner (after one checked proof)")
    ap.add_argument("--acc-variant", type=int, default=0)
    ap.add_argument("--ntt-radix8", type=int, default=0, help="1 = register radix-8 windows (k_ntt_pass8) instead of radix-2 sweeps in shared memory (k_ntt_pass)")
    ap.add_argument("--reduce-2d", type=int, default=1, help="0 = serial running-sum recursion over whole windows instead of row/column sums first")
    ap.add_argument("--affine-tma", type=int, default=0, help="1 = dense halving rounds of G1 jobs staged by cp.async.bulk + mbarrier")
    ap.add_argument("--affine-rounds", type=int, default=-1, help="batched-affine halving rounds per MSM (-1 = by size, 0 = XYZZ accumulation only)")
    ap.add_argument("--affine-batch", type=int, default=0, help="pairs per thread in the batched-affine rounds (0 = default)")
    ap.add_argument("--reduce-k", type=int, default=0)
    ap.add_argument("--reduce-k1", type=int, default=0)
    ap.add_argument("--witness", default="uniform", choices=["uniform", "boolean"],
                    help="boolean: every second aux value is overwritten with 0/1 (SURVEY.md 8d config 2's boolean-heavy variant; "
                         "exercises the Exponent::Zero/One fast paths; no longer a satisfying assignment)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to this back-end's arm only")
    return args


T0 = time.time()
_REAL_STDOUT = None


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def log(msg):
    print(f"[bench +{time.time() - T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE_ROWS = 1 << 16


def dump_outputs(out_dir, arrays):
    """Writes each result as out_dir/<name>.npy: its bytes (proof bytes, little-endian limbs of field elements and
    points) as float32, one value 0..255 per byte, which float32 holds exactly.  The inputs of every workload come
    from fixed seeds, so two builds run with the same arguments must write identical files."""
    os.makedirs(out_dir, exist_ok=True)
    out = {name: np.frombuffer(np.ascontiguousarray(a).tobytes(), np.uint8).reshape(np.shape(a)[:-1] + (-1,)).astype(np.float32)
           for name, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"{total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte dump limit")
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"outputs written to {out_dir}: " + ", ".join(f"{k} {v.shape}" for k, v in out.items()))


def sample_rows(n, k=DUMP_SAMPLE_ROWS):
    """a fixed, seeded choice of min(n, k) row indices of an n-row output, ascending"""
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def measured_traffic():
    """DRAM bytes per (base, scalar) pair of the dominant kernel from the committed ncu capture"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "roofline_r02.json")))
        return float(d["traffic_bytes_per_pair"]), d["source"]
    except Exception:
        return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle): the restated bellman rayon path, all host threads
# ------------------------------------------------------------------------------------------------
def host_cpu_info():
    """What this process may actually use: affinity mask, cgroup CPU quota, and the thread count the
    oracle's pool is sized to (the quota when there is one -- hardware_concurrency() still reports every
    core of the host on a quota'd lease, and a pool larger than the quota only adds contention)."""
    import math
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = None
    quota = None
    try:                                            # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        info["cgroup_cpu_max"] = f"{q} {per}"
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:                                        # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            info["cgroup_cpu_max"] = f"{q} {per}"
            if q > 0:
                quota = q / per
        except Exception:
            info["cgroup_cpu_max"] = None
    info["cgroup_quota_cpus"] = quota
    n = info["affinity"] or info["os_cpu_count"] or 1
    if quota:
        n = max(1, min(n, int(math.ceil(quota))))
    info["threads"] = int(os.environ.get("BB_ORACLE_THREADS", n))
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    return info


def cpu_prove_sample(sample_log, steps=1, warmup=0, budget_s=None):
    """create_proof of the 2^sample_log MiMC chain on the host through the oracle (restated bellman
    multicore path).  With a budget the warm-up, then the step count, shrink so that the whole leg
    stays inside it (projected from the first prove); what actually ran is returned."""
    from oracle import o1
    host = host_cpu_info()
    o1.set_threads(host["threads"])
    cores = o1.num_threads()
    rounds = (1 << (sample_log - 1)) - 1
    mc = o1.Mimc(rounds, seed=7)
    import random
    rng = random.Random(7)
    mc.set_toxic([rng.randrange(1, FR_MODULUS) for _ in range(5)])
    t0 = time.perf_counter()
    mc.generate()
    t_gen = time.perf_counter() - t0
    log(f"oracle CRS for 2^{sample_log} generated in {t_gen:.1f} s ({cores} threads)")
    times, warm_done, t_begin = [], 0, time.perf_counter()
    want_warm, want_steps = warmup, steps
    while warm_done < want_warm or len(times) < want_steps:
        r, s = rng.randrange(FR_MODULUS), rng.randrange(FR_MODULUS)
        t0 = time.perf_counter()
        mc.prove(r, s)
        dt = time.perf_counter() - t0
        if warm_done < want_warm:
            warm_done += 1
        else:
            times.append(dt)
        if budget_s is not None:                    # re-plan from the proves seen so far
            spent = time.perf_counter() - t_begin
            per = spent / (warm_done + len(times))
            left = max(0.0, budget_s - spent)
            room = int(left / per)
            need = (want_warm - warm_done) + (want_steps - len(times))
            if room < need:
                cut = need - room
                w_cut = min(cut, want_warm - warm_done)
                want_warm -= w_cut
                want_steps = max(1, want_steps - (cut - w_cut))
        log(f"oracle prove {warm_done + len(times)}: {dt:.2f} s")
    n = mc.num_constraints
    return dict(n=n, times=times, cores=cores, t_gen=t_gen, warmup=warm_done, host=host, shape=dict(
                    num_aux=mc.num_aux if hasattr(mc, "num_aux") else n - 1),
                sample=f"create_proof of a 2^{sample_log}-constraint MiMC chain, oracle/oracle1 C++ restatement of bellman's "
                       f"multicore path (c = ceil(ln n) windows, one task per window, 8 MSMs in flight, split FFT), {cores} threads")


def run_reference(args):
    """The reference arm: the restated bellman CPU prover (oracle-1; the Rust crate cannot be built in
    this image) on the SAME workload as the GPU arm -- the 2^20-constraint MiMC chain unless
    --log-size says otherwise -- with the same --steps / --warmup, on the host threads this process
    may use.  Only when --ref-budget-s is given does it bound the leg: if K+W proves do not fit inside
    it, the warm-up and then the step count shrink and the line reports what ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    log_n = args.log_size or 20
    res = cpu_prove_sample(log_n, steps=args.steps, warmup=args.warmup, budget_s=args.ref_budget_s)
    total = sum(res["times"])
    nsteps = len(res["times"])
    value = res["n"] * nsteps / total
    m = res["n"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "constraints/s", "n_gpus": args.gpus,
        "steps": nsteps, "warmup": res["warmup"], "ms_per_step": 1e3 * total / nsteps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64 limbs (381-bit Fp / 255-bit Fr Montgomery integers)",
        "data": "synthetic",
        "config": prove_config(log_n, m, m - 1, args.witness, f"host CPU, {res['cores']} threads (rayon-style pool)"),
        "cpu_baseline": {"value": value, "unit": "constraints/s", "cores": res["cores"], "kind": "port", "sample": res["sample"],
                         "host": res["host"], "crs_generation_s": res["t_gen"],
                         "step_seconds": [round(t, 3) for t in res["times"]]},
        "e2e": {"value": value, "unit": "constraints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if nsteps != args.steps or res["warmup"] != args.warmup:
        line["config"]["note"] = (f"asked for --steps {args.steps} --warmup {args.warmup}; the {args.ref_budget_s:.0f} s budget of this leg "
                                  f"allowed {nsteps} + {res['warmup']}")
    emit(line)


def tune_in_child(args, log_n, shard=(0, 1), reps=None):
    """The per-key tuner (bb_groth16_autotune) in a child process that builds the same synthetic key and witness: its
    report names the fastest eligible MSM form, which the parent then selects with bb_crs_apply_tuning.  Whatever happens
    to the child -- a CUDA fault in a form that has never run on this machine included -- the parent's context and its
    measurement are untouched and it stays on the default form."""
    cmd = [sys.executable, os.path.abspath(__file__), "--tune-child", "--log-size", str(log_n), "--witness", args.witness,
           "--autotune-reps", str(reps or args.autotune_reps), "--shard-index", str(shard[0]), "--shard-count", str(shard[1]),
           "--window-bits", str(args.window_bits), "--reduce-k", str(args.reduce_k),
           "--reduce-k1", str(args.reduce_k1), "--reduce-2d", str(args.reduce_2d), "--affine-tma", str(args.affine_tma),
           "--ntt-radix8", str(args.ntt_radix8), "--affine-batch", str(args.affine_batch)]
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        lines = [l for l in res.stdout.splitlines() if l.strip().startswith("{")]
        if res.returncode != 0 or not lines:
            tail = " | ".join((res.stderr or "").strip().splitlines()[-3:])
            return {"chosen": 0, "ms": None, "error": f"rc {res.returncode}: {tail[-400:]}"}
        rep = json.loads(lines[-1])["tune_child"]
        rep["error"] = None
        return rep
    except Exception as e:                               # timeout, unparsable report, ...
        return {"chosen": 0, "ms": None, "error": f"{type(e).__name__}: {e}"[:400]}


def tune_sharded_gated(args, log_n, rank, world, asg, params, r, s, dev):
    """The collective tuner (distributed.autotune_sharded) behind a gate: with --autotune 1 every rank first lets a child
    process tune its own key shard (all forms, on the shapes of the sharded proof's MSMs); only if every rank's child
    survives does the collective tuner run inside the ranks.  Otherwise every rank stays on the default form."""
    from bellman_b200.distributed import _all_reduce, autotune_sharded
    probe_error = None
    if args.autotune == 1:
        probe = tune_in_child(args, log_n, shard=(rank, world), reps=1)
        mine = probe.get("error")
        if _all_reduce(0.0 if mine is None else 1.0, "MAX") > 0.0:
            probe_error = mine or "the tuner child of another rank failed"
    if probe_error is None:
        tuning = autotune_sharded(asg, params, r, s, device_ptrs=dev, reps=args.autotune_reps)
        tuning["error"] = None
        return tuning
    log(f"tuner gate failed, staying on the default form: {probe_error}")
    return {"chosen": 0, "ms": None, "error": probe_error}


def prove_config(log_n, constraints, num_aux, witness, parallelism):
    """`config` of the prove workload: identical keys and values in both arms."""
    half = (constraints // 2) - 1 + 1
    return {"workload": f"groth16-prove-2^{log_n}-mimc-chain" + ("-boolean-heavy" if witness == "boolean" else ""),
            "constraints": constraints, "num_aux": num_aux,
            "msm_sizes": {"h": constraints - 1, "l": num_aux, "a": num_aux + 1, "b_g1": half, "b_g2": half},
            "ntts": "7 x 2^%d" % log_n, "parallelism": parallelism}


# ------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------
def run_prove(args):
    import torch
    import torch.distributed as dist

    import bellman_b200 as bb
    from bellman_b200.distributed import create_proof_sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    shard = (rank, world)
    if args.tune_child:                                  # a parent rank's sandboxed tuner: one process, that rank's GPU and key shard
        shard = (args.shard_index, args.shard_count)
        world, rank = 1, 0
    elif world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local)
    if world > 1:
        backend = os.environ.get("BB_BENCH_DIST_BACKEND", "nccl")         # gloo: the CPU dry run of tests/test_bench_contract.py
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    log_n = args.log_size or 20
    rounds = (1 << (log_n - 1)) - 1
    worker = bb.Worker(local)
    if args.window_bits:
        worker.set_option("msm_window_bits", args.window_bits)
    if args.reduce_k:
        worker.set_option("msm_reduce_k", args.reduce_k)
    if args.reduce_k1:
        worker.set_option("msm_reduce_k1", args.reduce_k1)
    if args.precompute:
        worker.set_option("msm_precompute", args.precompute)
    if args.acc_variant:
        worker.set_option("msm_acc_variant", args.acc_variant)
    worker.set_option("msm_affine_rounds", args.affine_rounds)
    worker.set_option("msm_reduce_2d", args.reduce_2d)
    worker.set_option("msm_affine_tma", args.affine_tma)
    worker.set_option("ntt_radix8", args.ntt_radix8)
    if args.affine_batch:
        worker.set_option("msm_affine_batch", args.affine_batch)
    log("synthesising the MiMC-chain witness (CPU, product-side generator)")
    asg, shape = bb.synth_mimc(rounds, seed=20, pinned=True)
    assert shape["num_constraints"] == 1 << log_n == shape["m"]
    if args.witness == "boolean":
        one = np.array([0x00000001fffffffe, 0x5884b7fa00034802, 0x998c4fefecbc4ff5, 0x1824b159acc5056f], dtype=np.uint64)  # R mod r
        asg.aux_assignment[1::4] = 0
        asg.aux_assignment[3::4] = one
    log("generating the synthetic CRS on the device")
    params = bb.Parameters.synthetic(worker, 21, shape, shard_index=shard[0], shard_count=shard[1])
    log("CRS resident")
    r, s = 0x1234567 % FR_MODULUS, 0x7654321 % FR_MODULUS

    # inputs resident in HBM for the `value` leg
    dev = {}
    keep = []
    for name, arr in (("a", asg.a), ("b", asg.b), ("c", asg.c), ("inputs", asg.input_assignment), ("aux", asg.aux_assignment)):
        t = torch.from_numpy(arr.view(np.int64)).to(f"cuda:{local}")
        keep.append(t)
        dev[name] = t.data_ptr()
    torch.cuda.synchronize()

    # Which MSM form this key runs is measured, not assumed: before any warm-up every form proves this witness on this
    # device (N > 1: the sharded proof, max over ranks), only forms whose results are byte-identical to the default's are
    # eligible, the fastest stays configured.  Outside every timed region; the timed steps run the chosen form only.
    tuning = None
    if args.tune_child:                                  # the sandboxed tuner of a parent bench.py (same key, same witness)
        rep = params.autotune(asg, reps=args.autotune_reps, device_ptrs=dev)
        emit({"tune_child": rep})
        worker.close()
        return
    proof_default = None
    if args.autotune and args.precompute is None and args.affine_rounds < 0:
        log("measuring the MSM forms on this key (autotune)")
        if world == 1 and args.autotune == 1:
            proof_default = bb.create_proof(asg, params, r, s, dev)          # default form, for the byte comparison after the timed legs
            tuning = tune_in_child(args, log_n)
            if tuning.get("error") is None:
                params.apply_tuning(tuning["chosen"])
            else:
                log(f"tuner process failed, staying on the default form: {tuning['error']}")
        elif world == 1:
            tuning = params.autotune(asg, reps=args.autotune_reps, device_ptrs=dev)
        else:
            tuning = tune_sharded_gated(args, log_n, rank, world, asg, params, r, s, dev)
        tuning["forms"] = bb.tuning_names()
        tuning.setdefault("name", tuning["forms"][tuning["chosen"]])
        tuning["where"] = ("child process" if world == 1 else "in the ranks, after every rank's child process survived all forms") if args.autotune == 1 else "in process"
        tuning["note"] = (f"ms per proof and form, fastest of {args.autotune_reps} after one checked proof (negative: -1 tables do not fit, -2 failed, "
                          "-3 results differ: never eligible); measured before the warm-up, outside the timed regions")
        log(f"autotune: {tuning.get('ms')} ms -> form {tuning['chosen']}: {tuning['name']}")

    def step(device_ptrs):
        if world == 1:
            return bb.create_proof(asg, params, r, s, device_ptrs)
        # shards -> one all-gather of partial sums (+ statuses) -> finalize on rank 0
        return create_proof_sharded(asg, params, params, r, s, device_ptrs)

    def sync():
        worker.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(device_ptrs, steps, warmup):
        proof = None
        for _ in range(warmup):
            proof = step(device_ptrs)
        sync()
        worker.profile_reset()
        if world > 1:
            from bellman_b200 import distributed as _dm
            _dm.HOST_MS.clear()
        l0 = worker.kernel_launches
        h0, d0 = worker.bytes_copied()
        t0 = time.perf_counter()
        for _ in range(steps):
            proof = step(device_ptrs)
        sync()
        dt = time.perf_counter() - t0
        if world > 1:
            from bellman_b200.distributed import max_over_ranks
            dt = max_over_ranks(dt)
        h1, d1 = worker.bytes_copied()
        return dt, proof, worker.kernel_launches - l0, (h1 - h0) / steps, (d1 - d0) / steps

    log("timed region: inputs resident in HBM")
    sampler = ClockSampler(local)
    worker.set_option("profile", 1)
    worker.profile_reset()
    sampler.start()
    dt_val, proof_val, launches, _, _ = timed(dev, args.steps, args.warmup)
    clocks = sampler.stop()
    from bellman_b200 import distributed as _dist_mod          # rank 0's host-side phases of the sharded prove (value leg)
    host_ms = {k: round(v / args.steps, 3) for k, v in _dist_mod.HOST_MS.items()} if world > 1 else None
    acc_ms, acc_launches, acc_units = worker.profile_read("msm_accumulate_g1")
    tot_ms, _, _ = worker.profile_read("msm_total_g1")
    acc2_ms, acc2_launches, acc2_units = worker.profile_read("msm_accumulate_g2")
    ent_ms, _, ent_units = worker.profile_read("msm_entries_g1")
    mul_ms, mul_rounds, mul_units = worker.profile_read("msm_fieldmuls_g1")
    mul2_ms, _, mul2_units = worker.profile_read("msm_fieldmuls_g2")
    timeline = read_timeline(worker)
    worker.set_option("profile", 0)
    log(f"value leg done: {1e3 * dt_val / args.steps:.2f} ms/step; timed region: host buffers (e2e)")
    dt_e2e, proof_e2e, _, h2d, d2h = timed(None, args.steps, args.warmup)
    log(f"e2e leg done: {1e3 * dt_e2e / args.steps:.2f} ms/step")
    proof_single = None
    if rank == 0:
        assert proof_val == proof_e2e and len(proof_val) == 192
        assert proof_default is None or proof_default == proof_val, "the tuned MSM form changed the proof bytes"
        if world > 1:
            # the N-GPU proof must be the single-GPU proof: rank 0 proves once more over an unsharded copy of the
            # same synthetic CRS (outside every timed region) and compares the bytes
            log("checking the sharded proof against a single-GPU prove of the same CRS and witness")
            full = bb.Parameters.synthetic(worker, 21, shape, shard_index=0, shard_count=1)
            full.apply_tuning(0)                        # the reference proof of this check comes from the default form
            proof_single = bb.create_proof(asg, full, r, s, dev)
            full.free()
            assert proof_single == proof_val, "sharded proof differs from the single-GPU proof"
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"proof": np.frombuffer(proof_val, np.uint8)})
    n_constraints = shape["num_constraints"]
    value = n_constraints * args.steps / dt_val
    e2e = n_constraints * args.steps / dt_e2e
    hbm_peak, peak_src = peaks()
    # dominant stage: G1 bucket accumulation (the batched-affine halving rounds k_aff_phase1 / k_aff_phase3 plus the
    # XYZZ kernel k_msm_accumulate), timed per job by CUDA events on the job's own stream.  Algorithmic bytes: 128 B
    # per (base, scalar) pair CONSUMED (SURVEY.md 8d) -- counted on the device by k_msm_digits: density-selected,
    # non-zero, in this rank's shard
    alg_bytes = 128.0 * acc_units
    achieved = alg_bytes / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else None
    tr_pair, tr_src = measured_traffic()
    if tr_src and tuning and tuning["chosen"] != 0:
        tr_src += " -- captured for the per-window MSM form; the form this run was tuned to has no ncu capture yet"
    pairs_per_launch = acc_units / acc_launches if acc_launches else 0
    line = {
        "metric": METRIC, "value": value, "unit": "constraints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt_val / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 limbs (381-bit Fp / 255-bit Fr Montgomery integers)", "data": "synthetic",
        "config": dict(prove_config(log_n, n_constraints, shape["num_aux"], args.witness, f"msm-base-range-shards x{world}, NTT replicated"),
                       crs="[k_i]G, pseudorandom k_i, made on device; witness: valid MiMC-chain assignment",
                       msm_form=("per-window bucket sets, no tables (the tuner process failed, see autotune.error)" if tuning and tuning.get("error")
                                 else tuning["name"] + " (measured fastest on this key before the warm-up, see autotune)") if tuning
                       else ("msm_precompute=%s (forced)" % args.precompute if args.precompute is not None else "per-window bucket sets, no tables (not tuned)"),
                       l2="working set (CRS 430 MB + witness 128 MB at 2^20) exceeds the 126 MB L2; no flush needed",
                       timing="host wall clock over K steps bracketed by device synchronize (+barrier), max over ranks; "
                              "kernel figures by CUDA events on the kernels' own streams"),
        "e2e": {"value": e2e, "unit": "constraints/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1e3 * dt_e2e / args.steps},
        "gpu_launches": int(launches),
        "proof_sha256": hashlib.sha256(proof_val).hexdigest() if rank == 0 else None,
        "autotune": tuning,
        "sharded_host_ms_per_step": host_ms,
        "proof_check": (None if rank else ("sharded proof == single-GPU proof of the same CRS/witness/r/s (192 bytes equal, rank 0)"
                                           if world > 1 else "value leg == e2e leg (192 bytes equal); parity with the oracle: tests/")),
        "clocks": clocks,
        "timeline": timeline, "roofline": {"bound": "hbm", "kernel": "G1 bucket accumulation stage: k_aff_phase1/k_aff_phase3<Fp> halving rounds + k_msm_accumulate<Fp>", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": (achieved / hbm_peak) if achieved else None,
                     "traffic": (tr_pair * pairs_per_launch) if tr_pair else None, "traffic_source": tr_src,
                     "algorithmic_bytes_per_launch": 128.0 * pairs_per_launch, "peak_source": peak_src,
                     "launches": int(acc_launches), "avg_launch_ms": acc_ms / acc_launches if acc_launches else None,
                     "algorithmic_bytes_per_pair": 128,
                     "share_of_step": acc_ms / (1e3 * dt_val) if dt_val else None,
                     "share_note": "sum over the G1 jobs of the stage's duration (CUDA events on each job's own stream) over the step time; "
                                   "the jobs overlap each other on different streams, so the sum can exceed the step",
                     "note": "integer-ALU bound, not HBM bound (SURVEY.md 8d): see integer_roofline",
                     "pairs_per_step": acc_units / args.steps, "bucket_entries_per_step": ent_units / args.steps,
                     "integer_roofline": {"bound": "int32 multiplier", "unit": "G Fp-mul/s",
                                          "achieved": (mul_units / (acc_ms * 1e-3) / 1e9) if acc_ms > 0 else None,
                                          "achieved_g2_in_fp_mul": (3.0 * mul2_units / (acc2_ms * 1e-3) / 1e9) if acc2_ms > 0 else None,
                                          "whole_step": ((mul_units + 3.0 * mul2_units) / (dt_val * 1e9)) if dt_val else None,
                                          "peak": 31.2, "peak_source": "profiles/ubench_r01.txt: 288 IMAD.WIDE-class products per Fp-mul at ~30/clk/SM",
                                          "note": "`achieved` is one job's stage rate while ~5 jobs share the machine; `whole_step` = all accumulation-stage "
                                                  "multiplications of the step (G2 counted as 3 Fp each) over the step's wall time; the dominant kernel alone "
                                                  "(k_aff_phase3<Fp>, ncu) runs at 22 G/s = 74 % of the ceiling (profiles/ncu_r02_call3_digest.txt)",
                                          "model": "field multiplications counted from the device's own entry count: 6 per batched-affine "
                                                   "addition (entries/2^(r+1) in halving round r), 10 per XYZZ mixed addition of what is left; "
                                                   "an Fp2 product = 3 Fp products; jobs overlap, so per-job rates share the machine"},
                     "g2_accumulate_ms_per_step": acc2_ms / args.steps, "g1_msm_total_ms_per_step": tot_ms / args.steps},
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("cpu_baseline leg (oracle, all host threads)")
        res = cpu_prove_sample(args.cpu_sample_log, steps=1, warmup=0)
        log("cpu_baseline done")
        cpu_v = res["n"] / res["times"][0]
        line["cpu_baseline"] = {"value": cpu_v, "unit": "constraints/s", "cores": res["cores"], "kind": "port", "sample": res["sample"],
                                "seconds": res["times"][0], "host": res["host"]}
    else:
        line["cpu_baseline"] = None
    if rank == 0:
        emit(line)
    worker.close()
    if world > 1:
        dist.destroy_process_group()


def read_timeline(worker):
    """Per-step averages from the profile counters of the timed `value` leg: for every MSM job of the
    prover the device times (ms since the prove was entered: job queued on its stream, bucket
    accumulation start / end, window sums on the host side of the copy) and the host milestones of
    bb_groth16_prove.  CUDA events on each job's own stream; N=1 path only (the sharded path reports
    the jobs, not the host milestones)."""
    out = {"device_ms_since_prove_start": {}, "host_ms_since_prove_start": {}}
    for job in ("h", "l", "a_inputs", "a_aux", "b_g1_inputs", "b_g1_aux", "b_g2_inputs", "b_g2_aux"):
        marks = []
        for mark in ("start", "acc_start", "acc_end", "end"):
            ms, cnt, _ = worker.profile_read(f"tl.{job}.{mark}")
            marks.append(round(ms / cnt, 3) if cnt else None)
        if any(m is not None for m in marks):
            out["device_ms_since_prove_start"][job] = dict(zip(("queued", "accumulate_start", "accumulate_end", "done"), marks))
    for mark in ("queued", "static_done", "msms_done", "proof_done"):
        ms, cnt, _ = worker.profile_read(f"host.{mark}")
        if cnt:
            out["host_ms_since_prove_start"][mark] = round(ms / cnt, 3)
    return out


def run_msm(args):
    """BASELINE.json configs[2]: G1 MSM microbench (benches/slow.rs shape), 2^24 by default."""
    import bellman_b200 as bb
    import torch
    log_n = args.log_size or 24
    n = 1 << log_n
    worker = bb.Worker(0)
    if args.window_bits:
        worker.set_option("msm_window_bits", args.window_bits)
    worker.set_option("msm_acc_variant", args.acc_variant)
    if args.reduce_k:
        worker.set_option("msm_reduce_k", args.reduce_k)
    if args.precompute:
        worker.set_option("msm_precompute", args.precompute)
    worker.set_option("msm_affine_rounds", args.affine_rounds)
    worker.set_option("msm_reduce_2d", args.reduce_2d)
    worker.set_option("msm_affine_tma", args.affine_tma)
    if args.affine_batch:
        worker.set_option("msm_affine_batch", args.affine_batch)
    log("generating bases and scalars on the device")
    bases = bb.Bases.synthetic(worker, bb.G1, 31, n)
    d_sc = worker.device_alloc(n * 32)
    bb.synth_scalars_device(worker, 32, n, d_sc)
    log("inputs resident")
    tuning = None
    if args.autotune and args.precompute is None and args.affine_rounds < 0:
        # the bases of this microbench are fixed like a key's: measure the per-window form against ONE bucket set over
        # resident window multiples (same point required), keep the faster; outside the timed region
        tuning = {"forms": ["per-window bucket sets, no tables", "one bucket set over resident window multiples"], "ms": []}
        ref = None
        for form in (0, 2):
            try:
                worker.set_option("msm_precompute", form)
                if form:
                    bases.precompute()
                got = bb.multiexp_device(worker, (bases, 0), d_sc, n, bb.FORM_CANONICAL).wait()
                ref = got if ref is None else ref
                if not np.array_equal(np.asarray(got), np.asarray(ref)):
                    tuning["ms"].append(-3.0)
                    continue
                best = None
                for _ in range(2):
                    worker.synchronize()
                    t0 = time.perf_counter()
                    bb.multiexp_device(worker, (bases, 0), d_sc, n, bb.FORM_CANONICAL).wait()
                    dt = time.perf_counter() - t0
                    best = dt if best is None or dt < best else best
                tuning["ms"].append(round(1e3 * best, 3))
            except bb.BackendError:
                if form == 0:
                    raise
                tuning["ms"].append(-1.0)
        chosen = min((i for i in range(2) if tuning["ms"][i] > 0), key=lambda i: tuning["ms"][i])
        tuning["chosen"] = chosen
        if chosen == 0:
            bases.drop_table()
        worker.set_option("msm_precompute", (0, 2)[chosen])
        log(f"autotune: {tuning['ms']} ms -> {tuning['forms'][chosen]}")
    worker.set_option("profile", 1)
    out = None
    sampler = ClockSampler(0)
    sampler.start()                  # before the warm-up: NVML start-up stalls driver calls for ~100 ms
    for _ in range(args.warmup):
        out = bb.multiexp_device(worker, (bases, 0), d_sc, n, bb.FORM_CANONICAL).wait()
    worker.synchronize()
    worker.profile_reset()
    l0 = worker.kernel_launches
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = bb.multiexp_device(worker, (bases, 0), d_sc, n, bb.FORM_CANONICAL).wait()
    worker.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    acc_ms, acc_l, acc_u = worker.profile_read("msm_accumulate_g1")
    tot_ms, _, _ = worker.profile_read("msm_total_g1")
    hbm_peak, peak_src = peaks()
    achieved = 128.0 * n * args.steps / (tot_ms * 1e-3) / 1e9 if tot_ms > 0 else None
    line = {"metric": "g1_msm_mpt_per_sec", "value": n * args.steps / dt / 1e6, "unit": "Mpt/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32 limbs", "data": "synthetic",
            "config": {"workload": f"g1-msm-2^{log_n}", "bases": "[k_i]G distinct, generated in HBM", "scalars": "pseudorandom < 2^254, canonical, resident in HBM",
                       "window_bits": args.window_bits or "auto"},
            "autotune": tuning,
            "gpu_launches": int(worker.kernel_launches - l0), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "whole MSM (all kernels of one job)", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": (achieved / hbm_peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                         "accumulate_ms": acc_ms / args.steps, "device_ms": tot_ms / args.steps, "algorithmic_bytes_per_pair": 128},
            "result_head": bytes(out[0, :2]).hex()}
    # multiexp.rs:334-378's property at full size: the bases are [k_i]G with k = synth stream 31, so the
    # MSM must equal [sum k_i e_i]G -- an Fr inner product on the device and one fixed-base multiplication
    d_k = worker.device_alloc(n * 32)
    bb.synth_scalars_device(worker, 31, n, d_k)
    dot = bb.fr_dot_device(worker, d_k, d_sc, n)
    worker.device_free(d_k)
    want = bb.fixed_base_mul(worker, bb.G1, dot.reshape(1, 4), form=bb.FORM_CANONICAL)
    line["config"]["result_check"] = "msm == [sum k_i e_i]G (device Fr inner product + fixed-base multiplication): " + \
        ("equal" if np.array_equal(np.asarray(out).reshape(-1), np.asarray(want).reshape(-1)) else "MISMATCH")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"msm": np.asarray(out)})
    emit(line)
    assert line["config"]["result_check"].endswith("equal"), "MSM result differs from [sum k_i e_i]G"
    worker.close()


def run_ntt(args):
    """BASELINE.json configs[3]: Fr NTT forward + inverse, 2^24 by default, data resident in HBM."""
    import bellman_b200 as bb
    log_n = args.log_size or 24
    n = 1 << log_n
    worker = bb.Worker(0)
    worker.set_option("ntt_radix8", args.ntt_radix8)
    d = worker.device_alloc(n * 32)
    bb.synth_scalars_device(worker, 41, n, d)
    v = np.zeros((n, 4), np.uint64)
    worker.download(d, v)
    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(args.warmup):
        bb.ntt_device(worker, d, log_n, bb.NTT_FFT)
        bb.ntt_device(worker, d, log_n, bb.NTT_IFFT)
    worker.synchronize()
    l0 = worker.kernel_launches
    t0 = time.perf_counter()
    for _ in range(args.steps):
        bb.ntt_device(worker, d, log_n, bb.NTT_FFT)
        bb.ntt_device(worker, d, log_n, bb.NTT_IFFT)
    worker.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    back = np.zeros_like(v)
    worker.download(d, back)
    ok = bool(np.array_equal(back, v))                      # domain.rs:444-450 round trip, bit exact
    if args.dump_outputs:
        # a step hands back its input (forward, then inverse), so the last step's forward result is computed once more,
        # untimed, from the buffer the step restored: bit for bit the same input whenever the round trip is exact
        rows = sample_rows(n)
        bb.ntt_device(worker, d, log_n, bb.NTT_FFT)
        fwd = np.zeros_like(v)
        worker.download(d, fwd)
        dump_outputs(args.dump_outputs, {"ntt": back[rows], "ntt_forward": fwd[rows]})
    hbm_peak, peak_src = peaks()
    achieved = 2 * 64.0 * n * args.steps / dt / 1e9        # 64 B per point per transform (SURVEY.md 8d)
    line = {"metric": "fr_ntt_mpt_per_sec", "value": 2 * n * args.steps / dt / 1e6, "unit": "Mpt/s (forward+inverse counted as 2n points)",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 limbs", "data": "synthetic",
            "config": {"workload": f"fr-ntt-2^{log_n}-fwd+inv", "round_trip_bit_exact": ok},
            "gpu_launches": int(worker.kernel_launches - l0), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_ntt_pass (all passes)", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_point": 64}}
    emit(line)
    assert ok
    worker.close()


def main():
    args = parse()
    # stdout carries exactly ONE JSON line: everything libraries print (NCCL banner, ...) goes
    # to stderr until the result is ready
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "msm":
        return run_msm(args)
    if args.workload == "ntt":
        return run_ntt(args)
    return run_prove(args)


if __name__ == "__main__":
    main()
