#!/usr/bin/env python3
"""bench.py -- witnesses/sec for main_proof_of_burn on B200 (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of B synthetic, valid test_pob_input.json-shaped inputs per
GPU for the circuit ProofOfBurn(16,4,16,50,31,2,10^19,10^20) (circuits/main_proof_of_burn.circom:27): every
instance is evaluated and its complete 215,907,954-entry witness vector (6.909 GB) is written to HBM.
  value : whole-job witnesses/s with the packed inputs already resident in HBM (pob_stage_inputs).
  e2e   : the same through the public call with HOST (pinned) input buffers: H2D of every step's inputs and
          D2H of its per-instance status + output signals inside the timed region.
  roofline : expand kernel, algorithmic bytes (32 B x n_signals x instances per launch) / CUDA-event duration.
  handoff  : the same batch with every witness CONSUMED on the GPU (the digest kernel reads all of it before its slot is
          reused) and a sample with every witness EXPORTED to host memory through the consumer-paced path
          (pob_export_batch): nothing is overwritten unread in either mode.  The headline `value` itself is the
          generation-only run (POB_RUN_DISCARD): BASELINE.json's metric counts witnesses written to HBM.
  latency  : one main-shape witness alone on the GPU (BASELINE.json configs[1]), input on the host -> witness in HBM.
  cpu_baseline : the CPU oracle (a restatement of the reference calculator -- "port"), P processes on host cores.
Instances shard by index across ranks with no data-path collective; NCCL is used only for the barrier, the
max-over-ranks time and the final ok-count reduction (weak scaling: B per GPU is fixed).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)
for p in (ROOT, os.path.join(ROOT, "proof-of-burn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

MAIN_SHAPE = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
MAIN_EXPR = "ProofOfBurn(16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)"
N_SIGNALS_MAIN = 215907954
METRIC = "main_proof_of_burn witnesses/sec"


def shape_expr(shape):
    return "ProofOfBurn(%s)" % ", ".join(str(v) for v in shape)


# ---- clocks sampler (B200_PROFILING.md "clocks DURING the timed region") ----------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """summary of the samples taken inside [t0, t1] (the timed region); nvidia-smi needs a second or two to come up on an
        8-GPU box, so the sampler is started before the warm-up and the window is cut out afterwards"""
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        rows = [r for t, r in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.2)]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": sorted(reasons), "samples": len(sm)}


# ---- CPU baseline: the oracle on host cores ------------------------------------------------------------------------
def _oracle_worker(args):
    expr, flat = args
    from oracle import oracle
    t = time.time()
    w = oracle.run_flat(*oracle.parse_main(expr), flat)
    ok, n, dig = w.ok, w.n_signals, w.digest()
    w.free()
    return ok, n, time.time() - t, dig


def cpu_baseline_run(expr, packed, procs, rounds=1):
    """`procs` single-threaded oracle processes on distinct inputs (the reference calculator is single-threaded:
    BASELINE.md section 3); returns witnesses/s over `rounds` rounds."""
    from oracle import oracle
    oracle.build()
    jobs = [(expr, packed[i % len(packed)][:, :].copy()) for i in range(procs)]
    t0 = time.time()
    done, digests = 0, []
    with mp.get_context("fork").Pool(procs) as pool:
        for _ in range(rounds):
            res = pool.map(_oracle_worker, jobs)
            assert all(r[0] for r in res), "oracle rejected a synthetic instance"
            done += len(res); digests = [r[3] for r in res]
    dt = time.time() - t0
    cpu_baseline_run.last_digests = digests        # whole-witness digests of jobs 0..procs-1 (parity check in the B200 arm)
    return done / dt, dt, done


def mem_limited_procs(want, bytes_per_proc):
    """never let the CPU baseline exhaust host RAM: bound the process count by MemAvailable and the cgroup limit"""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v.isdigit():
                avail = min(avail, int(v)) if avail else int(v)
        except Exception:
            pass
    if not avail:
        return min(want, 4)
    return max(1, min(want, int(avail * 0.5 // bytes_per_proc)))


def shared_config(a, expr, world):
    """identical in the B200 arm and the reference arm (the driver compares the two `config` objects)"""
    n_sig = 51277058 + 10289431 * a.layers
    return {"workload": "main_proof_of_burn %s, batch %d synthetic valid test_pob_input.json-shaped inputs per GPU per step (trie depth %d-%d)" % (
                expr.replace(" ", ""), a.batch, min(8, a.layers), min(10, a.layers)),
            "circuit": expr, "n_signals": n_sig, "witness_bytes": 32 * n_sig, "batch_per_gpu": a.batch,
            "parallelism": "instances sharded by index, %d per GPU" % a.batch,
            "l2": "each step writes %.1f GB per GPU, far beyond the 126 MB L2; no flush needed" % (a.batch * 32 * n_sig / 1e9)}


def dump_outputs(out_dir, circuit, res, n_instances=4, n_windows=16, window=4096):
    """Write what one timed step computed, so that two builds can be compared output for output on the same inputs:
    what the step returns (per-instance status and output signals) and a fixed sample of the witnesses it left resident
    in HBM (the last `n_instances` of the batch, the same `n_windows` windows of `window` entries in each, drawn from a
    fixed seed).  Every array is float64; a field element is stored as its 8 32-bit words, least significant first,
    which float64 holds exactly.  Some 17 MB at the defaults."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def words(limbs):
        limbs = np.asarray(limbs, dtype=np.uint64)
        w = np.stack([limbs & np.uint64(0xFFFFFFFF), limbs >> np.uint64(32)], axis=-1)
        return w.reshape(limbs.shape[:-1] + (2 * limbs.shape[-1],)).astype(np.float64)

    n, n_sig = len(res.status), circuit.n_signals
    window = min(window, n_sig)
    firsts = [0, n_sig - window] + sorted(int(v) for v in np.random.default_rng(0).integers(0, n_sig - window + 1, max(0, n_windows - 2)))
    entries = np.concatenate([np.arange(f, f + window) for f in firsts])
    insts = list(range(max(0, n - min(n_instances, circuit.desc["n_slots"])), n))
    sample = np.stack([np.concatenate([circuit.witness(i, f, window) for f in firsts]) for i in insts])
    arrays = {"status": res.status.astype(np.float64), "outputs": words(res.outputs_limbs),
              "witness_sample": words(sample), "witness_sample_entries": entries.astype(np.float64),
              "witness_sample_instances": np.array(insts, dtype=np.float64)}
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def bench_spend(a, rank, local_rank, world):
    """main_spend = Spend(31) (circuits/main_spend.circom:6), 2,603,360 entries = 83.3 MB per witness.  Informational:
    same timing rules as the headline run, single process."""
    import numpy as np
    import torch
    import pob_b200
    assert world == 1, "--circuit spend is a single-GPU informational run"
    torch.cuda.set_device(local_rank)
    rng = np.random.default_rng(a.seed)
    P = pob_b200.P
    insts = []
    for _ in range(a.batch):
        bal = int(rng.integers(1, 1 << 62))
        insts.append({"burnKey": str(int.from_bytes(rng.bytes(31), "big") % P), "balance": str(bal),
                      "withdrawnBalance": str(int(rng.integers(0, bal + 1))), "extraCommitment": int(rng.integers(0, 1 << 62))})
    c = pob_b200.Circuit("Spend(31)", device=local_rank)
    pinned = pob_b200.PinnedArray((a.batch, c.n_inputs, 4), np.uint64)
    pinned.array[...] = c.pack(insts)
    c.stage(pinned.array)
    for _ in range(a.warmup):
        c.run_packed(None, n=a.batch, staged=True, discard=True)
    torch.cuda.synchronize()
    dev_ms = exp_ms = e2e_ms = 0.0
    launches = ok = 0
    for _ in range(a.steps):
        r = c.run_packed(None, n=a.batch, staged=True, discard=True)
        dev_ms += r.timing["total_ms"]; exp_ms += r.timing["expand_ms"]; ok += r.n_ok
        launches += r.timing["expand_launches"] + r.timing["eval_launches"] + r.timing["other_launches"]
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, c, r)
    for _ in range(a.steps):
        r2 = c.run_packed(pinned.array, discard=True)
        e2e_ms += r2.timing["total_ms"]
    assert ok == a.batch * a.steps
    n = a.batch * a.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = 32.0 * c.n_signals * n / (exp_ms / 1e3) / 1e9
    print(json.dumps({"metric": "main_spend witnesses/sec", "value": n / (dev_ms / 1e3), "unit": "witnesses/s", "n_gpus": 1, "steps": a.steps,
                      "warmup": a.warmup, "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "u256 (BN254-Fr integer)", "data": "synthetic",
                      "config": {"workload": "main_spend Spend(31), batch %d synthetic valid inputs" % a.batch, "n_signals": c.n_signals,
                                 "witness_bytes": c.desc["witness_bytes"], "resident_slots": c.desc["n_slots"], "chunk": c.desc["chunk"], "expand_group": c.desc["expand_group"]},
                      "e2e": {"value": n / (e2e_ms / 1e3), "unit": "witnesses/s", "h2d_bytes_per_step": r2.timing["h2d_bytes"], "d2h_bytes_per_step": r2.timing["d2h_bytes"]},
                      "gpu_launches": launches,
                      "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                                   "kernel": "k_expand_round + k_expand_codes", "expand_share_of_step": exp_ms / dev_ms}}))
    c.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1024, help="instances per GPU per step (BASELINE.json configs[2]: 1024)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--layers", type=int, default=16, help="maxNumLayers of the circuit shape (config 5 sweep)")
    ap.add_argument("--circuit", default="pob", choices=["pob", "spend"], help="pob = main_proof_of_burn (the headline metric); spend = main_spend (Spend(31), informational)")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the timed oracle leg (the in-run digest parity check still runs: --parity)")
    ap.add_argument("--parity", type=int, default=2, help="instances whose whole-witness digest is compared with the oracle when the cpu baseline is skipped (0 = none)")
    ap.add_argument("--consume-batch", type=int, default=256, help="instances of the 'every witness consumed on the GPU' figure (0 = skip)")
    ap.add_argument("--no-selfcheck", dest="selfcheck", action="store_false", help="skip the on-GPU constraint check of one witness")
    ap.add_argument("--reduced-batch", type=int, default=256, help="instances of the reduced (--O1-style) witness figure (0 = skip)")
    ap.add_argument("--export-sample", type=int, default=24, help="instances of the 'every witness exported to the host' figure (0 = skip)")
    ap.add_argument("--seed", type=int, default=7503)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(status, output signals and a seeded sample of the resident witnesses; rank 0 only)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has none")
    a.warmup = max(a.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    shape = (a.layers,) + MAIN_SHAPE[1:]
    expr = shape_expr(shape)
    if a.circuit == "spend":
        return bench_spend(a, rank, local_rank, world)

    from pob_b200 import synth
    cores = host_cores()

    # ------------------------------------------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        procs = mem_limited_procs(a.cpu_procs or max(1, min(cores // 2, 32)), 34 * (51277058 + 10289431 * a.layers))
        insts = synth.make_batch(procs, shape, seed=a.seed)
        packed = synth.pack_instances(insts, shape)
        for _ in range(a.warmup):
            cpu_baseline_run(expr, packed, procs)
        v, dt, done = cpu_baseline_run(expr, packed, procs, rounds=a.steps)
        line = {"metric": METRIC, "value": v, "unit": "witnesses/s", "impl": "reference", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u256 (BN254-Fr integer)",
                "data": "synthetic", "config": shared_config(a, expr, world),
                "cpu_baseline": {"value": v, "unit": "witnesses/s", "cores": procs, "kind": "port",
                                 "sample": "each step = %d single-threaded oracle processes x one full %d-entry witness of the workload (a bounded sample of the %d-instance batch; circom is absent: the oracle is a restatement of the reference calculator)" % (procs, 51277058 + 10289431 * a.layers, a.batch)},
                "e2e": {"value": v, "unit": "witnesses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------------------ B200 arm
    import numpy as np
    import torch
    import pob_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU path; use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    # this rank's shard: instances [rank*B, (rank+1)*B) of the global batch (generated by a fork pool, before CUDA is touched)
    from pob_b200 import shard
    insts = synth.make_batch(a.batch, shape, seed=shard.shard_seed(a.seed, rank, a.batch))
    circuit = pob_b200.Circuit(expr, device=local_rank)
    desc = circuit.desc
    pinned = pob_b200.PinnedArray((a.batch, circuit.n_inputs, 4), np.uint64)
    synth.pack_instances(insts, shape, out=pinned.array)
    circuit.stage(pinned.array)

    def step_resident():
        return circuit.run_packed(None, n=a.batch, expand=True, staged=True, discard=True)

    def step_e2e():
        return circuit.run_packed(pinned.array, expand=True, discard=True)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(a.warmup):
        r = step_resident()
    barrier()
    t_wall = time.time()
    dev_ms, exp_ms, exp_launches, launches, ok, eval_ms, eval_launches = 0.0, 0.0, 0, 0, 0, 0.0, 0
    for _ in range(a.steps):
        r = step_resident()
        dev_ms += r.timing["total_ms"]; exp_ms += r.timing["expand_ms"]; exp_launches += r.timing["expand_launches"]
        eval_ms += r.timing["eval_ms"]; eval_launches += r.timing["eval_launches"]
        launches += r.timing["expand_launches"] + r.timing["eval_launches"] + r.timing["other_launches"]
        ok += r.n_ok
    barrier()
    wall_ms = 1e3 * (time.time() - t_wall)
    clocks = sampler.stop(t_wall, time.time())
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, circuit, r)       # before the end-to-end arm reuses the witness slots
    # end-to-end arm (host buffers)
    for _ in range(min(a.warmup, 1)):
        step_e2e()
    barrier()
    e2e_ms, h2d, d2h = 0.0, 0, 0
    for _ in range(a.steps):
        r2 = step_e2e()
        e2e_ms += r2.timing["total_ms"]; h2d, d2h = r2.timing["h2d_bytes"], r2.timing["d2h_bytes"]
    barrier()

    # ---- consumer-paced figures (SURVEY.md 8(f) rank 1): nothing is overwritten unread ------------------------------------
    handoff, latency = {}, None
    if a.consume_batch > 0:
        nb = min(a.batch, a.consume_batch)
        circuit.run_packed(None, n=min(nb, 32), staged=True, digest=True)
        rc = circuit.run_packed(None, n=nb, staged=True, digest=True)      # the digest kernel reads every entry of every witness
        handoff["consumed_on_gpu"] = {"value": nb / (rc.timing["total_ms"] / 1e3), "unit": "witnesses/s", "instances": nb,
                                      "consumer": "k_digest reads all %d entries of each witness before its slot is reused (adds 1 x witness bytes of HBM reads)" % desc["n_signals"]}
    if a.export_sample > 0 and rank == 0:
        ne = min(a.batch, a.export_sample)
        circuit.export_batch(None, n=min(ne, 2), staged=True)
        rx, st = circuit.export_batch(None, n=ne, staged=True)
        handoff["exported_to_host"] = {"value": st["witnesses"] / (st["total_ms"] / 1e3), "unit": "witnesses/s", "instances": int(st["witnesses"]), "d2h_gbs": st["d2h_gbs"],
                                       "sink": "pinned host staging ring over 2 copy streams (pob_export_batch, paths=NULL); PCIe-bound"}
    reduced = None
    if a.reduced_batch > 0 and rank == 0:
        # SURVEY.md 8(f) rank 2: the reduced (`--O1`-style) witness of the same instances (POB_CREATE_O1), informational
        nb = min(a.batch, a.reduced_batch)
        circuit.close()
        cr = pob_b200.Circuit(expr, device=local_rank, opt=1)
        cr.stage(pinned.array[:nb])
        cr.run_packed(None, n=nb, staged=True, discard=True)
        rr = cr.run_packed(None, n=nb, staged=True, discard=True)
        reduced = {"value": nb / (rr.timing["total_ms"] / 1e3), "unit": "witnesses/s", "instances": nb, "n_signals": cr.n_signals, "witness_bytes": 32 * cr.n_signals,
                   "fraction_of_o0": cr.n_signals / desc["n_signals"], "expand_gbs": 32.0 * cr.n_signals * nb / (rr.timing["expand_ms"] / 1e3) / 1e9,
                   "eval_ms_total": rr.timing["eval_ms"], "expand_ms_total": rr.timing["expand_ms"], "ok": int(rr.n_ok),
                   "what": "signals tied by signal=signal / signal=constant constraints dropped (pob_b200.h POB_CREATE_O1); order parity unpinned"}
        cr.close()
        circuit = pob_b200.Circuit(expr, device=local_rank)
        circuit.stage(pinned.array)
    selfcheck = None
    if a.selfcheck and rank == 0:
        # SURVEY.md 8(f) rank 4: every constraint of the circuit evaluated on the GPU against one freshly generated witness
        circuit.run_packed(pinned.array[:1])
        circuit.selfcheck(0)                                    # first call compiles + uploads the constraint system
        sc = circuit.selfcheck(0)
        selfcheck = {"ms": sc["ms"], "n_constraints": sc["n_constraints"], "n_nonlinear": sc["n_nonlinear"], "n_hints": sc["n_hints"], "n_failed": sc["n_failed"] + sc["n_hint_failed"],
                     "signals_read": sc["signals_read"], "what": "pob_selfcheck: every <== / === of the circom sources over witness indices, 100 % of the entries read"}
        assert selfcheck["n_failed"] == 0, "the generated witness violates a circuit constraint"
    if rank == 0:
        one = pinned.array[:1]
        circuit.run_packed(one)
        ms = sorted(circuit.run_packed(one).timing["total_ms"] for _ in range(5))
        tl = circuit.run_packed(one).timing
        latency = {"single_witness_ms": ms[len(ms) // 2], "eval_ms": tl["eval_ms"], "expand_ms": tl["expand_ms"],
                   "what": "one main-shape instance alone on the GPU (BASELINE.json configs[1]): host input -> status + outputs on host, witness complete in HBM"}
    (dev_ms_max, e2e_ms_max, wall_ms_max), (ok_total, launches_total) = shard.reduce_timing_and_counts(
        dist, "cuda", [dev_ms, e2e_ms, wall_ms], [ok, launches])     # time = max over ranks; counts summed over NCCL
    total_instances = world * a.batch * a.steps
    if rank == 0:
        assert ok_total == total_instances, "some synthetic instances were rejected: %d of %d ok" % (ok_total, total_instances)
        value = total_instances / (dev_ms_max / 1e3)
        e2e_value = total_instances / (e2e_ms_max / 1e3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # algorithmic bytes of all expand launches of the timed steps / their summed CUDA-event durations
        bytes_per_launch = 32.0 * desc["n_signals"] * a.batch * a.steps / max(1, exp_launches)
        per_launch_ms = exp_ms / max(1, exp_launches)
        achieved = bytes_per_launch / (per_launch_ms / 1e3) / 1e9
        traffic, traffic_src = None, None
        try:
            # ncu --set full captures of ONE-witness launches of both shipped expand kernels (profiles/), scaled to the
            # witnesses per launch pair timed here
            tj = json.load(open(os.path.join(ROOT, "profiles", "expand_traffic.json")))
            per_wit = tj.get("dram_bytes_per_witness")
            if per_wit and a.layers == 16:
                traffic = per_wit * (a.batch * a.steps / max(1, exp_launches)); traffic_src = tj.get("source")
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": "witnesses/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": dev_ms_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u256 (BN254-Fr integer)", "data": "synthetic",
                "config": shared_config(a, expr, world),
                "details": {"resident_slots": desc["n_slots"], "wall_ms_per_step": wall_ms_max / a.steps, "eval_chunk": desc["chunk"], "expand_group": desc["expand_group"],
                            "eval_kernel": {"ms_per_launch": eval_ms / max(1, eval_launches), "instances_per_launch": min(desc["chunk"], a.batch),
                                            "note": "runs concurrently with the expand kernels on a higher-priority stream"}},
                "handoff": handoff, "latency": latency, "reduced_witness": reduced, "selfcheck": selfcheck,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "witnesses/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "note": "host pinned inputs -> pob_run_batch(POB_RUN_DISCARD) -> status + output signals on host; generation-only: see `handoff` for the runs in which every witness is consumed / exported"},
                "gpu_launches": launches_total,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                             "kernel": "k_expand_round + k_expand_codes (one pair per %d witnesses)" % desc["expand_group"], "bytes_per_launch": bytes_per_launch, "ms_per_launch": per_launch_ms,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                             "expand_share_of_step": exp_ms / dev_ms}}
        k = 0
        if not a.no_cpu_baseline:
            procs = mem_limited_procs(a.cpu_procs or max(1, min(cores // 2, 32)), 34 * desc["n_signals"])
            v, dt, done = cpu_baseline_run(expr, pinned.array[: min(a.batch, procs)], procs)
            line["cpu_baseline"] = {"value": v, "unit": "witnesses/s", "cores": procs, "kind": "port",
                                    "sample": "%d single-threaded oracle processes x 1 witness of the same workload (%.1f s)" % (procs, dt)}
            k = min(a.batch, procs)
        elif a.parity > 0:
            k = min(a.batch, mem_limited_procs(a.parity, 34 * desc["n_signals"]))
            cpu_baseline_run(expr, pinned.array[:k], k)
        if k:
            # the oracle runs above double as an in-run parity check: whole-witness digests of the same instances on the GPU
            rg = circuit.run_packed(pinned.array[:k], digest=True)
            match = [int(rg.digests[i]) == int(cpu_baseline_run.last_digests[i]) for i in range(k)]
            line["parity"] = {"instances": k, "digest_match": all(match), "what": "64-bit digest of all %d witness entries, GPU vs oracle" % desc["n_signals"]}
            assert all(match), "GPU witness digest differs from the oracle"
        print(json.dumps(line))
    circuit.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
