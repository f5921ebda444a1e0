#!/usr/bin/env python
"""bench.py -- Groth16 withdraw proofs per second on B200 (BASELINE.json metric, config 4).

A "step" is one pass of the hot path over one batch of 1024 synthetic depth-32 withdraw witnesses:
MiMC7 Merkle-path witness generation -> A.w/B.w -> 6 NTTs -> 3 fixed-base MSMs -> 256-byte proofs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`value`   : whole-job proofs/s with the secret inputs already resident in HBM (og_*_dev entry points),
            timed with CUDA events on the library's stream, max over ranks.
`e2e`     : the same through the host-buffer C-ABI call og_groth16_prove_withdraw with pinned host
            memory, H2D of the inputs and D2H of the proofs inside the timed region.
`roofline`: the dominant kernel (k_bucket_acc_g1), algorithmic bytes = 96 B per (point, scalar) pair
            (SURVEY.md 8d) / its CUDA-event duration measured in the timed region, against the measured
            HBM peak; `imad` next to it is the bound that actually binds (integer multiply-add pipe).
`cpu_baseline`: the oracle's C port (this repo's own CPU prover -- the reference ships none) on the
            box's host cores, on a bounded sample.  --impl reference times that same CPU prover as the
            reference arm.
Multi-GPU: proofs are independent -> one process per GPU, each proving its own batch (weak scaling),
no data-path collective; NCCL is used only for the barrier and the max-over-ranks reduction.

--dump-outputs DIR: after the timed steps, the proofs and public inputs of the last timed step (rank 0) go to
DIR/proofs.npy and DIR/public_inputs.npy, one row per proof, byte values as float32.  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEPTH = 32
BATCH = 1024
METRIC = "groth16_withdraw_proofs_per_sec"
UNIT = "proofs/s"
TOXIC_SEED = 20260922
INPUT_SEED = 4096               # + rank: the secret inputs of the timed batch
DUMP_BYTES = 64 << 20           # cap on what --dump-outputs writes


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def synth_inputs(rng, batch, depth):
    """Seeded synthetic secret inputs (BASELINE config 4): uniform Fr nullifier/secret/siblings,
    160-bit recipient, uniform path bits; injected (r, s) per proof."""
    from owshen_b200.api import FR_MODULUS as R

    def frs(n):
        return b"".join(rng.randrange(R).to_bytes(32, "little") for _ in range(n))
    nul, sec = frs(batch), frs(batch)
    rec = b"".join(rng.randrange(1 << 160).to_bytes(32, "little") for _ in range(batch))
    sib = frs(batch * depth)
    bits = [rng.randrange(1 << depth) for _ in range(batch)]
    rs = frs(2 * batch)
    return nul, sec, rec, sib, bits, rs


def toxic(rng):
    from owshen_b200.api import FR_MODULUS as R
    return [rng.randrange(1, R) for _ in range(5)]


def parse_pk_blob(pk: bytes, n_vars, n_pub, log_m):
    """Split the product's OGPK blob into the byte arrays the oracle's C prover takes."""
    o = 8 + 20
    out = {}
    for name, size in (("alpha1", 64), ("beta1", 64), ("beta2", 128), ("delta1", 64), ("delta2", 128),
                       ("a", 64 * n_vars), ("b1", 64 * n_vars), ("b2", 128 * n_vars),
                       ("l", 64 * (n_vars - n_pub - 1)), ("h", 64 << log_m)):
        out[name] = pk[o:o + size]; o += size
    out["log_m"] = log_m
    return out


def dump_outputs(out_dir, proofs: bytes, pub: bytes, n: int):
    """--dump-outputs: n proofs (256 B) and their public inputs (96 B) as float32 arrays of byte values (exact);
    a batch too large for DUMP_BYTES is written as a fixed, seeded sample of rows."""
    import numpy as np
    rows = np.arange(n)
    cap = DUMP_BYTES // (4 * (256 + 96))
    if n > cap:
        rows = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, b, w in (("proofs", proofs, 256), ("public_inputs", pub, 96)):
        a = np.frombuffer(b, dtype=np.uint8).reshape(n, w)[rows].astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def physical_cores():
    """Host threads the CPU prover should use: physical cores (SMT siblings slow this integer-bound code down:
    6.4 proofs/s on 128 threads vs 8.8 on 64 on the round-1 box)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:
        pass
    try:      # a cgroup CPU quota caps what the threads can get whatever the affinity mask says (round 2: 16 of 128 on the bench box)
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.999)))
    except Exception:
        pass
    return n


def host_cpu_info():
    """What the CPU arm can actually use on this box, so that ratios compare across boxes: affinity mask, cgroup
    quota, SMT layout, load before the run (round 1 saw 8.6 vs 34 proofs/s on two boxes that both said "64 cores")."""
    info = {"affinity": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None, "os_cpu_count": os.cpu_count()}
    try:
        import psutil
        info["physical"] = psutil.cpu_count(logical=False)
        info["logical"] = psutil.cpu_count(logical=True)
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        info["cgroup_cpu_max"] = None if q == "max" else float(q) / float(per)
    except Exception:
        info["cgroup_cpu_max"] = "unreadable"
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["model"] = line.split(":", 1)[1].strip(); break
    except Exception:
        pass
    return info


def cpu_single_thread_seconds(pr, rng):
    """Seconds for ONE proof on ONE host thread (box-independent yardstick next to the all-cores rate)."""
    from oracle import cport
    cport.lib().oc_set_num_threads(1)
    nul, sec, rec, sib, bits, rs = synth_inputs(rng, 1, DEPTH)
    wit = cport.withdraw_witness(nul, sec, rec, sib, bits, DEPTH)
    t = time.perf_counter()
    pr.prove_batch(wit, rs)
    return time.perf_counter() - t


def cpu_prover_rate(pkb, n_proofs, rng, threads=None):
    """proofs/s of the oracle's C prover on `n_proofs` synthetic witnesses, one proof per host thread."""
    from oracle import cport
    from oracle import withdraw_circuit as wc
    cs = wc.build_r1cs(DEPTH)
    if threads:
        cport.lib().oc_set_num_threads(threads)
    cores = cport.lib().oc_num_threads()
    nul, sec, rec, sib, bits, rs = synth_inputs(rng, n_proofs, DEPTH)
    wit = cport.withdraw_witness(nul, sec, rec, sib, bits, DEPTH)
    pr = cport.Prover(cs, pkb)
    t = time.perf_counter()
    pr.prove_batch(wit, rs)
    dt = time.perf_counter() - t
    one = cpu_single_thread_seconds(pr, random.Random(11))
    return n_proofs / dt, cores, dt, one


def synth_scalars_dev(torch, seed, lo, hi, dev):
    """Scalars [lo, hi) of a seeded 253-bit sequence as a device uint8 tensor (32 B each, always canonical);
    reproducible per block of 2^16, so any rank can regenerate any range."""
    blk, parts = 1 << 16, []
    for b0 in range(lo - lo % blk, hi, blk):
        g = torch.Generator(device=dev)
        g.manual_seed(seed * 1000003 + b0 // blk)
        raw = torch.randint(0, 256, (blk, 32), dtype=torch.uint8, device=dev, generator=g)
        raw[:, 31] &= 0x1F
        a, b = max(lo, b0) - b0, min(hi, b0 + blk) - b0
        parts.append(raw[a:b].reshape(-1))
    return torch.cat(parts) if parts else torch.empty(0, dtype=torch.uint8, device=dev)


def sharded_msm_leg(torch, dist, ob, api, ctx, dev, rank, world, log_n, steps=3, warmup=1):
    """BASELINE config 5 through the product function owshen_b200.sharded.msm_sharded_dev: one G1 + one G2 MSM of
    2^log_n points (shared scalars) sharded by point range over the ranks, partial sums all-gathered over NCCL on
    the library's stream, CUDA-event timed on that stream, max over ranks.  Rank 0 then recomputes the whole MSM on
    its GPU alone: `matches_single_gpu` and the strong-scaling ratio come from that."""
    from owshen_b200.sharded import msm_sharded_dev, shard_range
    L = api.lib()
    n = 1 << log_n

    def inputs(lo, hi):
        m = hi - lo
        ks = synth_scalars_dev(torch, 5, lo, hi, dev)
        sc = synth_scalars_dev(torch, 55, lo, hi, dev)
        p1 = torch.empty(64 * m, dtype=torch.uint8, device=dev)
        p2 = torch.empty(128 * m, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        api._check(L.og_g1_generator_mul_dev(ctx._h, ks.data_ptr(), m, p1.data_ptr()), ctx)
        api._check(L.og_g2_generator_mul_dev(ctx._h, ks.data_ptr(), m, p2.data_ptr()), ctx)
        ctx.sync()
        return p1, p2, sc

    lo, hi = shard_range(n, rank, world)
    p1, p2, sc = inputs(lo, hi)
    out1 = torch.empty(64, dtype=torch.uint8, device=dev)
    out2 = torch.empty(128, dtype=torch.uint8, device=dev)

    def one():
        msm_sharded_dev(ctx, p1, sc, "g1", out=out1)
        msm_sharded_dev(ctx, p2, sc, "g2", out=out2)
    for _ in range(warmup):
        one()
    ctx.sync(); torch.cuda.synchronize()
    if dist:
        dist.barrier()
    ctx.timer_start()
    for _ in range(steps):
        one()
    ms = ctx.timer_stop() / steps
    tt = torch.tensor([ms], dtype=torch.float64, device=dev)
    mine = torch.cat([out1, out2]).clone()
    agree = torch.ones(1, dtype=torch.int32, device=dev)
    if dist:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ref = mine.clone(); dist.broadcast(ref, 0)
        agree = torch.tensor([int(torch.equal(mine, ref))], dtype=torch.int32, device=dev)
        dist.all_reduce(agree, op=dist.ReduceOp.MIN)
    ms = float(tt.item())
    single_ms, matches = None, None
    if rank == 0:
        if world > 1:
            del p1, p2, sc
            p1, p2, sc = inputs(0, n)
        s1 = torch.empty(64, dtype=torch.uint8, device=dev)
        s2 = torch.empty(128, dtype=torch.uint8, device=dev)

        def alone():
            api._check(L.og_msm_g1_dev(ctx._h, p1.data_ptr(), sc.data_ptr(), n, s1.data_ptr()), ctx)
            api._check(L.og_msm_g2_dev(ctx._h, p2.data_ptr(), sc.data_ptr(), n, s2.data_ptr()), ctx)
        alone(); ctx.sync()
        ctx.timer_start()
        for _ in range(steps):
            alone()
        single_ms = ctx.timer_stop() / steps
        matches = bool(torch.equal(torch.cat([s1, s2]), mine))
    if dist:
        dist.barrier()
    alg = (64 + 128 + 32) * n
    return {"workload": f"2^{log_n}-point G1 + G2 MSM, shared scalars, point-range sharded over {world} rank(s) (BASELINE config 5 shape; "
                        f"2^24 needs the 8-GPU box, see scripts/bench_sharded_msm.py)",
            "log_n": log_n, "n_gpus": world, "ms": ms, "points_per_s": n / (ms * 1e-3), "algorithmic_bytes": alg,
            "hbm_gbs_aggregate": alg / (ms * 1e-3) / 1e9, "exchange_bytes_per_rank": 192, "ranks_agree": bool(agree.item()),
            "matches_single_gpu": matches, "single_gpu_ms": single_ms,
            "strong_scaling_vs_n1": (single_ms / ms) if single_ms else None,
            "timing": "CUDA events on the library stream around MSM + NCCL all-gather (on that stream, no host hop) + final sum; max over ranks",
            "steps": steps, "warmup": warmup}


def run_reference(args):
    """Reference arm: the CPU prover on the host cores (the reference itself has no prover; this is the
    repo's own oracle port, kind = "port").  Each step proves one bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import cport
    from oracle import withdraw_circuit as wc
    rng = random.Random(TOXIC_SEED)
    cs = wc.build_r1cs(DEPTH)
    pkb, _ = cport.setup_bytes(cs, *toxic(rng))
    cport.lib().oc_set_num_threads(physical_cores())
    cores = cport.lib().oc_num_threads()
    sample = max(cores, 8)
    nul, sec, rec, sib, bits, rs = synth_inputs(random.Random(1), sample, DEPTH)
    wit = cport.withdraw_witness(nul, sec, rec, sib, bits, DEPTH)
    pr = cport.Prover(cs, pkb)
    host = host_cpu_info()
    for _ in range(args.warmup):
        pr.prove_batch(wit, rs)
    t = time.perf_counter()
    for _ in range(args.steps):
        proofs = pr.prove_batch(wit, rs)
    dt = time.perf_counter() - t
    if args.dump_outputs:
        nv = cs.n_vars
        dump_outputs(args.dump_outputs, proofs, b"".join(wit[32 * nv * i + 32:32 * nv * i + 128] for i in range(sample)), sample)
    value = sample * args.steps / dt
    one = cpu_single_thread_seconds(pr, random.Random(11))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u256 (4x64-bit Montgomery limbs)", "data": "synthetic",
        "config": {"workload": f"groth16 withdraw prove, depth-{DEPTH} MiMC7 Merkle, {sample} proofs per step on the CPU "
                               f"(bounded sample of the {BATCH}-proof batch: the full batch would take ~{BATCH * one / max(cores, 1):.0f} s "
                               f"per step on this host, x {args.steps + args.warmup} steps; proofs are independent, so the rate does not depend on the batch)",
                   "circuit_constraints": cs.n_constraints},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} proofs per step, one proof per OpenMP thread; own CPU prover -- the reference ships none",
                         "single_thread_s_per_proof": one, "parallel_efficiency": value * one / max(cores, 1), "host": host},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=BATCH, help=argparse.SUPPRESS)
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-parity", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sharded-log-n", type=int, default=22, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's proofs and public inputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import owshen_b200 as ob
    from owshen_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    batch = args.batch

    ctx = ob.Context(local_rank)
    rng = random.Random(TOXIC_SEED)
    pk_bytes, vk_bytes = ob.setup_withdraw(ctx, DEPTH, *toxic(rng))
    PK = ob.ProvingKey(ctx, pk_bytes)
    nul, sec, rec, sib, bits, rs = synth_inputs(random.Random(INPUT_SEED + rank), batch, DEPTH)

    def dev_u8(b):
        return torch.frombuffer(bytearray(b), dtype=torch.uint8).to(dev)
    d_nul, d_sec, d_rec, d_sib, d_rs = (dev_u8(x) for x in (nul, sec, rec, sib, rs))
    d_bits = torch.tensor([b if b < 2**31 else b - 2**32 for b in bits], dtype=torch.int32, device=dev)
    d_proofs = torch.empty(256 * batch, dtype=torch.uint8, device=dev)
    d_pub = torch.empty(96 * batch, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    L = api.lib()

    def step_dev():
        rc = L.og_groth16_prove_withdraw_dev(ctx._h, PK._h, d_nul.data_ptr(), d_sec.data_ptr(), d_rec.data_ptr(), d_sib.data_ptr(),
                                             d_bits.data_ptr(), batch, d_rs.data_ptr(), d_proofs.data_ptr(), d_pub.data_ptr())
        if rc != 0:
            raise ob.OwshenB200Error(rc, L.og_last_error(ctx._h).decode())

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    ctx.profile(True)
    ctx.timer_start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_dev()
    dev_ms = ctx.timer_stop()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    ctx.profile(False)
    prof = ctx.profile_dump()
    launches = ctx.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None

    # parity of what was timed: 16 proofs spread over the batch verify against their own public inputs (host pairing);
    # below (rank 0), four of them are compared byte for byte with the oracle's C prover
    proofs_host = bytes(d_proofs.cpu().numpy().tobytes())
    pub_host = bytes(d_pub.cpu().numpy().tobytes())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, proofs_host, pub_host, batch)
    vidx = sorted({(i * batch) // 16 for i in range(16)} | {batch - 1})
    n_verified = sum(bool(ob.verify(vk_bytes, pub_host[96 * i:96 * i + 96], proofs_host[256 * i:256 * i + 256])) for i in vidx)
    verified = n_verified == len(vidx)

    # e2e: host buffers (pinned) through the public host-pointer call
    def pinned(b):
        t = torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()
        return t
    h_in = [pinned(x) for x in (nul, sec, rec, sib)]
    h_bits = torch.tensor([b if b < 2**31 else b - 2**32 for b in bits], dtype=torch.int32).pin_memory()
    h_rs = pinned(rs)
    h_proofs = torch.empty(256 * batch, dtype=torch.uint8).pin_memory()
    h_pub = torch.empty(96 * batch, dtype=torch.uint8).pin_memory()

    def step_e2e():
        rc = L.og_groth16_prove_withdraw(ctx._h, PK._h, h_in[0].data_ptr(), h_in[1].data_ptr(), h_in[2].data_ptr(), h_in[3].data_ptr(),
                                         h_bits.data_ptr(), batch, h_rs.data_ptr(), h_proofs.data_ptr(), h_pub.data_ptr())
        if rc != 0:
            raise ob.OwshenB200Error(rc, L.og_last_error(ctx._h).decode())
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    e2e_match = bytes(h_proofs.numpy().tobytes()) == proofs_host
    h2d = len(nul) + len(sec) + len(rec) + len(sib) + 4 * batch + len(rs)
    d2h = 256 * batch + 96 * batch

    sharded = None
    if args.sharded_log_n > 0:
        try:
            sharded = sharded_msm_leg(torch, dist, ob, api, ctx, dev, rank, world, args.sharded_log_n, steps=args.steps)
        except Exception as e:      # an extra leg: its failure must not hide the headline
            sharded = {"error": f"{type(e).__name__}: {e}"}

    # max over ranks
    times = torch.tensor([dev_ms, wall_ms, e2e_ms], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms, e2e_ms = (float(x) for x in times.cpu())

    if rank == 0:
        hbm_peak, peak_kind = measured_peaks()
        info = api.r1cs_info(DEPTH)
        # dominant kernel and its roofline numbers
        top = sorted(prof.items(), key=lambda kv: -kv[1][1])
        total_prof_ms = sum(v[1] for v in prof.values())
        kname = "k_bucket_acc_g1"
        kn, kms = prof.get(kname, (0, 0.0))
        m = 1 << info["log_m"]
        # points per proof handled by the two G1 bucket launches of a chunk (A-MSM and C'-MSM); 96 B per pair
        # C' has n_priv + |supp B| + m + 1 points; |supp B| is ~ n_vars/2 for this circuit (exact value in DESIGN.md)
        n_supp = len(set(api.r1cs_export(DEPTH, "B")[1]))
        pairs_per_proof_g1 = (info["n_vars"] + 2) + ((info["n_vars"] - info["n_pub"] - 1) + n_supp + m + 1)
        alg_bytes_per_launch = 96.0 * pairs_per_proof_g1 * batch * args.steps / max(kn, 1)
        avg_ms = kms / max(kn, 1)
        achieved = alg_bytes_per_launch / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get(kname)
        except Exception:
            pass
        pipes = ctx.int_pipe_peaks()
        def cbits(name, dflt):      # mirrors groth16.cu: pk_load (defaults 15 / 15 / 16 bits for A / B / C')
            return int(os.environ.get(name) or os.environ.get("OG_WINDOW_BITS") or dflt)
        win = lambda c: (255 + c - 1) // c
        n_priv = info["n_vars"] - info["n_pub"] - 1
        madds_per_proof_g1 = (info["n_vars"] + 2) * win(cbits("OG_C_A", 15)) + (n_priv + n_supp + m + 1) * win(cbits("OG_C_C", 16))
        # 10 field multiplications per G1 mixed add, 128 32x32->64 multiply-adds per multiplication
        wide_mads = madds_per_proof_g1 * batch * args.steps * 10 * 128
        wide_rate = wide_mads / (kms * 1e-3) if kms > 0 else 0.0
        # arithmetic floor of the whole step: 32x32->64 multiply-adds of every arithmetic kernel by static count
        # (G1 mixed add 8M+2S = 1280, G2 8 x 320 + 2 x 246 = 3052, XYZZ+XYZZ add 14M = 1792 / 4332 at 2.29 additions per bucket,
        # NTT (m/2 log m - 0.75 m) x 128 per transform, 6 transforms per proof) against the carry-chain peak measured in this run
        nb_of = lambda c: 1 << (c - 1)
        cA, cB, cC = cbits("OG_C_A", 15), cbits("OG_C_B", 15), cbits("OG_C_C", 16)
        log_m = info["log_m"]
        per_proof = (madds_per_proof_g1 * 1280 + (n_supp + 2) * win(cB) * 3052
                     + (nb_of(cA) + nb_of(cC)) * 2.29 * 1792 + nb_of(cB) * 2.29 * 4332
                     + 6 * (m / 2 * log_m - 0.75 * m) * 128)
        step_mads = per_proof * batch
        parity = None
        if not args.no_parity:
            try:      # the oracle is the checker here, never the thing measured
                from oracle import cport
                from oracle import withdraw_circuit as wc
                prng = random.Random(99)
                pidx = [0, batch - 1] + (sorted(prng.sample(range(1, batch - 1), 2)) if batch > 3 else [])
                sel = lambda b, w: b"".join(b[w * i:w * i + w] for i in pidx)
                cs = wc.build_r1cs(DEPTH)
                pkb = parse_pk_blob(pk_bytes, info["n_vars"], info["n_pub"], info["log_m"])
                wit = cport.withdraw_witness(sel(nul, 32), sel(sec, 32), sel(rec, 32), sel(sib, 32 * DEPTH), [bits[i] for i in pidx], DEPTH)
                cport.lib().oc_set_num_threads(min(len(pidx), physical_cores()))
                exp = cport.Prover(cs, pkb).prove_batch(wit, sel(rs, 64))
                equal = [proofs_host[256 * i:256 * i + 256] == exp[256 * k:256 * k + 256] for k, i in enumerate(pidx)]
                parity = {"proofs_compared_with_oracle": pidx, "bit_exact": all(equal), "verified": f"{n_verified}/{len(vidx)}"}
            except Exception as e:
                parity = {"error": str(e)}
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # the CPU baseline is reported at N = 1 only
            try:
                from oracle import cport
                pkb = parse_pk_blob(pk_bytes, info["n_vars"], info["n_pub"], info["log_m"])
                cport.lib().oc_set_num_threads(physical_cores())
                cores = cport.lib().oc_num_threads()
                n_cpu = max(2 * cores, 16) if cores <= 64 else cores
                host = host_cpu_info()
                rate, cores, dt, one = cpu_prover_rate(pkb, n_cpu, random.Random(7))
                cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                       "sample": f"{n_cpu} proofs of the same workload, one per OpenMP thread, {dt:.1f} s wall; own CPU prover (oracle/cpu) -- the reference ships none",
                       "single_thread_s_per_proof": one, "parallel_efficiency": rate * one / max(cores, 1), "host": host}
            except Exception as e:  # the oracle is a checker; its absence must not hide the GPU number
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
        value = world * batch * args.steps / (dev_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u256 (8x32-bit Montgomery limbs, integer)", "data": "synthetic",
            "config": {"workload": f"groth16 withdraw prove, batch {batch} per GPU, depth-{DEPTH} MiMC7 Merkle witnesses (BASELINE config 4)",
                       "circuit_constraints": info["n_constraints"], "circuit_variables": info["n_vars"], "domain": m,
                       "parallelism": f"replicas x{world} (independent proofs, no data-path collective)",
                       "l2": "per-step working set (sorted digit lists + window tables, > 2 GB) exceeds the 126 MB L2; no flush needed",
                       "timing": "CUDA events on the library stream, max over ranks", "wall_ms_per_step": wall_ms / args.steps,
                       "proofs_verify": bool(verified), "e2e_bytes_equal_device_path": bool(e2e_match), "parity": parity},
            "e2e": {"value": world * batch * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak if hbm_peak else None, "frac_of_nominal_8tbs": achieved / 8000.0,
                         "traffic": traffic, "peak_source": peak_kind,
                         "avg_launch_ms": avg_ms, "launches": kn, "share_of_step": kms / total_prof_ms if total_prof_ms else None,
                         "note": "MSM is bound by the 32-bit integer multiply-add pipe, not HBM (DESIGN.md 5); see `imad`"},
            "imad": {"kernel": kname, "achieved_wide_mad_per_s": wide_rate, "peak_wide_mad_per_s": pipes["imad_wide_carry_chain_per_s"],
                     "frac": wide_rate / pipes["imad_wide_carry_chain_per_s"] if pipes["imad_wide_carry_chain_per_s"] else None,
                     "peak_imad_per_s": pipes["imad_per_s"], "peak_imad_wide_per_s": pipes["imad_wide_per_s"],
                     "note": "the binding roofline: 32x32->64 multiply-adds issued as carry chains (IMAD.WIDE.U32.X), peak measured "
                             "by og_int_pipe_peaks on this GPU in this run; achieved = mixed adds x 10 field muls x 128 products",
                     "step": {"wide_mads_per_step": step_mads,
                              "floor_ms": 1e3 * step_mads / pipes["imad_wide_carry_chain_per_s"] if pipes["imad_wide_carry_chain_per_s"] else None,
                              "frac_of_step": (1e3 * step_mads / pipes["imad_wide_carry_chain_per_s"]) / (dev_ms / args.steps) if pipes["imad_wide_carry_chain_per_s"] else None,
                              "note": "multiply-adds of the bucket accumulations, bucket reductions and NTTs of one step by static count / measured "
                                      "carry-chain peak = the time the step would take if only the multiplier mattered; the sort, the witness chains "
                                      "and the assembly are not arithmetic-bound and are not in the floor"}},
            "kernels": {k: {"launches": v[0], "ms": round(v[1], 3)} for k, v in top[:12]},
            "cpu_baseline": cpu,
            "sharded_msm": sharded,
        }
        print(json.dumps(line))
    PK.close()
    ctx.close()
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
