#!/usr/bin/env python
"""bench.py - the per-proof MSM + NTT kernel schedule of distributed_plonk on B200.

One "step" = the hot-path work of ONE TurboPlonk proof at n = 2^log_n gates exactly as the
reference's distributed prover issues it (src/dispatcher2.rs:192-713, SURVEY.md §3.4):
    13 x MSM over n+32 bases            (commit_polynomial, dispatcher2.rs:834-893)
     7 x iNTT(n)                        (Prover::fft, is_inv)
    25 x coset-NTT(8n) of n coefficients (Prover::fft, is_quot, is_coset)
     1 x coset-iNTT(8n)                 (dispatcher2.rs:507)
on synthetic data (uniform residues < 2^254, SRS = distinct multiples k_i*G generated on the GPU).
metric = proofs/sec of that schedule ("prover-kernel proofs/sec": the Rust protocol glue around it
- transcript, quotient evaluation, openings - cannot be built in this image, SURVEY.md §8d).

  value : schedule timed with every input already resident in HBM (device pointers in, device
          pointers out), whole job over all N GPUs; N > 1 = strong scaling: the same proof, MSMs
          split by index range (no collective), NTT rows/columns split with ONE NCCL all-to-all.
  e2e   : the same schedule through the reference-facing calls with HOST buffers (pinned):
          dp_msm / dp_fft_init + dp_fft1_rows + exchange + dp_fft2, H2D and D2H inside the timing.
  roofline / cpu_baseline / clocks: see DESIGN.md §Measurement.

`--impl reference` times the CPU restatement of the reference path (oracle/c/ark_oracle.c, the
arkworks algorithms incl. the per-element Fr::pow of worker.rs:79,93,113, all host cores) on a
bounded sample of the same workload and extrapolates to the schedule.  The Rust reference itself
cannot be built here (no cargo/rustc), so kind = "port".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_MSM, N_INTT_N, N_COSET_8N, N_COSET_INTT_8N = 13, 7, 25, 1


def ark_window_c(n: int) -> int:
    """ark-ec 0.3.0 window rule (the shared numerator of BASELINE.md §3)"""
    if n < 32:
        return 3
    return (n - 1).bit_length() * 69 // 100 + 2


def msm_work_adds(n_nonzero: int, n: int) -> float:
    c = ark_window_c(n)
    w = (255 + c - 1) // c
    return float(n_nonzero) * w + 2.0 * ((1 << c) - 1) * w


def butterflies(log_n: int) -> float:
    return (1 << log_n) / 2 * log_n


def schedule_units(log_n: int):
    n, nb = 1 << log_n, (1 << log_n) + 32
    adds = N_MSM * msm_work_adds(n + 2, nb)
    bf = N_INTT_N * butterflies(log_n) + (N_COSET_8N + N_COSET_INTT_8N) * butterflies(log_n + 3)
    return adds, bf


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(sm)[len(sm) // 2:]          # upper half = samples under load
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ CPU arm
CPU_MAX_LOG_MSM, CPU_MAX_LOG_NTT = 22, 25      # largest single samples (about 5 s + 8 s on 64 threads)


def cpu_sample(log_n: int, full: bool = True):
    """The reference's CPU path (oracle restatement, every host thread): ONE MSM(2^log_n + 32) with ark's
    window rule and ONE 2-D coset NTT(2^(log_n+3)) through the worker's four RPC bodies, at FULL size for
    log_n <= 22 (so the schedule time is these two measurements times their counts, 13 and 33.375 - the
    7 iNTT(n) weighted by butterflies - with no extrapolation across sizes); larger log_n time the 2^22 /
    2^25 samples and scale by the shared work units.  The NTT is timed twice: "as written" (two Fr::pow
    per element, worker.rs:79,93,113) and "fair" (incremental twiddles, BASELINE.md section 2)."""
    from oracle import loader as orc
    threads = orc.lib().orc_num_threads()
    log_m = min(log_n, CPU_MAX_LOG_MSM) if full else min(log_n, 14)
    nb = (1 << log_m) + 32
    bases = orc.gen_bases(5, nb, 2048, True)
    sc = orc.gen_fr(6, nb, False)
    t0 = time.perf_counter()
    orc.msm(bases, sc)
    t_msm = time.perf_counter() - t0
    del bases, sc
    adds_rate = msm_work_adds(nb, nb) / t_msm
    log_f = min(log_n + 3, CPU_MAX_LOG_NTT) if full else min(log_n + 3, 17)
    x = orc.gen_fr(7, 1 << log_f)
    t0 = time.perf_counter()
    orc.distributed_fft(x, 1 << log_f, False, True, 1, True)
    t_ntt = time.perf_counter() - t0
    t0 = time.perf_counter()
    orc.distributed_fft(x, 1 << log_f, False, True, 1, False)
    t_ntt_fair = time.perf_counter() - t0
    del x
    adds, bf = schedule_units(log_n)
    exact = full and log_m == log_n and log_f == log_n + 3
    t_proof = adds / adds_rate + bf / (butterflies(log_f) / t_ntt)
    t_proof_fair = adds / adds_rate + bf / (butterflies(log_f) / t_ntt_fair)
    how = ("schedule time = 13 x MSM + (26 + 7 x butterflies(n)/butterflies(8n)) x NTT, both measured at full size" if exact else
           f"samples smaller than the 2^{log_n} schedule: scaled by G1-adds and butterflies")
    return {
        "value": 1.0 / t_proof, "unit": "proofs/s", "cores": int(threads), "kind": "port",
        "sample": (f"1 MSM(2^{log_m}+32, ark window rule) {t_msm:.2f}s + 1 2-D coset NTT(2^{log_f}) {t_ntt:.2f}s as written (per-element pow) / "
                   f"{t_ntt_fair:.2f}s fair (incremental twiddles) on {threads} threads; {how}"),
        "value_fair": 1.0 / t_proof_fair, "msm_g1_adds_per_sec": adds_rate, "ntt_butterflies_per_sec": butterflies(log_f) / t_ntt,
        "ntt_butterflies_per_sec_fair": butterflies(log_f) / t_ntt_fair, "proof_seconds": t_proof, "proof_seconds_fair": t_proof_fair,
        "msm_seconds": t_msm, "ntt_seconds": t_ntt, "ntt_seconds_fair": t_ntt_fair, "sample_is_full_size": exact,
        "sample_seconds": t_msm + t_ntt + t_ntt_fair,
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its children; the CPU arm is meant to use every host core
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    from oracle import loader as orc
    orc.build()
    samples = []
    for _ in range(args.warmup):
        cpu_sample(args.log_n, full=False)
    for _ in range(args.steps):
        samples.append(cpu_sample(args.log_n))
    best = max(samples, key=lambda s: s["value"])
    value = statistics.median(s["value"] for s in samples)
    line = {
        "impl": "reference", "metric": "proofs_per_sec", "value": value, "unit": "proofs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        # one step of THIS metric = one proof's schedule on the CPU: 1000 / value.  The timed sample of a step (one
        # MSM + one NTT, as written and fair) is `sample_ms_per_step`.
        "ms_per_step": 1e3 / value, "sample_ms_per_step": statistics.median(s["sample_seconds"] for s in samples) * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64 limbs (255/381-bit modular integer)",
        "data": "synthetic", "config": workload_config(args.log_n, args.gpus),
        "cpu_baseline": {k: best[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "value_fair_variant": statistics.median(s["value_fair"] for s in samples),
        "msm_g1_adds_per_sec": best["msm_g1_adds_per_sec"], "extrapolated": not best["sample_is_full_size"],
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("each step times ONE full-size MSM and ONE full-size 2-D NTT of the schedule on every host thread and multiplies by "
                 "their counts (the schedule repeats them 13 and ~33.4 times); Rust reference not buildable here, kind = port"),
    }
    line["cpu_baseline"]["value"] = value
    print(json.dumps(line), flush=True)


def workload_config(log_n: int, n_gpus: int):
    return {
        "workload": f"per-proof MSM+NTT schedule of a synthetic 2^{log_n}-gate TurboPlonk circuit: "
                    f"{N_MSM} MSM(2^{log_n}+32) + {N_INTT_N} iNTT(2^{log_n}) + {N_COSET_8N} coset-NTT(2^{log_n + 3}) + "
                    f"{N_COSET_INTT_8N} coset-iNTT(2^{log_n + 3})",
        "log_gates": log_n, "parallelism": f"{n_gpus} GPU(s): MSM index-range shards, 2-D NTT rows/cols + 1 all-to-all",
        "l2": "inputs larger than L2 (>=128 MiB each), rotated between calls",
        "inputs": "coset-NTT(8n) inputs are n coefficients zero-padded to 8n (rows with c/8 non-zero leading entries), declared as such",
    }


# ------------------------------------------------------------------------------------------ GPU arm
GEN_SEED = 0xD15791B07E5EED


def synthetic_k(seed: int, idx: np.ndarray) -> np.ndarray:
    """the 64-bit multipliers k_i of the synthetic SRS (g1_gen_bases_kernel: P_i = k_i * G, SplitMix64 of seed, i)"""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (idx.astype(np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    return z | np.uint64(1)


DUMP_ROWS = 1 << 18       # elements kept per transform output over all ranks: 16 MiB as float64 words


def dump_outputs(out_dir, transforms, commitments, rank=0, world=1):
    """--dump-outputs: what the last timed step handed back, as float64 .npy files two builds can be compared by.
    A field element becomes its eight 32-bit words (exact in float64).  A transform output longer than
    DUMP_ROWS / world is sampled at that many positions drawn from a fixed seed, so the same arguments sample the same
    positions.  The commitments are normalized to affine (x and y as 32-bit words, then the infinity flag): the
    projective form a build returns is one of many for the same point.  With several ranks every rank writes its own
    share (its columns, its partial commitments) as <name>_rank<r>.npy."""
    import torch

    from oracle import loader as orc
    os.makedirs(out_dir, exist_ok=True)
    suffix, rows = ("", DUMP_ROWS) if world == 1 else (f"_rank{rank}", DUMP_ROWS // world)
    for name, t in transforms.items():
        if t.shape[0] > rows:
            idx = np.sort(np.random.default_rng(0xD0).choice(t.shape[0], rows, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), t.cpu().numpy().view(np.uint32).astype(np.float64))
    points = []
    for c in commitments:
        aff = orc.normalize(np.frombuffer(c.cpu().numpy().tobytes(), dtype=np.uint8))
        points.append(np.concatenate([aff[:96].view(np.uint32), aff[96:97]]).astype(np.float64))
    np.save(os.path.join(out_dir, f"commitments{suffix}.npy"), np.stack(points))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=22, dest="log_n")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N > 1: row kernel stores into peer memory over NVLink (fused) or one NCCL all-to-all")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; see dump_outputs)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    import distributed_plonk_b200 as dp
    from distributed_plonk_b200 import dispatcher as disp
    from distributed_plonk_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = world
    lib = dp.load()                       # raises if the CUDA extension is missing: no fallback
    # batched-affine MSM levels: opt in per run, and only if a child process on this GPU found them identical and faster for
    # this rank's shard (distributed_plonk_b200/tune.py); DP_MSM_AFFINE in the environment overrides the probe
    tune_probe = None
    if "DP_MSM_AFFINE" not in os.environ and os.environ.get("DP_BENCH_NO_MSM_PROBE", "0") != "1":
        from distributed_plonk_b200 import tune
        tune_probe = tune.probe(local, rank, W, args.log_n)
        if "error" not in tune_probe:     # (a probe that did not finish decides nothing: dp_init's own tuning, plain vs two levels, stands)
            os.environ["DP_MSM_AFFINE"] = str(tune.choose(tune_probe))
    ctx = dp.Context(lib, local, rank, W)

    log_n = args.log_n
    n, m, nb = 1 << log_n, 1 << (log_n + 3), (1 << log_n) + 32
    log_m = log_n + 3

    # ---- synthetic SRS, generated and kept on the device: n distinct points k_i*G, index 3 = infinity and
    # 32 infinity entries of padding (dispatcher2.rs:207-208, 1097-1104)
    bases_t = torch.empty((nb, 104), dtype=torch.uint8, device="cuda")
    ctx.gen_bases_into(GEN_SEED, nb, bases_t.data_ptr())
    inf = torch.zeros(104, dtype=torch.uint8, device="cuda")      # infinity flag set; x, y are ignored by the import kernel
    inf[96] = 1
    bases_t[3] = inf
    bases_t[n:] = inf
    torch.cuda.synchronize()
    ctx.init_ptr(bases_t.data_ptr(), nb, n, m)
    del bases_t

    gen = torch.Generator(device="cuda")
    gen.manual_seed(0xB200 + 7 * rank)

    def rand_fr(count, g=gen):
        """uniform 254-bit residues: valid canonical scalars and valid Montgomery-form Fr"""
        t = torch.randint(-(1 << 63), (1 << 63) - 1, (count, 4), dtype=torch.int64, device="cuda", generator=g)
        t[:, 3] &= (1 << 62) - 1
        return t

    lo, hi = parallel.msm_shard(nb, rank, W)
    r_n, r_m = 1 << (log_n >> 1), 1 << (log_m >> 1)
    c_n, c_m = n // r_n, m // r_m
    rows_n, cols_n, rows_m, cols_m = r_n // W, c_n // W, r_m // W, c_m // W

    # device-resident inputs (rotated so that consecutive calls never reuse an L2-resident buffer)
    scal = [rand_fr(hi - lo) for _ in range(3)]
    for s in scal:
        s[max(0, n + 2 - lo):] = 0                       # coefficients beyond degree n+1 are the zero padding
    in_n = [rand_fr(rows_n * c_n) for _ in range(2)]
    out_n = torch.empty((cols_n * r_n, 4), dtype=torch.int64, device="cuda")
    # coset-NTT(8n) input = n coefficients zero-padded to 8n, as rows [r][c]: x[b + a*r] != 0 only for a < c/8
    in_m = []
    for _ in range(3):
        t = rand_fr(rows_m * c_m).view(rows_m, c_m, 4)
        t[:, c_m // 8:, :] = 0
        in_m.append(t.view(-1, 4))
    out_m = torch.empty((cols_m * r_m, 4), dtype=torch.int64, device="cuda")
    out_mi = torch.empty_like(out_m)       # the coset-iNTT's own output: the step's last coset-NTT result stays readable
    # what the dispatcher feeds the quotient-domain transforms is n coefficients (dispatcher2.rs:386-388): the row
    # kernels are told that columns >= c/8 of these rows are zero, as short rows tell them on the wire path (dp_fft1)
    ctx.fft_dev_hint_valid_cols(True, c_m // 8)
    msm_out = torch.zeros(18, dtype=torch.int64, device="cuda")
    exchange = parallel.make_exchange() if W > 1 else None
    fused = False
    if W > 1 and args.exchange == "fused":
        try:
            fused = parallel.attach_peers(ctx, 2 * (m // W) * 32)
        except dp.DpError as e:                       # e.g. no P2P path between the devices
            if rank == 0:
                print(f"fused exchange unavailable ({e}); using the NCCL all-to-all", file=sys.stderr)
        flag = torch.tensor([1 if fused else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        fused = bool(flag.item())

    def all_agree(ok):
        if W == 1:
            return bool(ok)
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return bool(flag.item())

    # Exchange modes of the resident transform at W > 1 (DESIGN.md section 4):
    #   devbarrier  rows -> peer stores -> device-side barrier kernel -> columns, queued asynchronously on ONE stream
    #   hostbarrier rows -> peer stores | dist.barrier() | columns
    #   nccl        rows | all_to_all_single | columns
    def fft_resident(src, dst, is_quot, is_inv, is_coset, mode):
        if W == 1:
            ctx.fft_dev(src.data_ptr(), dst.data_ptr(), is_quot, is_inv, is_coset)
        elif mode == "devbarrier":
            ctx.fft_dev_p2p_async(src.data_ptr(), dst.data_ptr(), is_quot, is_inv, is_coset)
        elif mode == "hostbarrier":
            ctx.fft_dev_rows_p2p(src.data_ptr(), is_quot, is_inv, is_coset)
            dist.barrier()                            # every rank's stores into my arena are complete
            ctx.fft_dev_cols(dst.data_ptr())
        else:
            s, r, blk = ctx.fft_dev_rows(src.data_ptr(), is_quot, is_inv, is_coset)
            exchange(s, r, blk)
            ctx.fft_dev_cols(dst.data_ptr())

    def barrier():
        torch.cuda.synchronize()
        ctx.sync()
        if W > 1:
            dist.barrier()

    # ---------------------------------------------------------------------------------- verification
    # Before anything is timed: the paths the timed region uses must reproduce the oracle on seeded input,
    # on every rank (dispatcher.rs:177-244 test_msm, 246-350 test_fft are the reference's versions of this).
    mode = "single" if W == 1 else ("nccl" if not fused else os.environ.get("DP_BENCH_EXCHANGE_MODE", "devbarrier"))
    verify = None
    if not args.no_verify:
        verify, mode = run_verify(args, torch, dist, ctx, rank, W, log_n, rand_fr, fft_resident, barrier, all_agree, mode, fused,
                                  dict(n=n, m=m, nb=nb, lo=lo, hi=hi, r_n=r_n, c_n=c_n, r_m=r_m, c_m=c_m))
        bad = [k for k, v in verify.items() if v is False]
        if bad:
            if rank == 0:
                print(json.dumps({"metric": "proofs_per_sec", "value": None, "verify": verify, "error": f"verification failed: {bad}"}), flush=True)
            barrier()
            if W > 1:
                dist.destroy_process_group()
            raise SystemExit(3)

    stats = {"msm_ms": [], "msm_acc_ms": [], "ntt_n_ms": [], "ntt_m_ms": [], "ntt_m_launches": 0, "sections_ms": {}}

    msm_outs = [torch.zeros(18, dtype=torch.int64, device="cuda") for _ in range(5)]
    ROUNDS = (5, 1, 5, 2)        # commitments per prover round (rounds 1, 2, 3, 5): issued together like join_all

    def step_resident(record=False):
        def section(name, t0):
            barrier()
            dt = (time.perf_counter() - t0) * 1e3
            if W > 1:
                t = torch.tensor([dt], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            stats["sections_ms"][name] = dt
            return time.perf_counter()

        if record:               # per-kernel timing wants one MSM at a time
            barrier()
            for k in range(N_MSM):
                ctx.msm_dev(lo, hi, scal[k % 3].data_ptr(), hi - lo, msm_out.data_ptr())
                stats["msm_ms"].append(ctx.last_timing()[0])
                stats["msm_acc_ms"].append(ctx.msm_breakdown()[1])
            barrier()
            t0 = time.perf_counter()
        k = 0
        for cnt in ROUNDS:
            ctx.msm_dev_batch([(lo, hi, scal[(k + j) % 3].data_ptr(), hi - lo, msm_outs[j].data_ptr()) for j in range(cnt)])
            k += cnt
        if record:
            t0 = section("msm_batches", t0)
        for k in range(N_INTT_N):
            fft_resident(in_n[k % 2], out_n, False, True, False, mode)
            if record and W == 1:
                stats["ntt_n_ms"].append(ctx.last_timing()[0])
        if record:
            t0 = section("intt_n", t0)
        for k in range(N_COSET_8N):
            fft_resident(in_m[k % 3], out_m, True, False, True, mode)
            if record and W == 1:
                ms, nl = ctx.last_timing()
                stats["ntt_m_ms"].append(ms)
                stats["ntt_m_launches"] = nl
        fft_resident(in_m[0], out_mi, True, True, True, mode)
        if record:
            section("coset_ntt_8n", t0)

    ext_stream = torch.cuda.ExternalStream(ctx.compute_stream())

    def timed(fn, steps, warmup, device_events=True):
        """seconds for `steps` calls of fn, max over ranks: CUDA events on the context's compute stream (every step
        ends with work on that stream), cross-checked by the host clock around barrier + synchronize"""
        for _ in range(warmup):
            fn()
        barrier()
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(ext_stream)
        for _ in range(steps):
            fn()
        e1.record(ext_stream)
        barrier()
        dt_host = time.perf_counter() - t0
        dt = e0.elapsed_time(e1) * 1e-3 if device_events else dt_host
        launches = ctx.launch_count() - l0
        if W > 1:
            t = torch.tensor([dt, dt_host], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt, dt_host = float(t[0].item()), float(t[1].item())
        timed.last_host = dt_host
        return dt, launches

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dt, launches = timed(step_resident, args.steps, args.warmup)
    dt_host = timed.last_host
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"intt_n": out_n, "coset_ntt_8n": out_m, "coset_intt_8n": out_mi}, msm_outs, rank, W)
    step_resident(record=True)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = dt / args.steps * 1e3
    value = args.steps / dt

    # ---- e2e through the host-buffer API (pinned host memory, copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        # staging buffers next to the GPU: pinned pages land on the NUMA node of the CPU that allocates them, and with
        # one process per GPU about half of the ranks would otherwise copy across the inter-socket link
        import contextlib
        aff_stack = contextlib.ExitStack()
        host_aff = aff_stack.enter_context(parallel.near_gpu(local)) if os.environ.get("DP_BENCH_NO_AFFINITY", "0") != "1" else "unchanged (DP_BENCH_NO_AFFINITY)"

        def pinned(t):
            return t.cpu().pin_memory()

        h_scal = pinned(scal[0])
        h_in_n = pinned(in_n[0])
        # what the dispatcher holds for a quotient-domain transform is the n coefficients: each of my rows has c/8
        # non-zero leading entries, and only those cross PCIe (dp_fft1_rows_short zero-extends on the device the way
        # Radix2EvaluationDomain::fft_in_place resizes its input, worker.rs:81-85)
        short = c_m // 8
        h_in_m = pinned(in_m[0].view(rows_m, c_m, 4)[:, :short, :].contiguous())
        h_in_m_full = pinned(in_m[0])                 # the inverse transform of round 3 takes full rows
        h_out_n = torch.empty((cols_n * r_n, 4), dtype=torch.int64).pin_memory()
        h_out_m = torch.empty((cols_m * r_m, 4), dtype=torch.int64).pin_memory()
        wl_n, wl_m = disp.fft_workloads(log_n, W), disp.fft_workloads(log_m, W)
        from distributed_plonk_b200 import schedule

        # fft_init + fft1 (async H2D) + fft2_prepare (async row/column kernels) ... fft2 (D2H, blocks for
        # that task only); at W > 1 every task has its own send/recv buffers and the all-to-all is enqueued on
        # the context's compute stream (no host synchronisation per transform)
        e2e_exchange = None
        if W > 1:
            e2e_exchange = exchange if os.environ.get("DP_BENCH_ASYNC_EXCHANGE", "1") != "1" else parallel.make_stream_ordered_exchange(ctx)
        runner = schedule.Runner(ctx, e2e_exchange)
        t_n = schedule.Transform(h_in_n.data_ptr(), h_out_n.data_ptr(), h_out_n.numel() * 8, wl_n, rows_n, False, True, False)
        t_m = schedule.Transform(h_in_m.data_ptr(), h_out_m.data_ptr(), h_out_m.numel() * 8, wl_m, rows_m, True, False, True, row_len=short)
        t_mi = schedule.Transform(h_in_m_full.data_ptr(), h_out_m.data_ptr(), h_out_m.numel() * 8, wl_m, rows_m, True, True, True)
        jobs = [t_n] * N_INTT_N + [t_m] * N_COSET_8N + [t_mi] * N_COSET_INTT_8N
        com = schedule.Commitment(lo, hi, h_scal.data_ptr(), hi - lo)
        host_of = {h_out_n.data_ptr(): h_out_n, h_out_m.data_ptr(): h_out_m}

        # Two host schedules over the same work (distributed_plonk_b200/schedule.py): serial = the commitments of
        # each prover round as one batch, then the transforms with two tasks of look-ahead; overlapped = a
        # commitment queued (dp_msm_submit) after every second transform.  The overlapped one is timed only if it
        # first reproduces the serial one bit for bit on this box and is not slower in a one-step trial.
        e_steps = max(1, args.steps)
        try:
            step_e2e, e2e_mode = schedule.pick_schedule(
                runner, jobs, com, ROUNDS, checksum=lambda t: int(host_of[t.out_ptr].sum()), timed=lambda f: timed(f, 1, 0, False)[0],
                all_agree=all_agree, allow_overlap=os.environ.get("DP_BENCH_E2E_SERIAL", "0") != "1")
            dt_e, _ = timed(step_e2e, e_steps, 1, False)
        except Exception as exc:   # whatever went wrong while choosing: the serial schedule is the one round 1 measured
            if W > 1:
                raise
            ctx.sync()
            e2e_mode = f"serial (schedule selection failed: {str(exc)[:120]})"
            dt_e, _ = timed(lambda: runner.run_serial(jobs, com, ROUNDS, 2), e_steps, 1, False)
        h2d = W * (N_MSM * (hi - lo) * 32 + N_INTT_N * rows_n * c_n * 32 + N_COSET_8N * rows_m * short * 32 + N_COSET_INTT_8N * rows_m * c_m * 32)
        d2h = W * (N_MSM * 144 + N_INTT_N * cols_n * r_n * 32 + (N_COSET_8N + N_COSET_INTT_8N) * cols_m * r_m * 32)
        e2e = {"value": e_steps / dt_e, "unit": "proofs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": dt_e / e_steps * 1e3, "steps": e_steps, "schedule": e2e_mode,
               "exchange": "none" if W == 1 else ("all_to_all_single enqueued on the compute stream" if getattr(e2e_exchange, "stream_ordered", False)
                                                  else "all_to_all_single, host-synchronised"),
               "timing": "host clock between barrier+synchronize (copies run on three streams)", "host_affinity": host_aff}
        del h_scal, h_in_n, h_in_m, h_in_m_full, h_out_n, h_out_m

    # ---- the same proof with every polynomial resident on the worker (SURVEY 8f-1): witness in once, commitments and
    # evaluations out - what the schema's round3*/round4*/round5* RPCs (hello_world.capnp:26-44) make possible
    e2e_res = None
    if W == 1 and not args.no_e2e and os.environ.get("DP_BENCH_SKIP_RESIDENT", "0") != "1":
        try:
            from distributed_plonk_b200 import resident
            e2e_res = resident.bench_leg(ctx, torch, log_n, rand_fr, timed, steps=max(1, args.steps))
        except Exception as e:  # the headline numbers above must survive a failure of this extra
            e2e_res = {"error": str(e)[:300]}
            ctx.sync()

    if not args.no_e2e:
        aff_stack.close()   # back on every host CPU (the CPU baseline below uses all of them)

    # ---- "next" row, measured beside the schedule (not part of the step): round-2 grand product
    perm = None
    if W == 1:
        wt = [rand_fr(5 * n) for _ in range(3)]
        zt = torch.empty((n, 4), dtype=torch.int64, device="cuda")
        bg = np.array([[3, 1, 4, 1], [5, 9, 2, 6]], dtype=np.uint64)
        for _ in range(3):
            ctx.perm_product_dev(wt[0].data_ptr(), wt[1].data_ptr(), wt[2].data_ptr(), 5, n, bg[0], bg[1], zt.data_ptr())
        perm = {"n": n, "wire_types": 5, "gpu_ms": ctx.last_timing()[0], "gpu_rows_per_sec": n / (ctx.last_timing()[0] * 1e-3)}
        del wt, zt

    # ---- "next" row 8f-1, measured beside the schedule: rounds 3-5 on device-resident polynomials
    rounds = None
    if W == 1 and os.environ.get("DP_BENCH_SKIP_ROUNDS", "0") != "1":
        try:
            arrs = [rand_fr(m) for _ in range(25)]
            qo = torch.empty((m, 4), dtype=torch.int64, device="cuda")
            ch = np.array([[3, 1, 4, 1], [5, 9, 2, 6], [5, 3, 5, 8], [9, 7, 9, 3], [2, 3, 8, 4], [6, 2, 6, 4], [3, 3, 8, 3], [2, 7, 9, 5]], dtype=np.uint64)
            ptr = [t.data_ptr() for t in arrs]
            ms = {}
            for _ in range(2):
                ctx.quotient_evals_dev(ptr[:13], ptr[13:18], ptr[18:23], ptr[23], ptr[24], ch[:5], ch[5], ch[6], ch[7], qo.data_ptr())
            ms["quotient_evals_8n"] = ctx.last_timing()[0]
            for _ in range(2):
                ctx.poly_eval(ptr[0], ch[5], n + 3)
            ms["poly_eval_n"] = ctx.last_timing()[0]
            for _ in range(2):
                ctx.poly_div_linear(ptr[0], ch[5], n + 3, qo.data_ptr())
            ms["poly_div_linear_n"] = ctx.last_timing()[0]
            for _ in range(2):
                ctx.poly_lincomb(ptr[:12], ch[[0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3]], out_len=n + 3, lens=[n + 3] * 12, out_ptr=qo.data_ptr())
            ms["poly_lincomb_12xn"] = ctx.last_timing()[0]
            rounds = {"gpu_ms": ms, "note": "device-resident polynomials; quotient over the 8n coset domain (25 input arrays), the others over n+3 coefficients"}
            del arrs, qo
        except Exception as e:  # the headline numbers above must survive a failure of this extra
            rounds = {"error": str(e)[:200]}

    if rank != 0:
        if W > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (largest share of the step)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    adds, bf = schedule_units(log_n)
    msm_total = sum(stats["msm_ms"])
    acc_total = sum(stats["msm_acc_ms"])
    ntt_m_total = sum(stats["ntt_m_ms"]) if stats["ntt_m_ms"] else stats["sections_ms"].get("coset_ntt_8n", 0.0)
    shares = {"msm_accumulate_kernel": acc_total, "ntt_tile_kernel(8n)": ntt_m_total}
    dominant = max(shares, key=shares.get)
    n_pass = max(1, stats["ntt_m_launches"])
    if dominant == "msm_accumulate_kernel" and stats["msm_acc_ms"]:
        per_launch_ms = statistics.mean(stats["msm_acc_ms"])
        alg_bytes = (hi - lo) * (32 + 96)                 # SURVEY 8d: each scalar and each affine base once
    else:
        per_launch_ms = statistics.mean(stats["ntt_m_ms"]) / n_pass if stats["ntt_m_ms"] else float("nan")
        alg_bytes = 64 * m                                 # one read + one write of every element per pass
    achieved = alg_bytes / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms == per_launch_ms else None
    traffic = None
    try:  # DRAM bytes per launch of the same kernel at this size, from the committed ncu capture (profiles/)
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = "msm_accumulate_kernel" if dominant.startswith("msm") else "ntt_tile_kernel"
        if W == 1:
            ent = tr.get(key, {}).get(str(log_n) if dominant.startswith("msm") else str(log_m))
            if ent:
                traffic = ent["bytes"]
    except (OSError, ValueError, KeyError):
        pass
    # the bound that actually applies: 32x32+64 multiply-accumulates on the FMA pipe.  Peak = plain
    # IMAD.WIDE.U32 rate measured on this part (profiles/r01_microbench_pipes.txt: 61.9 lane-MAC/clk/SM);
    # the carry form IMAD.WIDE.U32.X that multi-precision chains need sustains 28.3 (r01_microbench_carry_chains.txt)
    sm_clk = (clocks or {}).get("sm_mhz") or 1965.0
    mac_peak = 61.9 * 148 * sm_clk * 1e6
    tuning = ctx.msm_tuning()                                          # dp_init's choice: plain XYZZ chunks or batched-affine tree levels first
    lv = tuning["levels"]
    # Fq products per bucket addition: 10 (XYZZ mixed addition), or with L tree levels 6.4 for the (1 - 2^-L) of the additions the
    # levels do and 10 for the rest
    prod_per_add = 10.0 if lv == 0 else 6.4 * (1 - 0.5 ** lv) + 10.0 * 0.5 ** lv
    macs_msm = (hi - lo) * 1.0 * ((256 + 19) // 20) * prod_per_add * 288   # digits x Fq products x 12x12x2 MACs
    macs_ntt = (m / 2) * log_m * 128 + 4 * m * 128                     # butterflies + twiddle/coset products, 8x8x2 MACs
    compute = {
        "bound": "int32 multiply-add pipe", "peak_mac_per_s": mac_peak, "peak_source": "measured IMAD.WIDE.U32 rate x 148 SMs x sampled SM clock",
        "msm_accumulate_frac": (macs_msm / (statistics.mean(stats["msm_acc_ms"]) * 1e-3) / mac_peak) if stats["msm_acc_ms"] else None,
        "ntt_tile_8n_frac": (macs_ntt / (statistics.mean(stats["ntt_m_ms"]) * 1e-3) / mac_peak) if stats["ntt_m_ms"] else None,
        "carry_form_ceiling_frac": 28.3 / 61.9,
    }
    ntt_traffic = None
    try:
        ent = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get("ntt_tile_kernel", {}).get(str(log_m))
        if W == 1 and ent:
            ntt_traffic = ent["bytes"]
    except (OSError, ValueError, KeyError):
        pass
    ntt_hbm = None
    if stats["ntt_m_ms"]:
        per_tr = statistics.mean(stats["ntt_m_ms"])
        per = per_tr / n_pass
        ntt_hbm = {"kernel": "ntt_tile_kernel(8n)", "achieved": 64 * m / (per * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                   "frac": 64 * m / (per * 1e-3) / 1e9 / peak, "avg_launch_ms": per, "algorithmic_bytes_per_launch": 64 * m,
                   "passes_per_transform": n_pass, "transform_ms": per_tr, "traffic": ntt_traffic,
                   # against SURVEY 8d's bytes_min = 64 N for the WHOLE transform (one read + one write of every element)
                   "per_transform_frac_of_bytes_min": 64 * m / (per_tr * 1e-3) / 1e9 / peak}
    if lv and dominant.startswith("msm"):
        traffic = None          # the committed ncu capture is of the plain accumulation kernel, not of the tree levels
    roofline = {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg_bytes), "avg_launch_ms": per_launch_ms,
                "note": "both kernels are bound by the INT32 multiply pipe, not HBM (DESIGN.md); HBM fraction reported as BASELINE asks"
                        + ("" if lv == 0 or not dominant.startswith("msm") else
                           f"; the accumulation phase timed here is {lv} batched-affine tree levels (aff_k1/k2/k3) + msm_accumulate_kernel, chosen by dp_init's tuning"),
                "step_share_ms": shares}
    exch = {"single": "none", "devbarrier": "fused peer-memory stores + device-side barrier kernel, transforms queued asynchronously",
            "hostbarrier": "fused peer-memory stores, host barrier per transform", "nccl": "nccl all_to_all_single"}[mode]
    line = {
        "metric": "proofs_per_sec", "value": value, "unit": "proofs/s", "n_gpus": W, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 limbs (255/381-bit modular integer)", "data": "synthetic",
        "config": dict(workload_config(log_n, W), exchange=exch),
        "timing": {"how": "CUDA events on the library's compute stream, max over ranks", "host_clock_ms_per_step": dt_host / args.steps * 1e3},
        "gpu_launches": int(launches), "clocks": clocks, "verify": verify,
        "msm_g1_adds_per_sec": (adds / N_MSM) * (hi - lo) / nb / (statistics.mean(stats["msm_ms"]) * 1e-3) * W if stats["msm_ms"] else None,
        "ntt_butterflies_per_sec": butterflies(log_m) / (statistics.mean(stats["ntt_m_ms"]) * 1e-3) if stats["ntt_m_ms"] else None,
        "breakdown_ms": {"msm_total_one_at_a_time": msm_total, "msm_accumulate": acc_total, "intt_n_total": sum(stats["ntt_n_ms"]),
                         "coset_ntt_8n_total": sum(stats["ntt_m_ms"]), "sections_max_over_ranks": stats["sections_ms"]},
        "roofline": roofline, "roofline_ntt": ntt_hbm, "roofline_compute": compute, "e2e": e2e, "e2e_resident": e2e_res,
        "msm_tuning": {"levels_used": lv, "probe": tune_probe, "in_process": {k: v for k, v in tuning.items() if k != "levels"},
                       "what": "a child process timed one MSM over this rank's window table with the plain pipeline and with 1, 2 and 3 batched-affine "
                               "tree levels in front of it (dp_init with DP_MSM_TUNE=2, ms_by_levels); levels are used in this run only if every "
                               "result was identical to the plain pipeline's and the best candidate >= 2 % faster"},
        "next_row_perm_product": perm, "next_row_rounds_3_to_5": rounds,
    }
    if not args.no_cpu and W == 1:
        from oracle import loader as orc
        orc.build()
        orc.set_num_threads(os.cpu_count() or 1)
        cb = cpu_sample(log_n)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "value_fair")}
        line["cpu_baseline"]["msm_g1_adds_per_sec"] = cb["msm_g1_adds_per_sec"]
        if perm:   # the dispatcher's serial loop with one division per row (dispatcher2.rs:329-345), sampled
            pn = 1 << 14
            pw = [np.stack([orc.gen_fr(90 + 7 * k + i, pn) for i in range(5)]) for k in range(3)]
            t0 = time.perf_counter()
            orc.perm_product(pw[0], pw[1], pw[2], orc.gen_fr(98, 1)[0], orc.gen_fr(99, 1)[0])
            perm["cpu_rows_per_sec"] = pn / (time.perf_counter() - t0)
            perm["cpu_note"] = "oracle restatement, 1 thread (the reference loop is serial), 2^14-row sample"
        if rounds and "gpu_ms" in rounds:   # dispatcher2.rs:434-504 restated (all host threads), 2^17-point sample
            qm, qn = 1 << 17, 1 << 14
            qa = [np.stack([orc.gen_fr(200 + 20 * k + i, qm) for i in range(c)]) for k, c in enumerate((13, 5, 5))]
            t0 = time.perf_counter()
            orc.quotient_evals(qa[0], qa[1], qa[2], orc.gen_fr(290, qm), orc.gen_fr(291, qm), orc.gen_fr(292, 5), orc.gen_fr(293, 1)[0],
                               orc.gen_fr(294, 1)[0], orc.gen_fr(295, 1)[0], qn)
            rounds["cpu_quotient_points_per_sec"] = qm / (time.perf_counter() - t0)
            rounds["gpu_quotient_points_per_sec"] = m / (rounds["gpu_ms"]["quotient_evals_8n"] * 1e-3)
    print(json.dumps(line), flush=True)
    if W > 1:
        dist.destroy_process_group()


def run_verify(args, torch, dist, ctx, rank, W, log_n, rand_fr, fft_resident, barrier, all_agree, mode, fused, g):
    """Seeded inputs through the paths the timed region uses, checked against the oracle (tests/ hold the
    small-size byte-for-byte comparisons; this is the full-size, every-rank check the driver can see):
      * coset-NTT(8n) of n coefficients through the resident multi-GPU transform: output positions in every
        rank's column block against an O(n) Horner evaluation by the oracle; at W > 1 the fused peer-store paths
        must also equal the NCCL all-to-all path bit for bit (the whole output, on every rank);
      * iNTT(n): the same spot check with the inverse flags;
      * sharded MSM(n+32): the sum of the ranks' partials against the oracle's Pippenger (log_n <= 22) and against
        (sum s_i k_i) * G for the synthetic bases k_i * G (every size)."""
    from oracle import loader as orc
    if rank == 0:
        orc.build()
        orc.set_num_threads(os.cpu_count() or 1)
    n, m, nb, lo, hi = g["n"], g["m"], g["nb"], g["lo"], g["hi"]
    r_n, c_n, r_m, c_m = g["r_n"], g["c_n"], g["r_m"], g["c_m"]
    out = {}
    vgen = torch.Generator(device="cuda")
    vgen.manual_seed(0x5EED)                              # the same on every rank: every rank can build its own rows

    def gather_rows(vec, r, c, n_valid_cols):
        """my rows of the dispatcher's [r][c] matrix of vec (x[i + r*j]), zero beyond column n_valid_cols"""
        rows = r // W
        t = torch.zeros((rows, c, 4), dtype=torch.int64, device="cuda")
        t[:, :n_valid_cols, :] = vec.view(n_valid_cols, r, 4)[:, rank * rows:(rank + 1) * rows, :].permute(1, 0, 2)
        return t.view(-1, 4)

    def spot_positions(r, c):
        """(local column, k1) pairs in my column block: the ends and the middle of the block, pseudo-random rows"""
        cols = c // W
        picks = [(0, 1), (cols - 1, r - 1), (cols // 2, (7919 * (rank + 1)) % r), (cols // 3, (104729 * (rank + 3)) % r)]
        return picks

    def spot_check(name, dst, vec_host, n_coeffs, r, c, inverse, coset):
        cols = c // W
        picks = spot_positions(r, c)
        vals = torch.stack([dst[k2 * r + k1] for k2, k1 in picks]).contiguous()            # [P,4] int64
        ks = torch.tensor([(rank * cols + k2) + c * k1 for k2, k1 in picks], dtype=torch.int64, device="cuda")
        if W > 1:
            all_v = [torch.empty_like(vals) for _ in range(W)]
            all_k = [torch.empty_like(ks) for _ in range(W)]
            dist.all_gather(all_v, vals)
            dist.all_gather(all_k, ks)
            vals, ks = torch.cat(all_v), torch.cat(all_k)
        ok = True
        if rank == 0:
            got = vals.cpu().numpy().view(np.uint64)
            want = orc.ntt_outputs_at(vec_host, r * c, ks.cpu().numpy().astype(np.uint64), inverse, coset)
            ok = bool(np.array_equal(got, want))
        out[name] = all_agree(ok)
        out[name + "_positions"] = int(ks.numel())

    # ---- coset NTT on the quotient domain (25 of the 33 transforms of a proof)
    p = rand_fr(n, vgen)
    p_host = p.cpu().numpy().view(np.uint64) if rank == 0 else None
    rows_in = gather_rows(p, r_m, c_m, c_m // 8)
    dst = torch.empty(((c_m // W) * r_m, 4), dtype=torch.int64, device="cuda")
    modes = ["single"] if W == 1 else ([mode] + [x for x in ("devbarrier", "hostbarrier") if x != mode and fused] + (["nccl"] if mode != "nccl" else []))
    results = {}
    for md in modes:
        dst.zero_()
        torch.cuda.synchronize()      # torch's stream (inputs just built) -> the library's own streams
        try:
            fft_resident(rows_in, dst, True, False, True, md)
            barrier()
            results[md] = dst.clone()
            ok = True
        except Exception as exc:      # e.g. a barrier time-out: the mode is reported as failed and not used
            if rank == 0:
                print(f"verify: exchange mode {md} failed: {exc}", file=sys.stderr)
            ok = False
            try:
                barrier()
            except Exception:
                pass
        if not all_agree(ok):
            results.pop(md, None)
            out[f"ntt_mode_{md}_ran"] = False
    ref_mode = "nccl" if "nccl" in results else (modes[0] if modes[0] in results else None)
    if ref_mode is None:
        out["coset_ntt_8n_horner"] = False
        return out, mode
    spot_check("coset_ntt_8n_horner", results[ref_mode], p_host, n, r_m, c_m, False, True)
    out["coset_ntt_8n_path_checked"] = ref_mode
    for md in [x for x in results if x != ref_mode]:
        out[f"ntt_{md}_equals_{ref_mode}_bitwise"] = all_agree(bool(torch.equal(results[md], results[ref_mode])))
    # choose the timed mode: the preferred one if it ran and agreed, else the next that did
    def good(md):
        return md in results and (md == ref_mode or out.get(f"ntt_{md}_equals_{ref_mode}_bitwise", False))
    if not good(mode):
        for md in ("hostbarrier", "nccl"):
            if good(md):
                out["fallback_from"] = mode
                mode = md
                break
    del results, rows_in, dst, p

    # ---- iNTT on the gate domain (7 of the 33)
    q = rand_fr(n, vgen)
    q_host = q.cpu().numpy().view(np.uint64) if rank == 0 else None
    rows_in = gather_rows(q, r_n, c_n, c_n)
    dst = torch.empty(((c_n // W) * r_n, 4), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    fft_resident(rows_in, dst, False, True, False, mode)
    barrier()
    spot_check("intt_n_horner", dst, q_host, n, r_n, c_n, True, False)
    del rows_in, dst, q

    # ---- sharded MSM (dispatcher.rs:177-244): every rank its index range, partials summed by the checker
    s_all = rand_fr(nb, vgen)
    s_all[n + 2:] = 0
    part = torch.zeros(18, dtype=torch.int64, device="cuda")
    s_mine = s_all[lo:hi].contiguous()
    torch.cuda.synchronize()
    ctx.msm_dev(lo, hi, s_mine.data_ptr(), hi - lo, part.data_ptr())
    parts = [part]
    if W > 1:
        parts = [torch.empty_like(part) for _ in range(W)]
        dist.all_gather(parts, part)
    ok_dlog, ok_orc = True, None
    if rank == 0:
        total = np.frombuffer(parts[0].cpu().numpy().tobytes(), dtype=np.uint8).copy()
        for t in parts[1:]:
            total = orc.g1_add(total, np.frombuffer(t.cpu().numpy().tobytes(), dtype=np.uint8).copy())
        s_host = s_all.cpu().numpy().view(np.uint64)
        k = synthetic_k(GEN_SEED, np.arange(nb, dtype=np.uint64))
        k[3] = 0
        k[n:] = 0                                               # the infinity entries contribute nothing
        t_dlog = orc.fr_dot_u64(s_host, k)
        want = orc.affine_to_jacobian(orc.g1_mul(orc.g1_generator(), t_dlog))
        ok_dlog = bool(np.array_equal(orc.normalize(total), orc.normalize(want)))
        if log_n <= 22:
            bases_host = ctx.get_bases(0, nb)
            ok_orc = bool(np.array_equal(orc.normalize(total), orc.normalize(orc.msm(bases_host, s_host))))
            del bases_host
    out["sharded_msm_vs_dlog_identity"] = all_agree(ok_dlog)
    if log_n <= 22:
        out["sharded_msm_vs_oracle_pippenger"] = all_agree(ok_orc if rank == 0 else True)
    out["timed_exchange_mode"] = mode
    return out, mode


if __name__ == "__main__":
    main()
