#!/usr/bin/env python3
"""bench.py — BLS12-381 G1 MSM/s @ 2^26 (primary) and Fr NTT/s @ 2^24 on N B200s, next to the CPU restatement of
the reference.  Contract: one JSON line on stdout (rank 0).

  python bench.py --gpus 1 --steps 5 --warmup 3            # our arm
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # ... and the last timed step's outputs as DIR/*.npy
  python bench.py --impl reference --steps 2 --warmup 1    # the reference's algorithms on the host cores (oracle port)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full MSM over n = 2^26 synthetic (base, scalar) pairs (bases P_i = b_i*G generated on the device,
uniform scalars); with N > 1 the MSM shards with no data-path collective: the device-resident leg by bucket slices
(every rank holds all pairs and owns 1/N of every window's buckets; --shard chunks: contiguous input chunks), the
host-buffer leg by input chunks; one NCCL all-gather exchanges a partial point per rank and every rank adds the N
points ("strong" scaling: total work fixed).  The NTT leg (n = 2^24, forward) is timed the same way right after and reported under
"ntt" ("replicas only": with N > 1 every rank transforms its own vector).
`value` has inputs resident in HBM; `e2e` goes through the host-buffer C-ABI call (H2D of bases+scalars from pinned
host memory and D2H of the result inside the timed region)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# IMAD.WIDE.U32(.X) issues at 32 per clock per SM on B200 (tools/imad_microbench.cu, profiles/r01_imad_microbench.jsonl):
# 32 x 148 SMs x 1.965 GHz = 9.31 T/s; the element-wise Fq multiplication kernel reaches 9.05 T/s of it
# (profiles/r01_field_bench.jsonl), the synthetic carry-chain microbenchmark 8.5 T/s.
IMAD_PEAK_WIDE_PER_S = 9.31e12
IMAD_PEAK_SOURCE = "32 IMAD.WIDE/clk/SM x 148 SMs x 1.965 GHz (tools/imad_peak.cu: SASS-verified count, profiles/r02_imad_peak.jsonl)"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_NTT_ROWS = 1 << 16    # --dump-outputs: rows of an NTT output kept (a fixed, seeded sample; 4 MB per transform)


def u64_as_f64(limbs: np.ndarray) -> np.ndarray:
    """u64 limbs -> their 32-bit halves (low half first) as float64, which holds every such value exactly"""
    return np.ascontiguousarray(limbs, dtype=np.uint64).view(np.uint32).astype(np.float64)


def msm_work(n: int, c: int, W: int, limbs32: int):
    """SURVEY.md §8(d): Fq modmuls = 10*n*W + 14*2^c*W ; wide MADs per modmul = 2L^2 + L ; bytes = n*(2*8N + 32)"""
    modmuls = 10.0 * n * W + 14.0 * (1 << c) * W
    return modmuls, modmuls * (2 * limbs32 * limbs32 + limbs32), n * (2 * 4 * limbs32 + 32)


# ------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference arm: the C restatement of ark-ec / ark-poly (oracle/ark_oracle.c — the Rust crates cannot be built
    in this image) on all host threads.  Each step is a bounded sample: n/8 pairs for the MSM on all threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import coracle as C
    from oracle import pyoracle as O
    threads = C.num_threads()
    log_n = args.log_n_msm
    n = 1 << log_n
    # bounded sample: n/4 pairs per step (x4) above 2^22 unless --ref-full; the window is the one ark-ec would pick for the FULL
    # problem (c = ln_without_floats(chunk)+2 for chunks of n / (threads/2) pairs, variable_base/mod.rs:445-449,521-535), so the
    # sample does the same work per pair as the full run
    shrink = 1 if (args.ref_full or log_n <= 22) else 4
    ns = n // shrink
    c_full = C.window_size(max(1, n // max(1, threads // 2)))
    cv = O.BLS12_381
    rng = np.random.default_rng(args.seed)
    bases, base_kind = None, ""
    try:   # real distinct bases b_i*G: produced by the device generator when a GPU is present (input preparation, not the timed path)
        import torch
        if torch.cuda.is_available():
            from algebra_b200 import _lib
            d = torch.empty((ns, 12), dtype=torch.int64, device="cuda")
            _lib.check(_lib.lib().b200_gen_bases_dev(0, args.seed, ns, d.data_ptr(), None, torch.cuda.current_stream().cuda_stream))
            bases = d.cpu().numpy().view(np.uint64)
            del d
            torch.cuda.empty_cache()
            base_kind = "distinct bases b_i*G"
    except Exception:
        bases = None
    if bases is None:   # no GPU: a block of 64 real points tiled (the arithmetic cost is data-independent)
        ks = [int(x) for x in rng.integers(1, 1 << 62, size=64)]
        pts = cv.encode_affine([cv.mul(cv.G, k) for k in ks])
        bases = np.ascontiguousarray(np.tile(pts, (ns // 64 + 1, 1))[:ns])
        base_kind = "64 distinct points tiled"
    scal = rng.integers(0, 1 << 64, size=(ns, 4), dtype=np.uint64)
    scal[:, 3] &= np.uint64((1 << 62) - 1)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        C.msm(0, bases, scal, threads=threads, c=c_full)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    t_full = statistics.mean(times) * shrink
    # NTT leg: full 2^log_n_ntt forward transform, all threads
    x = rng.integers(0, 1 << 64, size=(1 << args.log_n_ntt, 4), dtype=np.uint64)
    x[:, 3] &= np.uint64((1 << 62) - 1)
    C.fft(1, x[: 1 << 16], False, None, threads)
    tn = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        C.lib().ark_fft(1, x.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), args.log_n_ntt, 0, None, threads)
        tn.append(time.perf_counter() - t0)
    sample = f"MSM: {ns} of {n} pairs (1/{shrink}) on {threads} threads, time x{shrink}, {base_kind}; chunking of ark-ec with the " \
             f"window of the full problem (c={c_full} per chunk of n/{max(1, threads // 2)}); NTT: full 2^{args.log_n_ntt}"
    v = 1.0 / t_full
    line = {
        "impl": "reference", "metric": "BLS12-381 G1 MSM/s @2^%d" % log_n, "value": v, "unit": "MSM/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_full * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64 limbs (Montgomery, 6x64-bit Fq / 4x64-bit Fr)", "data": "synthetic",
        "config": {"workload": "BLS12-381 G1 VariableBaseMSM n=2^%d, uniform scalars" % log_n, "seed": args.seed},
        "cpu_baseline": {"value": v, "unit": "MSM/s", "cores": threads, "kind": "port", "sample": sample, "steps": args.steps,
                         "warmup": args.warmup},
        "e2e": {"value": v, "unit": "MSM/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ntt": {"metric": "BLS12-381 Fr NTT/s @2^%d" % args.log_n_ntt, "value": 1.0 / statistics.mean(tn), "unit": "NTT/s",
                "ms_per_step": statistics.mean(tn) * 1e3, "steps": len(tn)},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of every leg of the arm; the b200 arm's cpu_baseline is one step of the reference arm (its own "
                         "steps/warmup are reported in it), a bounded sample: at 2^26 that step alone takes about a minute")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n-msm", type=int, default=26)
    ap.add_argument("--log-n-ntt", type=int, default=24)
    ap.add_argument("--curve", type=int, default=0, help="0 = BLS12-381 G1 (metric), 1 = BN254 G1")
    ap.add_argument("--window", type=int, default=0, help="Pippenger window override (0 = auto)")
    ap.add_argument("--affine-levels", type=int, default=-1, help="batched-affine pre-reduction levels (-1 = auto)")
    ap.add_argument("--shard", default="auto", choices=["auto", "buckets", "chunks"],
                    help="N > 1, device-resident leg: bucket slices over replicated inputs (auto) or input chunks")
    ap.add_argument("--seed", type=int, default=20260922)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-ntt", action="store_true", help="skip the NTT leg (MSM tuning runs)")
    ap.add_argument("--ref-full", action="store_true", help="--impl reference: time the full n instead of the n/4 sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl b200: write what the last timed step of the device-resident legs returned as DIR/<name>.npy (float64, "
                         "exact 32-bit halves of the u64 limbs): msm_affine (the MSM `value` leg), ntt_fft and ntt_ifft (%d seeded rows "
                         "of each transform); the host-buffer e2e legs compute the same MSM, checked by e2e.same_result" % DUMP_NTT_ROWS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import algebra_b200 as ab
    from algebra_b200 import _lib
    from algebra_b200 import variable_base as VB

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    cv = ab.params.CURVES[args.curve]
    N = cv.N
    n_total = 1 << args.log_n_msm
    # N > 1, device-resident leg: "buckets" = every rank holds all n pairs (replicated, as an SRS is) and owns 1/N of every
    # window's buckets; "chunks" = rank r holds and processes the pairs [n*r/N, n*(r+1)/N).  The host-buffer (e2e) leg always
    # ships chunks: each GPU then receives 1/N of the bytes.
    shard = args.shard if world > 1 else "chunks"
    if shard == "auto":
        shard = "buckets"
    n_chunk = n_total // world
    n_local = n_total if shard == "buckets" else n_chunk
    c_lo = rank * n_chunk if shard == "buckets" else 0     # this rank's chunk inside its resident arrays
    st = torch.cuda.current_stream().cuda_stream
    hbm_peak, peak_src = measured_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- synthetic inputs, generated on the device
    d_bases = torch.empty((n_local, 2 * N), dtype=torch.int64, device=dev)
    d_b = torch.empty((n_local,), dtype=torch.int64, device=dev)
    d_scal = torch.empty((n_local, 4), dtype=torch.int64, device=dev)
    gen_seed = args.seed + (0 if shard == "buckets" else 1000 * rank)    # replicated inputs: the same stream on every rank
    _lib.check(L.b200_gen_bases_dev(cv.cid, gen_seed, n_local, d_bases.data_ptr(), d_b.data_ptr(), st))
    _lib.check(L.b200_gen_scalars_dev(cv.ntt_field_id, gen_seed + 7777, n_local, d_scal.data_ptr(), st))
    VB.set_window(args.window)
    VB.set_affine_levels(args.affine_levels)

    from algebra_b200 import dist as D

    def msm_step(bases, scal):
        # C ABI MSM on this rank's chunk (synchronises), then — for N > 1 — NCCL all-gather of the 144-byte partial
        # points and the local sum of N points (algebra_b200/dist.py)
        if shard == "buckets" and bases.__class__.__module__.startswith("torch"):
            return D.msm_bucket_sliced(cv, bases, scal)
        return D.msm_sharded(cv, bases, scal)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, out

    # ---------------- MSM, device resident
    for _ in range(args.warmup):
        res = msm_step(d_bases, d_scal)
    phase = {k: 0.0 for k in ["digits_hist", "scan", "scatter", "accumulate", "reduce", "combine", "total"]}
    launches0 = L.b200_launch_count()

    def counted_step():
        r = msm_step(d_bases, d_scal)
        t = VB.last_timings()
        for k in phase:
            phase[k] += t[k]
        return r

    with ClockSampler(local_rank) as clk:
        ms_msm, res = timed(counted_step, args.steps)
    launches = int(L.b200_launch_count() - launches0)
    tm = VB.last_timings()
    for k in phase:
        phase[k] /= args.steps
    clocks = clk.summary()

    dump = {}     # --dump-outputs: name -> float64 array, written by rank 0 once the legs are done

    def write_dump():
        if rank == 0 and args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    if args.dump_outputs:
        # the affine point is the group element itself; the Jacobian limbs the call returns depend on the order of the additions
        dump["msm_affine"] = u64_as_f64(ab.into_affine(cv, res))

    # ---------------- verification: MSM(b_i*G, s_i) == (sum s_i*b_i mod r) * G, all ranks' shards included
    verified = None
    if not args.no_verify:
        r_mod = cv.fr.modulus
        sc = d_scal[c_lo:c_lo + n_chunk].cpu().numpy().view(np.uint64)     # every rank checks one chunk; the totals are gathered
        bb = d_b[c_lo:c_lo + n_chunk].cpu().numpy().view(np.uint64)
        # scalars are Montgomery residues: value = limbs * R^-1; do the dot product on the raw limbs, fix up at the end
        # 16-bit pieces in float64: products < 2^32, 2^20-term sums < 2^52 -> exact BLAS dot products
        tot, CH = 0, 1 << 20
        for lo in range(0, n_chunk, CH):
            s16 = sc[lo:lo + CH].view(np.uint16).reshape(-1, 16).astype(np.float64)
            b16 = bb[lo:lo + CH].view(np.uint16).reshape(-1, 4).astype(np.float64)
            m = s16.T @ b16
            for j in range(16):
                for k in range(4):
                    tot += int(m[j, k]) << (16 * (j + k))
        tot = tot * pow(cv.fr.R, -1, r_mod) % r_mod
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, tot)
            tot = sum(parts) % r_mod
        if rank == 0:
            # k*G through the library itself would be circular; use the fixed-base identity with a 1-point MSM on the
            # *reference restatement* (oracle) — checker only
            from oracle import coracle as C
            from oracle import pyoracle as O
            ocv = O.CURVES[args.curve]
            want = ocv.encode_affine([ocv.mul(ocv.G, tot)])[0]
            got = ab.into_affine(cv, res)
            verified = bool((got == want).all())
            del C

    # ---------------- e2e: host buffers through the C ABI, H2D + D2H inside the timed region; measured from pinned host
    # memory (the headline e2e, as the contract asks) and from ordinary pageable memory (what a Rust Vec is): the library
    # stages pageable sources through its pinned ring
    e2e = None
    if not args.no_e2e:
        def timed_host(hb, hs, steps):
            msm_step(hb, hs)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                r = msm_step(hb, hs)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            barrier()
            return max_over_ranks(dt) / steps, r
        e2e_steps = args.steps
        h_bases = torch.empty((n_chunk, 2 * N), dtype=torch.int64).pin_memory()
        h_scal = torch.empty((n_chunk, 4), dtype=torch.int64).pin_memory()
        h_bases.copy_(d_bases[c_lo:c_lo + n_chunk])
        h_scal.copy_(d_scal[c_lo:c_lo + n_chunk])
        dt, r2 = timed_host(h_bases.numpy().view(np.uint64), h_scal.numpy().view(np.uint64), e2e_steps)
        e2e = {"value": 1.0 / dt, "unit": "MSM/s", "ms_per_step": dt * 1e3, "steps": e2e_steps, "host_memory": "pinned",
               "h2d_bytes_per_step": int(n_chunk * (2 * N * 8 + 32)) * world, "d2h_bytes_per_step": 3 * N * 8 * world,
               "sharding": "input chunks x%d (host buffers: each GPU receives 1/%d of the bytes)" % (world, world),
               "same_result": bool((ab.into_affine(cv, r2) == ab.into_affine(cv, res)).all())}
        pb, ps = h_bases.numpy().copy(), h_scal.numpy().copy()       # pageable copies
        del h_bases, h_scal
        dtp, r3 = timed_host(pb.view(np.uint64), ps.view(np.uint64), e2e_steps)
        e2e["pageable"] = {"value": 1.0 / dtp, "unit": "MSM/s", "ms_per_step": dtp * 1e3,
                           "same_result": bool((ab.into_affine(cv, r3) == ab.into_affine(cv, res)).all())}
        del pb, ps

    # ---------------- NTT leg (replicas only for N > 1)
    del d_bases, d_b, d_scal
    torch.cuda.empty_cache()
    if args.no_ntt:
        if rank == 0:
            print(json.dumps({"metric": "msm-only tuning run", "value": 1000.0 / ms_msm, "unit": "MSM/s", "ms_per_step": ms_msm,
                              "phases_ms": phase, "window_c": tm["c"], "windows": tm["windows"], "verified": verified,
                              "e2e": e2e, "clocks": clocks, "gpu_launches": launches}), flush=True)
        write_dump()
        if world > 1:
            dist.destroy_process_group()
        return
    n_ntt = 1 << args.log_n_ntt
    dom = ab.Radix2EvaluationDomain.new(cv.ntt_field_id, n_ntt)
    d_x = torch.empty((n_ntt, 4), dtype=torch.int64, device=dev)
    _lib.check(L.b200_gen_scalars_dev(cv.ntt_field_id, args.seed + 99, n_ntt, d_x.data_ptr(), st))
    x0 = d_x.clone()
    for _ in range(args.warmup):
        dom.fft_in_place(d_x)
    ntt_l0 = L.b200_launch_count()
    ms_ntt, _ = timed(lambda: dom.fft_in_place(d_x), args.steps)
    ntt_launches = int(L.b200_launch_count() - ntt_l0)
    if args.dump_outputs:
        rows = np.random.default_rng(args.seed).choice(n_ntt, size=min(n_ntt, DUMP_NTT_ROWS), replace=False)
        rows = torch.from_numpy(np.sort(rows)).to(dev)
        dump["ntt_fft"] = u64_as_f64(d_x[rows].cpu().numpy().view(np.uint64))
    for _ in range(args.warmup):   # also builds the inverse plan outside the timed region
        dom.ifft_in_place(d_x)
    ms_intt, _ = timed(lambda: dom.ifft_in_place(d_x), args.steps)
    if args.dump_outputs:
        dump["ntt_ifft"] = u64_as_f64(d_x[rows].cpu().numpy().view(np.uint64))
    # round trip property on the timed data: (warmup + steps) forward then as many inverse transforms restore x0
    ntt_ok = bool(torch.equal(d_x, x0))
    ntt_e2e = None
    if not args.no_e2e:
        hx = torch.empty((n_ntt, 4), dtype=torch.int64).pin_memory()
        hx.copy_(x0)
        hxn = hx.numpy().view(np.uint64)
        dom.fft_in_place(hxn)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            dom.fft_in_place(hxn)
        dt = (time.perf_counter() - t0) / args.steps
        ntt_e2e = {"value": world / max_over_ranks(dt), "unit": "NTT/s", "h2d_bytes_per_step": n_ntt * 32 * world,
                   "d2h_bytes_per_step": n_ntt * 32 * world}

    # ---------------- CPU baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
                            "--log-n-msm", str(args.log_n_msm), "--log-n-ntt", str(args.log_n_ntt)], capture_output=True, text=True)
        try:
            ref = json.loads(p.stdout.strip().splitlines()[-1])
            cpu = ref["cpu_baseline"]
            cpu["ntt"] = ref["ntt"]
        except Exception as ex:  # pragma: no cover
            cpu = {"error": f"{ex}: {p.stderr[-300:]}"}

    if rank == 0:
        c, W = tm["c"], tm["windows"]
        # per-rank work: n/N points x W windows either way; a bucket slice also reduces only 1/N of the buckets
        modmuls, wide, byts = msm_work(n_chunk, c, W, 2 * N)
        bshare = (1.0 / world) if shard == "buckets" else 1.0
        wide -= (1.0 - bshare) * 14.0 * (1 << c) * W * (2 * (2 * N) ** 2 + 2 * N)
        acc_s = phase["accumulate"] * 1e-3
        acc_wide = 10.0 * n_chunk * W * (2 * (2 * N) ** 2 + 2 * N)
        # multiplications actually executed: 4 affine levels leave 1/16 of the entries to the XYZZ kernel (10 each), the levels cost
        # 6 + 570/batch (~6.6) per addition; bucket reduction ~28 per bucket; BN254 runs without levels
        lv = 4 if N == 6 else 0
        executed_modmuls = n_chunk * W * ((1 - 0.5 ** lv) * 6.6 + 0.5 ** lv * 10.0) + 28.0 * (1 << (c - 1)) * W * bshare
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp) and world == 1 and args.log_n_msm == 26 and args.curve == 0:
            traffic = json.load(open(tp))
        line = {
            "metric": "BLS12-381 G1 MSM/s @2^%d" % args.log_n_msm if args.curve == 0 else "BN254 G1 MSM/s @2^%d" % args.log_n_msm,
            "value": 1000.0 / ms_msm, "unit": "MSM/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_msm, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32 limbs (Montgomery; 12x32-bit Fq, 8x32-bit Fr)", "data": "synthetic",
            "config": {"workload": f"{cv.name} VariableBaseMSM n=2^{args.log_n_msm}, bases b_i*G generated on device, uniform scalars; "
                                   f"NTT leg: Fr radix-2 fft n=2^{args.log_n_ntt}",
                       "window_c": c, "windows": W, "sharding": (f"bucket slices x{world} over inputs replicated in every GPU's HBM" if shard == "buckets"
                                    else f"input chunks x{world}") + ", NCCL all-gather of partial points",
                       "l2": "inputs (>= 2 GiB) larger than L2; no flush needed", "seed": args.seed, "verified_vs_sum_identity": verified},
            "clocks": clocks,
            "phases_ms": phase,
            # MSM is bound by the integer-multiply pipe (SURVEY.md §8d), so the roofline block is the IMAD one: algorithmic wide MADs of
            # the WHOLE step (10*n*W + 14*2^c*W Fq multiplications x 300) over the step time, against the measured IMAD.WIDE issue rate
            "roofline": {"bound": "imad", "kernel": "whole MSM step (dominant kernel: msm_pair_add*_kernel, batched-affine levels)",
                         "achieved": wide / (ms_msm * 1e-3) / 1e12, "peak": IMAD_PEAK_WIDE_PER_S / 1e12, "unit": "T wide-MAD/s",
                         "frac": wide / (ms_msm * 1e-3) / IMAD_PEAK_WIDE_PER_S,
                         "frac_accumulation_phase": (acc_wide / acc_s) / IMAD_PEAK_WIDE_PER_S if acc_s else None,
                         "frac_executed": (executed_modmuls * 300.0 if N == 6 else executed_modmuls * 136.0) / (ms_msm * 1e-3) / IMAD_PEAK_WIDE_PER_S,
                         "traffic": traffic.get("msm_dominant_kernel_dram_bytes_per_launch"),
                         "traffic_whole_step": traffic.get("msm_step_dram_bytes"),
                         "algorithmic_bytes": byts,
                         "peak_source": IMAD_PEAK_SOURCE,
                         "note": "frac = the reference's 10-multiplication XYZZ formula per bucket addition; frac_executed = multiplications "
                                 "actually issued (batched-affine additions cost ~6.6 each); traffic = dram read+write bytes from the ncu "
                                 "capture of this command committed as profiles/r02_traffic.json"},
            "hbm_roofline": {"bound": "hbm", "achieved": byts / (ms_msm * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": byts / (ms_msm * 1e-3) / 1e9 / hbm_peak, "peak_source": peak_src},
            "gpu_launches": launches,
            "e2e": e2e,
            "cpu_baseline": cpu,
            "ntt": {"metric": "BLS12-381 Fr NTT/s @2^%d" % args.log_n_ntt, "value": world * 1000.0 / ms_ntt, "unit": "NTT/s",
                    "ms_per_step": ms_ntt, "ifft_ms_per_step": ms_intt, "scaling": "replicas only", "gpu_launches": ntt_launches,
                    "roundtrip_ok": ntt_ok, "e2e": ntt_e2e,
                    "roofline": {"bound": "hbm", "achieved": 64.0 * n_ntt / (ms_ntt * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": 64.0 * n_ntt / (ms_ntt * 1e-3) / 1e9 / hbm_peak,
                                 "traffic": traffic.get("ntt_dram_bytes_per_transform") if args.log_n_ntt == 24 else None, "peak_source": peak_src,
                                 "note": "contractual HBM figure; the transform is bound by the integer pipe (imad_roofline)"},
                    "imad_roofline": {"achieved": 136.0 * (n_ntt / 2 * args.log_n_ntt) / (ms_ntt * 1e-3) / 1e12,
                                      "peak": IMAD_PEAK_WIDE_PER_S / 1e12, "unit": "T wide-MAD/s",
                                      "frac": 136.0 * (n_ntt / 2 * args.log_n_ntt) / (ms_ntt * 1e-3) / IMAD_PEAK_WIDE_PER_S}},
        }
        print(json.dumps(line), flush=True)
    write_dump()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
