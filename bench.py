#!/usr/bin/env python
"""bench.py -- the find_arb! dual-gradient sweep on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
  python bench.py --gpus 1 --steps K --dump-outputs DIR    # + [Ψ; acc] of the last timed step as .npy

Every timed region runs exactly K steps (the e2e region too, unless --e2e-steps says otherwise).
The inputs are drawn from fixed seeds, so two runs with the same arguments sweep the same pools
at the same ν.  The outputs agree to summation-order noise, not bit for bit: the kernel sizes
each CTA's pool range from measured CTA speed (option `balance`), so the fp64 parts of the sums
(acc, pools outside the fixed-point slice) are added in a timing-dependent order; on a B200,
two runs of the default workload differed by at most 2e-12 relative in Ψ.  The run writes
nothing into the source tree.

A "step" is ONE dual-gradient sweep: find_arb! over every pool at the current
ν plus the Ψ / acc folds (src/router.jl:38-42, 79-83, 98-100) -- exactly what
one L-BFGS-B function/gradient evaluation of route! costs on the pool side.

Workload (config.workload): BASELINE.json configs[4] -- 10M ProductTwoCoin
pools, 50k tokens -- per GPU.  It is the configuration the metric's target is
quoted on (">= 10M find_arb! evaluations per sweep"), it fits one GPU, and at
320 MB it is larger than the 126 MB L2, so every timed sweep streams from HBM
without an explicit flush.  For N > 1 each rank owns its own 10M-pool shard
(weak scaling) and the only exchange is the sum of [Ψ; acc] over NVLink peer
memory after each sweep; `--scaling strong` splits the same 10M pools instead.

Prints ONE JSON line (rank 0).  `value` = pools evaluated per second with ν and
Ψ resident in HBM (CUDA events, max over ranks); `e2e` = the same through the
public C-ABI call cfmm_sweep() with pinned HOST buffers (H2D ν and D2H Ψ inside
the timed region).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ from the imports below

METRIC = "find_arb_pools_per_sec_per_dual_gradient_sweep"
UNIT = "pools/s"

WORKLOADS = {
    # name: (pools per GPU, n_tokens, kind)
    "config5_10M_product_50k_tokens": (10_000_000, 50_000, "product"),
    "config2_100k_product_1k_tokens": (100_000, 1_000, "product"),
    "config3_1M_mixed_10k_tokens": (1_000_000, 10_000, "mixed"),
    "config4_500k_univ3_5k_tokens": (500_000, 5_000, "univ3"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default="config5_10M_product_50k_tokens", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak")
    ap.add_argument("--exchange", choices=["peer", "nccl"], default="peer")
    ap.add_argument("--protocol", type=int, default=0,
                    help="peer exchange protocol: 0 = library default (direct 8-byte push up to 4 ranks, LL "
                         "two-shot beyond), 1 = LL one-shot, 2 = LL two-shot, 3 = direct")
    ap.add_argument("--nu", choices=["near", "wide", "ones"], default="near")
    ap.add_argument("--exact", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = same as --steps")
    ap.add_argument("--sustained-ms", type=float, default=0.0,
                    help="when the K timed steps take less than this many ms, also time a longer region of the "
                         "same steps (`sustained`, clocks sampled under load); 0 = off, so that only K steps "
                         "are timed per region")
    ap.add_argument("--no-flush", action="store_true", help="small workloads: L2-warm timing only")
    ap.add_argument("--verify", type=int, default=1, help="N > 1: check the reduced [Psi; acc] (outside the timed regions)")
    ap.add_argument("--opt", action="append", default=[], help="library option key=value (measurement)")
    ap.add_argument("--strong", type=int, default=1, help="N > 1 (weak): also time the same total pool count split over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed, the float64 arrays a caller of the sweep "
                         "receives, to DIR/psi.npy and DIR/acc.npy (inputs are seeded: two builds can be "
                         "compared output for output, within summation-order noise)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the reference arm times a machine-dependent sample)")
    return args


def make_shard(workload, rank, world, scaling):
    from cfmmrouter_b200 import synth
    m, n, kind = WORKLOADS[workload]
    if scaling == "strong":
        lo, hi = (m * rank) // world, (m * (rank + 1)) // world
    else:
        lo, hi = 0, m
    seed = 1234 + (rank if scaling == "weak" else 0)
    out = {"n": n, "kind": kind, "m_local": hi - lo}
    if kind == "product":
        R, g, Ai = synth.product_pools(m, n, seed=seed)
        out["product"] = (R[lo:hi], g[lo:hi], Ai[lo:hi])
        out["bytes"] = (hi - lo) * 32
    elif kind == "mixed":
        h = m // 2
        R, g, Ai = synth.product_pools(h, n, seed=seed)
        Rg, gg, Ag, wg = synth.geomean_pools(h, n, seed=seed + 1)
        l2, h2 = lo // 2, hi // 2
        out["product"] = (R[l2:h2], g[l2:h2], Ai[l2:h2])
        out["geomean"] = (Rg[l2:h2], gg[l2:h2], Ag[l2:h2], wg[l2:h2])
        out["m_local"] = 2 * (h2 - l2)
        out["bytes"] = (h2 - l2) * (32 + 48)
    else:
        cp, g, Ai, off, lt, lq = synth.univ3_pools(m, n, seed=seed)
        sl = slice(lo, hi)
        out["univ3"] = (cp[sl], g[sl], Ai[sl], off[lo:hi + 1] - off[lo], lt[off[lo]:off[hi]], lq[off[lo]:off[hi]])
        out["bytes"] = (hi - lo) * 32 + (off[hi] - off[lo]) * 16
    return out


# ---------------------------------------------------------------------------
# clocks: sampled DURING the timed region (NVML, falls back to nvidia-smi)
# ---------------------------------------------------------------------------

class ClockSampler:
    def __init__(self, device_index):
        self.idx = device_index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self._nvml = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    _BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
             0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def _loop(self):
        n = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
                try:
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self._BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def _sample_once(self):
        n = self._nvml
        try:
            self.samples.append(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
            try:
                r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
            except Exception:
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for bit, name in self._BITS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def start(self):
        if self._nvml:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._sample_once()  # at least one sample taken while the last steps are in flight
            self._stop.set()
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle "faithful" port)
# ---------------------------------------------------------------------------

def cpu_faithful_rate(workload, sample_pools, sweeps, threads):
    """pools/s of the faithful-layout CPU restatement (oracle/) on a sample of
    the workload: threaded sweep + serial acc / scatter folds, like
    src/router.jl:38-42, 79-83, 98-100."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from cfmmrouter_b200 import synth
    o = oracle_lib.load()
    m, n, kind = WORKLOADS[workload]
    sample_pools = int(min(sample_pools, m))
    f = o.faithful(n)
    if kind in ("product", "univ3"):  # (univ3 has no faithful flavour: product stands in)
        R, g, Ai = synth.product_pools(sample_pools, n)
        f.add_product(R, g, Ai)
    else:
        R, g, Ai = synth.product_pools(sample_pools // 2, n)
        Rg, gg, Ag, wg = synth.geomean_pools(sample_pools // 2, n)
        f.add_product(R, g, Ai)
        f.add_geomean(Rg, gg, Ag, wg)
    v = synth.dual_prices(n, "near")
    f.sweep(v, threads)  # warm
    t0 = time.perf_counter()
    for _ in range(sweeps):
        f.sweep(v, threads)
    dt = time.perf_counter() - t0
    f.close()
    return sample_pools * sweeps / dt, dt / sweeps, sample_pools


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    o = oracle_lib.load()
    threads = o.max_threads()
    m, n, kind = WORKLOADS[args.workload]
    # bound the whole run to ~2 minutes of CPU time: pools per step from a probe
    # all host threads, unless half of them (one per physical core) is faster on this box
    probe_rate, _, _ = cpu_faithful_rate(args.workload, 200_000, 2, threads)
    if threads >= 4:
        half_rate, _, _ = cpu_faithful_rate(args.workload, 200_000, 2, threads // 2)
        if half_rate > probe_rate:
            threads, probe_rate = threads // 2, half_rate
    # the whole workload per step when the run still ends within ~3 minutes, else a bounded sample
    budget = 180.0 / max(1, args.steps + args.warmup)
    sample = int(max(10_000, min(m, probe_rate * budget)))
    from cfmmrouter_b200 import synth
    f = o.faithful(n)
    R, g, Ai = synth.product_pools(sample, n)
    f.add_product(R, g, Ai)
    v = synth.dual_prices(n, "near")
    for _ in range(args.warmup):
        f.sweep(v, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        f.sweep(v, threads)
    dt = time.perf_counter() - t0
    f.close()
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "pools_per_step_sample": sample, "pools_total": m,
                   "sample_is_whole_workload": sample == m, "n_tokens": n,
                   "note": "reference = CFMMRouter.jl's CPU algorithm; Julia is not installed, so this is "
                           "the oracle's faithful-layout C restatement (threaded sweep, serial folds)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} ProductTwoCoin pools of the workload per step, "
                                   f"{args.steps} steps, {threads} OpenMP threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    import cfmmrouter_b200 as cr

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    shard = make_shard(args.workload, rank, world, args.scaling)
    n = shard["n"]
    pools = cr.DevicePools(n, device=local_rank)
    t_ing0 = time.perf_counter()
    if "product" in shard:
        pools.add_product(*shard["product"])
    if "geomean" in shard:
        pools.add_geomean(*shard["geomean"])
    if "univ3" in shard:
        pools.add_univ3(*shard["univ3"])
    t_ing1 = time.perf_counter()
    pools.finalize()  # validate-free part: orientation, (bucket(b), a) sort, SoA gather, upload, scale table
    t_ing2 = time.perf_counter()
    ingest = {"pools": shard["m_local"], "add_s": t_ing1 - t_ing0, "finalize_s": t_ing2 - t_ing1,
              "host_threads": os.cpu_count(),
              "note": "cfmm_add_* (validation + staging copy) and cfmm_finalize (layout on the host cores with "
                      "OpenMP, upload, device-side scale table) wall time on this rank"}
    pools.set_option("exact", args.exact)
    pools.set_option("sweep_events", 0)
    for kv in args.opt:
        pools.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    m_local = shard["m_local"]
    alg_bytes = float(shard["bytes"])
    # working sets that fit in the 126 MB L2 are timed with an L2 flush before every step
    # (value, roofline) AND warm (reported beside it); larger ones stream from HBM anyway
    flushed = alg_bytes <= 126e6 and not args.no_flush
    if not (world > 1 and args.verify):
        shard = None

    exchange = "none"
    if world > 1:
        exchange = args.exchange
        if exchange == "peer":
            try:
                pools.attach_group(dist.group.WORLD)
            except cr.CFMMError as e:
                if rank == 0:
                    print(f"[bench] peer exchange unavailable ({e}); using NCCL", file=sys.stderr)
                exchange = "nccl"
            if exchange == "peer" and args.protocol > 0:
                pools.set_option("exchange_protocol", args.protocol)
            flag = torch.tensor([1 if exchange == "peer" else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() == 0 and exchange == "peer":
                exchange = "nccl"

    from cfmmrouter_b200 import synth
    nu_host = synth.dual_prices(n, args.nu)
    d_nu = torch.from_numpy(nu_host).to(dev)
    d_psi = torch.zeros(n + 1, dtype=torch.float64, device=dev)
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flushed else None
    flush_rd = torch.zeros(32 << 20, dtype=torch.int64, device=dev) if flushed else None

    def flush_l2():
        """Write 256 MB (> L2), then READ another 256 MB: the write alone would leave ~126 MB of dirty
        lines whose write-back the next (timed) kernel pays for; after the read pass the L2 holds
        clean lines of an unrelated buffer.  Both passes are outside the timed intervals."""
        flush_buf.zero_()
        flush_rd.sum()

    last_out = [d_psi.data_ptr()]  # device address of the [Ψ; acc] the last step wrote

    def make_step(p):
        def step():
            if exchange == "nccl":  # NCCL needs the partial in a torch tensor
                p.sweep_device(d_nu.data_ptr(), d_psi.data_ptr(), False, sptr)
                dist.all_reduce(d_psi)
            else:  # zero-copy: [Ψ; acc] stays in the context's device buffer
                last_out[0] = p.sweep_device_view(d_nu.data_ptr(), False, sptr)
        return step

    step = make_step(pools)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler_ref = [None]
    host_enqueue_us = [0.0]

    def timed_region(steps, fn=None, flush=False):
        """ms of `steps` steps on the stream (CUDA events, barrier + synchronize on both sides).
        flush: write a 256 MB buffer (> L2) before every step and time each step with its own
        event pair, so the flush itself is outside the timed intervals."""
        fn = fn or step
        barrier()
        if flush:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for a, b in ev:
                flush_l2()
                a.record(stream)
                fn()
                b.record(stream)
            if sampler_ref[0] is not None:
                sampler_ref[0]._sample_once()
            barrier()
            pools.comm_check()
            return float(sum(a.elapsed_time(b) for a, b in ev))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        th0 = time.perf_counter()
        for _ in range(steps):
            fn()
        host_enqueue_us[0] = 1e6 * (time.perf_counter() - th0) / max(steps, 1)  # host time to ENQUEUE a step
        e1.record(stream)
        if sampler_ref[0] is not None:
            sampler_ref[0]._sample_once()  # GPU still busy with the queued steps
        barrier()
        pools.comm_check()  # a timed-out exchange must fail the run, not slow it
        return e0.elapsed_time(e1)

    def spin_up(min_ms=20.0):
        """Untimed sweeps until the GPU has been busy for min_ms: after an idle period (setup, a
        host-side pause between regions) the first ~20 launches run 2-4 us slower than the steady
        state (tools/ramp_probe.py: 59.9 -> 57.8 -> 55.9 us over launches 0-5 / 5-20 / 20+); a short
        synchronize does not bring that back.  Called right before every timed region's barrier."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        done = 0
        while True:
            for _ in range(64):
                step()
            done += 64
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:  # every rank must run the same number of sweeps: they exchange
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                ms = t.item()
            if ms >= min_ms or done >= 50_000:
                return done

    extra = {}
    with torch.cuda.stream(stream):
        for _ in range(max(3, args.warmup)):
            step()
        extra["spin_up"] = {"min_ms": 20.0, "steps": spin_up(),
                            "note": "untimed sweeps after the W warm-up steps and before each timed region, until "
                                    "the GPU has been busy 20 ms (clock / launch pipeline ramp after idle)"}
        barrier()
        # ---- timed region 1: K steps, nothing but the sweeps on the stream -> `value`
        l0 = pools.launch_count
        sampler = ClockSampler(local_rank)
        sampler_ref[0] = sampler if sampler._nvml else None
        sampler.start()
        ms_total = timed_region(args.steps, flush=flushed)
        launches = pools.launch_count - l0
        # the result of the last timed step, before any later sweep overwrites the context's buffer
        outputs = _view(torch, last_out[0], n + 1, dev).clone() if args.dump_outputs and rank == 0 else None
        extra["host_enqueue_us_per_step"] = host_enqueue_us[0]
        # a small K can be a millisecond of GPU time: on request, also a region of at least
        # --sustained-ms of the same steps (`sustained`), so that the clocks are sampled under load
        ms_dec = ms_total
        if world > 1:  # every rank must take the same branch and launch the same number of sweeps
            t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_dec = t.item()
        if ms_dec < args.sustained_ms and not flushed:
            k2 = int(min(50_000, max(args.steps, np.ceil(1.2 * args.sustained_ms * args.steps / max(ms_dec, 1e-3)))))
            ms2 = timed_region(k2)
            extra["sustained"] = {"steps": k2, "ms_per_step": ms2 / k2}
        sampler.stop()
        sampler_ref[0] = None
        if flushed:
            ms_warm = timed_region(args.steps)
            extra["l2_warm"] = {"steps": args.steps, "ms_per_step": ms_warm / args.steps}
        # ---- timed region 2: the same K steps with a CUDA-event pair around every
        # kernel launch (on the launching stream) -> per-kernel durations for `roofline`
        n_kernels = 2 if args.workload.startswith("config3") else 1
        spin_up()
        pools.set_option("profile", args.steps * (n_kernels + (1 if exchange == "peer" else 0)))
        timed_region(args.steps, flush=flushed)
        prof = {t: pools.profile_read(t) for t in (0, 1, 2, 3)}
        prof_times = {t: pools.profile_times(t) for t in (0, 1, 2)}
        pools.set_option("profile", 0)

        # ---- e2e: public C-ABI call with pinned host buffers, copies inside ----
        e2e_steps = args.e2e_steps or args.steps
        h_nu = torch.from_numpy(nu_host).pin_memory()
        h_out = torch.zeros(n + 1, dtype=torch.float64).pin_memory()  # [psi ; acc] contiguous
        h_psi, h_acc = h_out[:n], h_out[n:]
        for _ in range(3):
            pools.sweep_into(h_nu.data_ptr(), h_psi.data_ptr(), h_acc.data_ptr())
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            pools.sweep_into(h_nu.data_ptr(), h_psi.data_ptr(), h_acc.data_ptr())
            if exchange == "nccl":  # host-visible result must be the global sum
                t = torch.cat([h_psi, h_acc]).to(dev)
                dist.all_reduce(t)
                t.cpu()
        barrier()
        e2e_s = time.perf_counter() - t0

        # ---- per-phase timeline of the fused sweep+exchange kernel on rank 0 (%globaltimer stamps of
        # every CTA; measurement option "trace", outside the timed regions) ---------------------
        if world > 1 and exchange == "peer" and WORKLOADS[args.workload][2] == "product":
            extra["phases_rank0_us"] = phase_trace(pools, step, barrier, rank, dist=dist, world=world)
        # ---- N > 1, outside every timed region: is the reduced [Ψ; acc] right? --------------
        if world > 1 and args.verify and exchange == "peer":
            extra["parity_checked"], extra["parity"] = verify_reduction(
                torch, dist, pools, shard, nu_host, d_nu, sptr, n, dev, rank, world)
            shard = None
        # ---- N > 1: the same TOTAL pool count split over the ranks (BASELINE configs[4] as
        # written: "10M pools pool-sharded across 8 GPUs") next to the weak-scaling value ------
        if world > 1 and args.scaling == "weak" and args.strong and exchange == "peer" \
                and WORKLOADS[args.workload][2] == "product":
            extra["strong"] = strong_scaling_run(torch, dist, cr, args, pools, make_step, timed_region, barrier,
                                                 rank, world, local_rank, dev, host_enqueue_us)

    # max over ranks
    if world > 1:
        t = torch.tensor([ms_total, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s = t[0].item(), t[1].item()
    total_pools = m_local * world if args.scaling == "weak" else WORKLOADS[args.workload][0]
    if args.scaling == "weak" and world > 1:
        tp = torch.tensor([m_local], dtype=torch.float64, device=dev)
        dist.all_reduce(tp)
        total_pools = int(tp.item())
    value = total_pools * args.steps / (ms_total * 1e-3)
    e2e_value = total_pools * e2e_steps / e2e_s
    for key in ("sustained", "l2_warm"):
        if key in extra:
            t = torch.tensor([extra[key]["ms_per_step"]], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extra[key]["ms_per_step"] = t.item()
            extra[key]["value"] = total_pools / (t.item() * 1e-3)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            with open(peaks_path) as f:
                peak, peak_src = float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        kind = WORKLOADS[args.workload][2]
        roofline = roofline_object(prof, prof_times, ms_total, args.steps, launches, kind, m_local,
                                   alg_bytes, peak, peak_src, args.workload, flushed,
                                   geomean_tma=not any(o.replace(" ", "") in ("geomean_tma=0", "use_tma=0", "geomean_log2=0")
                                                       for o in args.opt))
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib
            threads = oracle_lib.load().max_threads()
            rate, per_sweep, sample = cpu_faithful_rate(args.workload, 2_000_000, 3, threads)
            rate1, _, sample1 = cpu_faithful_rate(args.workload, 500_000, 2, 1)
            cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{sample} pools of the workload x 3 sweeps, faithful-layout C restatement of "
                             f"router.jl:38-42,79-83,98-100 (Julia unavailable), {threads} OpenMP threads; "
                             f"1 thread (Julia's default): {rate1:.3g} pools/s on {sample1} pools"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "pools_per_gpu": m_local, "pools_total": total_pools,
                       "n_tokens": n, "nu": args.nu, "exact_mode": args.exact, "exchange": exchange,
                       "exchange_protocol": (None if exchange != "peer" else
                                             {0: "direct 8-byte push (1 hop)" if world <= 4 else "LL two-shot",
                                              3: "direct 8-byte push (1 hop)",
                                              1: "LL one-shot", 2: "LL two-shot"}[args.protocol]),
                       "l2": "inputs larger than L2 (320 MB algorithmic, 240-320 MB streamed per launch per GPU > 126 MB)" if alg_bytes > 126e6
                             else ("L2 flushed (256 MB written, then 256 MB read so that no dirty lines remain) before every timed step; the warm figure is in l2_warm"
                                   if flushed else "L2-WARM: working set fits in L2, no flush between steps")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 8 * n,
                    "d2h_bytes_per_step": 8 * (n + 1), "steps": e2e_steps,
                    "ms_per_step": 1e3 * e2e_s / e2e_steps, "api": "cfmm_sweep (C ABI), pinned host buffers"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        line["ingest"] = ingest
        line.update(extra)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs.cpu().numpy(), n)
        emit(line)
    pools.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, psi_acc, n):
    """[Ψ; acc] of one sweep (float64, n_tokens + 1: at most 400 KB for the workloads above) as
    DIR/psi.npy [n_tokens] and DIR/acc.npy [1]."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "psi.npy"), np.ascontiguousarray(psi_acc[:n], dtype=np.float64))
    np.save(os.path.join(out_dir, "acc.npy"), np.ascontiguousarray(psi_acc[n:], dtype=np.float64))


def _view(torch, ptr, count, dev):
    class _H:
        pass
    h = _H()
    h.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(h, device=dev)


def phase_trace(pools, step, barrier, rank, dist=None, world=1):
    """Median over 8 sweeps of the kernel's phases on this rank, from the per-CTA %globaltimer stamps:
    chunk loop done (slowest CTA), partials flushed, grid barrier passed, exit (exchange done)."""
    pools.set_option("trace", 1)
    rows = []
    for _ in range(8):
        barrier()
        step()
        barrier()
        grid = ctypes.c_int64()
        pools._lib.cfmm_debug_read_trace(pools._ctx, None, 0, ctypes.byref(grid))
        buf = np.zeros(max(int(grid.value), 1) * 8, dtype=np.uint64)
        rc = pools._lib.cfmm_debug_read_trace(pools._ctx, buf.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                              grid.value, ctypes.byref(grid))
        if rc != 0 or grid.value == 0:
            break
        t = buf.reshape(-1, 8).astype(np.int64)
        t0 = t[:, 0].min()
        rel = lambda col: (t[:, col] - t0) / 1e3
        rows.append({"slice_ready_med": float(np.median(rel(1))), "chunk_loop_done_med": float(np.median(rel(3))),
                     "chunk_loop_done_max": float(rel(3).max()), "flushed_max": float(rel(4).max()),
                     "grid_barrier_passed_med": float(np.median(rel(6))) if t[:, 6].any() else None,
                     "exit_max": float(rel(5).max())})
    pools.set_option("trace", 0)
    mine = None
    if rows:
        mine = {k: (float(np.median([r[k] for r in rows])) if rows[0][k] is not None else None) for k in rows[0]}
    if dist is not None and world > 1:
        # every rank's own timeline (each relative to its own first CTA): who waits for whom
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        if mine is not None:
            mine["by_rank"] = [None if r is None else {"flushed_max": r["flushed_max"],
                                                        "grid_barrier_passed_med": r["grid_barrier_passed_med"],
                                                        "exit_max": r["exit_max"]} for r in allr]
    return mine if rank == 0 else None


def verify_reduction(torch, dist, pools, shard, nu_host, d_nu, sptr, n, dev, rank, world):
    """(1) every rank's partial [Ψ; acc] (option exchange_bypass) against the CPU oracle on that
    rank's own pools; (2) the peer-exchanged vector == the sum of the partials (NCCL all_reduce
    of the same partials) within summation-order noise; (3) the exchanged vector is bitwise
    identical on every rank."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    o = oracle_lib.load()
    res = {}
    ptr = pools.sweep_device_view(d_nu.data_ptr(), False, sptr)
    torch.cuda.synchronize()
    reduced = _view(torch, ptr, n + 1, dev).clone()
    pools.set_option("exchange_bypass", 1)
    ptr = pools.sweep_device_view(d_nu.data_ptr(), False, sptr)
    torch.cuda.synchronize()
    partial = _view(torch, ptr, n + 1, dev).clone()
    pools.set_option("exchange_bypass", 0)
    dist.barrier()
    # (1) partial vs oracle on this rank's pools (ProductTwoCoin shards; mixed/univ3: skipped)
    ok1 = True
    if shard is not None and "product" in shard and "geomean" not in shard:
        R, g, Ai = shard["product"]
        threads = max(1, (os.cpu_count() or 1) // world)
        D, L = o.sweep_product(R, g, Ai, nu_host, threads=threads)
        accx, Gx, absG = o.fold_compensated(Ai, D, L, nu_host, n)
        eps = np.finfo(np.float64).eps
        slack, S, deg = np.zeros(n), np.zeros(n), np.zeros(n)
        for side in (0, 1):
            np.add.at(slack, Ai[:, side] - 1, 32 * eps * (R[:, 0] + R[:, 1]) / g)  # economized math
            np.add.at(S, Ai[:, side] - 1, R[:, side])
            np.add.at(deg, Ai[:, side] - 1, 1.0)
        slack += deg * S * 2.0 ** -53  # fixed-point slice quantum
        h = partial.cpu().numpy()
        err = np.abs(h[:n] - Gx.astype(np.float64))
        ok1 = bool(np.all(err <= 1e-12 * absG + slack))
        ok1 &= abs(h[n] - float(accx)) <= 1e-12 * float(np.sum(absG * nu_host)) + float(np.sum(slack * nu_host))
        res["partial_vs_oracle_max_err_over_tol"] = float(np.max(err / (1e-12 * absG + slack + 1e-300)))
    # (2) exchanged vector vs NCCL sum of the partials
    total = partial.clone()
    dist.all_reduce(total)
    mag = partial.abs()
    dist.all_reduce(mag)
    diff = (reduced - total).abs()
    ok2 = bool(torch.all(diff <= 1e-13 * mag + 1e-300).item())
    res["exchange_vs_nccl_max_rel"] = float((diff / (mag + 1e-300)).max().item())
    # (3) bitwise identical on every rank
    bits = reduced.view(torch.int64)
    lo, hi = bits.clone(), bits.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    ok3 = bool(torch.equal(lo, hi))
    flag = torch.tensor([1 if (ok1 and ok2 and ok3) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res.update({"partial_vs_oracle": ok1, "exchange_equals_sum": ok2, "bitwise_identical_across_ranks": ok3})
    return bool(flag.item() == 1), res


def strong_scaling_run(torch, dist, cr, args, pools_weak, make_step, timed_region, barrier, rank, world,
                       local_rank, dev, host_enqueue_us=None):
    """The workload's pool count split over the ranks (strong scaling), timed like `value`, plus
    the single-GPU time of the same pools (rank 0's weak shard IS that pool set, swept with the
    exchange bypassed) so that the line carries its own speed-up."""
    from cfmmrouter_b200 import synth
    m, n, _ = WORKLOADS[args.workload]
    lo, hi = (m * rank) // world, (m * (rank + 1)) // world
    R, g, Ai = synth.product_pools(m, n, seed=1234)
    ps = cr.DevicePools(n, device=local_rank)
    ps.add_product(R[lo:hi], g[lo:hi], Ai[lo:hi])
    del R, g, Ai
    ps.finalize()
    ps.set_option("sweep_events", 0)
    ps.attach_group(dist.group.WORLD)
    if args.protocol > 0:
        ps.set_option("exchange_protocol", args.protocol)
    fn = make_step(ps)
    steps = args.steps
    for _ in range(10):
        fn()
    ms = timed_region(steps, fn)
    host_us = host_enqueue_us[0] if host_enqueue_us is not None else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    phases = phase_trace(ps, fn, barrier, rank, dist=dist, world=world)  # per-phase timeline of the strong step
    # the same shards without the exchange (and without its grid barrier): kernel + launch per rank
    ps.set_option("exchange_bypass", 1)
    for _ in range(5):
        fn()
    msb = timed_region(steps, fn)
    ps.set_option("exchange_bypass", 0)
    tb = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(tb, torch.tensor([1e3 * msb / steps], dtype=torch.float64, device=dev))
    bypass_us = [float(x.item()) for x in tb]
    # single GPU, same 10M pools: every rank sweeps its weak shard without the exchange; rank 0's is seed 1234
    pools_weak.set_option("exchange_bypass", 1)
    fn1 = make_step(pools_weak)
    for _ in range(5):
        fn1()
    ms1 = timed_region(steps, fn1)
    pools_weak.set_option("exchange_bypass", 0)
    t1 = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(t1, torch.tensor([ms1], dtype=torch.float64, device=dev))
    weak_alone_us = [1e3 * float(x.item()) / steps for x in t1]  # GPU-to-GPU spread of the same kernel
    ms1 = float(t1[0].item())
    barrier()
    ps.close()
    return {"pools_total": m, "pools_per_gpu": hi - lo, "steps": steps, "us_per_step": 1e3 * ms / steps,
            "value": m * steps / (ms * 1e-3), "unit": UNIT,
            "single_gpu_us_per_step": 1e3 * ms1 / steps, "speedup_vs_single_gpu": ms1 / ms,
            "phases_rank0_us": phases, "host_enqueue_us_per_step": host_us,
            "no_exchange_us_per_step_by_rank": bypass_us,
            "weak_shard_alone_us_per_step_by_rank": weak_alone_us,
            "note": "same total pools split over the ranks (BASELINE configs[4] as written); single_gpu = "
                    "rank 0 sweeping all of them alone, in the same run"}


def roofline_object(prof, prof_times, ms_total, steps, launches, kind, m_local, alg_bytes, peak, peak_src,
                    workload, flushed, geomean_tma=True):
    """The `roofline` object of the JSON line, from the event-bracketed launches of timed
    region 2.  prof[t] = (total_ms, launches) and prof_times[t] = per-launch ms for pool type
    t (3 = peer exchange); ms_total / launches belong to timed region 1 (no events between
    launches)."""
    # dominant kernel = the one with the most event-timed device time
    dom = max((0, 1, 2), key=lambda t: prof[t][0])
    dom_ms, dom_cnt = prof[dom]
    dom_name = {0: "product_sweep_tma<ProductTwoCoin> (gradient sweep, TMA ring kernel)",
                1: "product_sweep_tma<GeometricMeanTwoCoin> (gradient sweep, TMA ring kernel, 48-byte records)"
                   if geomean_tma else "sweep_kernel<GeomeanPools>",
                2: "sweep_kernel<Univ3Pools>"}[dom]
    traffic = read_traffic(workload, {0: "product_sweep_tma", 1: "product_sweep_tma_geomean" if geomean_tma
                                      else "sweep_kernel_geomean", 2: "sweep_kernel_univ3"}[dom])
    if kind == "mixed":
        dom_bytes = (m_local // 2) * (32 if dom == 0 else 48)
    else:
        dom_bytes = alg_bytes
    achieved = dom_bytes / (dom_ms / max(dom_cnt, 1) * 1e-3) / 1e9 if dom_cnt else None
    roofline = {
        "bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": (achieved / peak) if achieved else None, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": dom_bytes, "avg_launch_us": 1e3 * dom_ms / max(dom_cnt, 1),
        "launches_timed": dom_cnt, "traffic": traffic,
        "l2_state": "flushed before every timed launch" if flushed else "inputs larger than L2",
    }
    if len(prof_times[dom]):
        # spread of the individual event-bracketed launches: `avg_launch_us` is their mean
        # (what `achieved` uses); a bracket also holds the stream's event/launch front-end
        # latency, which differs between hosts, so the quantiles are reported beside it
        us = 1e3 * np.sort(np.asarray(prof_times[dom], dtype=np.float64))
        roofline["launch_us"] = {"mean": float(us.mean()), "min": float(us[0]),
                                 "p05": float(us[int(0.05 * (len(us) - 1))]),
                                 "median": float(us[(len(us) - 1) // 2]),
                                 "p95": float(us[int(0.95 * (len(us) - 1))]), "max": float(us[-1])}
    if dom_cnt and launches == steps and ms_total > 0:
        # one launch per step and nothing else on the stream: timed region 1 is the same
        # kernel back to back.  Consecutive launches of the persistent kernel overlap their
        # ramp and tail, so this is shorter than a bracketed (serialised) launch; reported
        # beside `frac`, not instead of it.
        step_us = 1e3 * ms_total / steps
        b2b = dom_bytes / (step_us * 1e-6) / 1e9
        roofline["back_to_back"] = {"launch_us": step_us, "achieved": b2b, "frac": b2b / peak}
    if prof[3][1]:
        roofline["exchange_avg_us"] = 1e3 * prof[3][0] / prof[3][1]
    return roofline



def read_traffic(workload, kernel_key):
    """dram bytes (read+write) per launch of the dominant kernel from the committed
    ncu --set full capture (profiles/traffic.json) -- only when that capture was taken on THIS
    workload and kernel; otherwise null (a constant from another run is not a measurement)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                for entry in json.load(f).get("captures", []):
                    if entry.get("workload") == workload and entry.get("kernel_key") == kernel_key:
                        return entry.get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line, on the real stdout (libraries such as NCCL print
    banners to fd 1; everything else this process writes goes to stderr)."""
    def plain(o):  # numpy scalars that reach the line through the parity / phase objects
        if isinstance(o, np.generic):
            return o.item()
        raise TypeError(f"not JSON serialisable: {type(o).__name__}")
    data = (json.dumps(line, default=plain) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
