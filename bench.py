#!/usr/bin/env python
"""bench.py — tagged send/recv throughput of starway_b200 (driver contract: see the task brief).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, sm_100a)
  python bench.py --impl reference --gpus N ...            reference arm: the reference's CPU path
                                                           (restated, oracle/cpu_engine.cpp) on host cores
  python bench.py ... --dump-outputs DIR                   also write what the last timed step received (.npy)
Every line also carries `sweep`: BASELINE config 3 sampled at 64 B ... 1 GiB in the same run (--no-sweep skips it;
the full 25-size sweep, uni- and bidirectional, is `bench_scenarios.py sweep`).

Workload (BASELINE.json configs[1]): point-to-point asend/arecv of 1 MiB buffers, tag=1,
tag_mask=0xFFFF.  One step = a window of WINDOW messages: the receiver posts WINDOW receives,
the sender issues WINDOW sends then aflush(); the step ends when every receive has completed.
  N == 1: Server and Client on the same GPU (loopback; HBM-bound: 2 x payload bytes of traffic)
  N  > 1: rank r sends to rank (r+1) % N over NVLink and receives from (r-1) % N; per-GPU work is
          fixed (weak scaling); no collective on the data path (torch.distributed/gloo is used only
          to exchange address blobs and to take the max time over ranks).
`value` uses device-resident buffers; `e2e` runs the same steps with (pinned) HOST buffers through the
public API, so host->device and device->host copies are inside the timed region.
"""
from __future__ import annotations

import argparse
import asyncio
import gc
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
os.environ.setdefault("STARWAY_QUIET", "1")  # no "Connected!" banners: stdout carries JSON lines only
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MSG_BYTES = 1 << 20
WINDOW = 64
POOL_SETS = 4  # 4 x 64 MiB sources + 4 x 64 MiB destinations = 512 MiB > 126 MB L2
TAG, MASK = 1, 0xFFFF
METRIC = "tagged send/recv GB/s & Mmsg/s vs size, 1/2/4/8 B200; NVLink roofline %"
NVLINK_NOMINAL_GBS = 900.0  # BASELINE.md: score NVLink against the nominal 900 GB/s per direction (measured peer copy: 770)


def new_loop_runner():
    try:
        import uvloop

        return uvloop.run
    except Exception:
        return asyncio.run


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if self._nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1)
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
        }


SWEEP_SIZES = [64, 4096, 65536, 1 << 20, 16 << 20, 256 << 20, 1 << 30]   # config 3, sampled


def sweep_plan(n):
    """(window, iterations) of one sweep point: SURVEY 8d shape (window = min(64, max(1, 2^28 / n)) sends in flight,
    then aflush), bounded so that the whole sweep adds a fraction of a second to the run."""
    window = min(64, max(1, (1 << 28) // n))
    # at least 16 GiB per point above 16 MiB: the device-wide synchronisation that ends the timed region also waits
    # for the resident control kernels to notice the silence and leave (linger_us, 150 us) -- a fixed cost that a
    # handful of iterations would not amortise
    iters = max(8, min(100, (1 << 34) // (window * n)))
    return window, iters


async def run_sweep(torch, dev, server, client, rank, world, barrier, allreduce_max, allreduce_sum, sizes):
    """BASELINE config 3, sampled: for every size a stream of `window` messages per iteration (receives pre-posted,
    sends in flight, aflush), device buffers, public asyncio API; GB/s and Mmsg/s per direction per GPU, the
    fraction of the payload roofline, and a bit-exact check of the last window against the SENDER's pattern."""
    pool_bytes = max(sizes)
    def pattern(r):
        t = torch.arange(pool_bytes // 8, device=dev, dtype=torch.int64)
        t.mul_(2654435761).add_(r * 0x9E3779B1)
        return t.view(torch.uint8)
    src_pool = pattern(rank)
    exp_pool = src_pool if world == 1 else pattern((rank - 1) % world)
    dst_pool = torch.empty(pool_bytes, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    out = []
    for n in sizes:
        window, iters = sweep_plan(n)
        offs = [((j * n) % (pool_bytes - n + 1)) & ~255 for j in range(window)]   # 256-byte aligned whatever the pool size
        srcs = [src_pool[o:o + n] for o in offs]
        dsts = [dst_pool[o:o + n] for o in offs]
        dst_pool[: min(pool_bytes, window * n)].fill_(0xEE)
        torch.cuda.synchronize()

        async def one():
            recvs = [server.arecv(d, TAG, MASK) for d in dsts]
            sends = [client.asend(x, TAG) for x in srcs]
            for f in sends:
                await f
            await client.aflush()
            for f in recvs:
                await f

        await one()   # warm-up (mappings, pools)
        await one()
        gc.collect()  # the garbage of the set-up is collected here, not inside the timed iterations (same in the CPU arm)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            await one()
        torch.cuda.synchronize()
        el = allreduce_max(time.perf_counter() - t0)
        bad = allreduce_sum(sum(int(not torch.equal(dst_pool[o:o + n], exp_pool[o:o + n])) for o in offs))
        gbs = window * iters * n / el / 1e9
        out.append({"bytes": n, "window": window, "iters": iters, "gbs_per_gpu": round(gbs, 3),
                    "mmsg_per_s_per_gpu": round(window * iters / el / 1e6, 4), "bit_exact": bad == 0, "_gbs": gbs})
        barrier()
    del src_pool, dst_pool, exp_pool
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------- our arm
async def window_step(server, client, eps, srcs, dsts):
    recvs = [server.arecv(d, TAG, MASK) for d in dsts]
    sends = [client.asend(s, TAG) for s in srcs]
    for f in sends:  # awaiting in order is cheaper than asyncio.gather (no per-future callbacks)
        await f
    await client.aflush()
    return [await f for f in recvs]


DUMP_SAMPLE = 1 << 22  # received bytes kept by --dump-outputs: 16 MiB as float32, far below the 64 MB the dump may take


def dump_outputs(out_dir, torch, dsts, results):
    """Writes what the receiver got in one step, as a caller of window_step sees it:
      recv_results.npy  float64 (window, 2): (sender_tag, length) of every receive, in posting order
      recv_bytes.npy    float32: the received bytes, the window's buffers end to end; above DUMP_SAMPLE bytes a
                        sample at sorted positions drawn from a fixed seed (the same positions for the same arguments)
    The sample is gathered buffer by buffer, so no copy of the whole window is made."""
    import numpy as np

    total = sum(d.numel() for d in dsts)
    pos = np.arange(total) if total <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).integers(0, total, DUMP_SAMPLE))
    parts, start = [], 0
    for d in dsts:
        lo, hi = np.searchsorted(pos, [start, start + d.numel()])
        parts.append(d[torch.from_numpy(pos[lo:hi] - start).to(d.device)].cpu())
        start += d.numel()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "recv_results.npy"), np.asarray(results, dtype=np.float64))
    np.save(os.path.join(out_dir, "recv_bytes.npy"), torch.cat(parts).numpy().astype(np.float32))


def run_ours(args):
    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    torch.cuda.set_device(local_rank)
    os.environ["STARWAY_DEVICE"] = str(local_rank)
    import starway_b200 as sw

    # one process per GPU, bound to the GPU's NUMA node before any host buffer is allocated (the
    # launcher's job -- `numactl --cpunodebind` -- done here because the driver launches us bare)
    numa_bound = False if os.environ.get("STARWAY_BENCH_NO_BIND") else sw.bind_to_device_numa(local_rank)

    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("gloo", rank=rank, world_size=world)

    def barrier():
        if dist is not None:
            dist.barrier()

    ctx = sw.get_context()
    ctx.set_option("profile", 1)
    peaks, peaks_src = measured_peaks()
    msg, window = args.msg_bytes, args.window
    dev = torch.device("cuda", local_rank)

    async def main():
        server = sw.Server()
        addr = server.listen_address()
        addrs = [addr]
        if dist is not None:
            addrs = [None] * world
            dist.all_gather_object(addrs, addr)
        client = sw.Client()
        await client.aconnect_address(addrs[(rank + 1) % world])
        for _ in range(2000):
            if server.list_clients():
                break
            await asyncio.sleep(0.005)
        eps = list(server.list_clients())
        assert eps, "no inbound endpoint"
        barrier()

        # ---- device-resident buffers (inputs larger than L2: POOL_SETS rotating sets)
        g = torch.Generator(device=dev).manual_seed(0xB200 + rank)
        src = [[torch.randint(0, 256, (msg,), dtype=torch.uint8, device=dev, generator=g) for _ in range(window)]
               for _ in range(POOL_SETS)]
        dst = [[torch.full((msg,), 0xEE, dtype=torch.uint8, device=dev) for _ in range(window)]
               for _ in range(POOL_SETS)]
        torch.cuda.synchronize()

        async def timed(nsteps, srcs, dsts, sync):
            res = None
            for i in range(nsteps):
                k = i % POOL_SETS
                res = await window_step(server, client, eps, srcs[k], dsts[k])
                assert all(r == (TAG, msg) for r in res)
            sync()
            return res

        # the set-up garbage (torch import, buffer lists) goes to the permanent generation: full
        # collections inside the timed region would otherwise walk ~10^6 objects (same in the reference arm)
        if not os.environ.get("STARWAY_BENCH_NO_GC_FREEZE"):
            gc.collect()
            gc.freeze()
        # warm-up, then bit-exactness of one full window against the sources of the sending rank
        # The clock sampler (NVML from a thread, every 50 ms) runs from here to the end of the timed region: its first
        # query -- the slow one, and NVML queries can hold up kernel launches for milliseconds -- falls into the
        # warm-up instead of the first timed steps (a K = 20 region lasts 3 ms).
        late_clocks = bool(os.environ.get("STARWAY_BENCH_CLOCKS_LATE"))
        clocks = ClockSampler(local_rank)
        if not late_clocks:
            clocks.start()
        await timed(max(args.warmup, 3), src, dst, torch.cuda.synchronize)
        # Every rank checks the window it received against the sources of the rank that sent it (rank r-1;
        # its own at N == 1): the sources are a seeded sequence (Philox: seed and offset only), so any rank
        # can regenerate them.  The mismatch count is summed over ranks and asserted.
        peer = (rank - 1) % world
        gp = torch.Generator(device=dev).manual_seed(0xB200 + peer)
        bad = 0
        for j in range(window):
            exp = torch.randint(0, 256, (msg,), dtype=torch.uint8, device=dev, generator=gp)
            bad += int(not torch.equal(exp, dst[0][j]))
        if dist is not None:
            t = torch.tensor([bad], dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            bad = int(t[0])
        assert bad == 0, f"payload mismatch: {bad} of {world * window} messages differ from the sender's sources"
        payload_check = (f"asserted on every rank: {world} x {window} messages bit-exact vs the sending rank's regenerated sources")
        if args.dump_outputs:
            # the set the last timed step fills may have been filled by the warm-up already: clear it, so that what
            # --dump-outputs writes can only have come from the timed steps
            for d in dst[(args.steps - 1) % POOL_SETS]:
                d.fill_(0xEE)
        barrier()
        torch.cuda.synchronize()
        warm_batches = ctx.stats()["pull_batches"]
        ctx.reset_stats()
        if late_clocks:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        last_res = await timed(args.steps, src, dst, torch.cuda.synchronize)
        t1 = time.perf_counter()
        e1.record()
        e1.synchronize()
        barrier()
        clk = clocks.stop()
        st = ctx.stats()
        dev_ms = e0.elapsed_time(e1)
        wall_ms = (t1 - t0) * 1e3
        ms = max(dev_ms, wall_ms)
        per_rank = [(round(ms / args.steps, 4), len(os.sched_getaffinity(0)))]
        if dist is not None:
            per_rank = [None] * world
            dist.all_gather_object(per_rank, (round(ms / args.steps, 4), len(os.sched_getaffinity(0))))
            t = torch.tensor([ms], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        st["_per_rank"] = per_rank
        step_bytes = window * msg
        value = world * step_bytes * args.steps / (ms * 1e-3) / 1e9
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, torch, dst[(args.steps - 1) % POOL_SETS], last_res)

        # ---- the metric's "vs size" half: sampled sweep (config 3) at this N, same run
        def allreduce_max(x):
            if dist is None:
                return x
            t = torch.tensor([x], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])

        def allreduce_sum(x):
            if dist is None:
                return x
            t = torch.tensor([x], dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return int(t[0])

        sweep = []
        if not args.no_sweep:
            del src, dst
            torch.cuda.empty_cache()
            sweep = await run_sweep(torch, dev, server, client, rank, world, barrier, allreduce_max, allreduce_sum,
                                    [n for n in SWEEP_SIZES if n <= args.sweep_max_bytes])

        # ---- e2e: same steps with HOST buffers through the public API (H2D + D2H inside the timed region):
        #      page-locked NumPy arrays (the headline e2e) and ordinary pageable NumPy arrays (what a caller of the
        #      reference passes)
        def host_bufs(pinned):
            mk = (lambda a: a.pin_memory().numpy()) if pinned else (lambda a: a.numpy().copy())
            hs = [[mk(torch.from_numpy(np.random.default_rng(rank * 1000 + k * 100 + j).integers(0, 256, msg, dtype=np.uint8)))
                   for j in range(window)] for k in range(2)]
            hd = [[mk(torch.empty(msg, dtype=torch.uint8)) for _ in range(window)] for k in range(2)]
            return hs, hd

        marks = []

        async def e2e_leg(pinned):
            hsrc, hdst = host_bufs(pinned)

            async def timed_host(nsteps):
                for i in range(nsteps):
                    k = i % 2
                    marks.append(("e2e_step_begin", time.monotonic()))
                    res = await window_step(server, client, eps, hsrc[k], hdst[k])
                    marks.append(("e2e_step_end", time.monotonic()))
                    assert all(r == (TAG, msg) for r in res)

            await timed_host(3)
            if world == 1:
                for s_, d_ in zip(hsrc[0], hdst[0]):
                    assert np.array_equal(s_, d_), "host payload mismatch"
            barrier()
            torch.cuda.synchronize()
            steps = max(3, min(args.steps, 40))
            ctx.reset_stats()
            t0 = time.perf_counter()
            await timed_host(steps)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            barrier()
            ms_ = allreduce_max((t1 - t0) * 1e3)
            return world * step_bytes * steps / (ms_ * 1e-3) / 1e9, ms_, steps, ctx.stats()

        if args.no_e2e:
            await client.aclose()
            barrier()
            await server.aclose()
            return value, ms, st, clk, float("nan"), step_bytes, {}, payload_check, warm_batches, sweep
        e2e_value, e2e_ms, e2e_steps, st2 = await e2e_leg(True)
        e2e_pageable, pg_ms, pg_steps, _ = (float("nan"), float("nan"), 1, None) if os.environ.get("STARWAY_BENCH_SKIP_PAGEABLE") else await e2e_leg(False)
        if os.environ.get("STARWAY_TRACE"):
            with open(os.environ["STARWAY_TRACE"] + f".py.{os.getpid()}", "w") as f:
                for name, t in marks:
                    f.write(f"{t:.7f} {name} 0 0\n")
        e2e_diag = {"ms_per_step": round(e2e_ms / e2e_steps, 3),
                    "copy_kernel_ms_per_step": round((st2["bulk_event_ms"] + st2["pull_busy_ms"]) / e2e_steps, 3),
                    "bulk_launches_per_step": round((st2["bulk_tma_launches"] + st2["bulk_simt_launches"]) / e2e_steps, 1),
                    "pull_batches_per_step": round(st2["pull_batches"] / e2e_steps, 1),
                    "staged_h2d_bytes_per_step": int(st2["h2d_bytes"] / e2e_steps),
                    "staged_d2h_bytes_per_step": int(st2["d2h_bytes"] / e2e_steps),
                    "pageable_value": round(e2e_pageable, 2), "pageable_ms_per_step": round(pg_ms / pg_steps, 3)}

        await client.aclose()
        barrier()
        await server.aclose()
        return value, ms, st, clk, e2e_value, step_bytes, e2e_diag, payload_check, warm_batches, sweep

    value, ms, st, clk, e2e_value, step_bytes, e2e_diag, payload_check, st0_batches, sweep = new_loop_runner()(main())

    # ---- roofline of the dominant kernel: the rendezvous copy.  On the resident path the copies are made by the
    #      pull CTAs (sw_pull_kernel), which stay on the GPU across many batches: the time base is the union of the
    #      batches' active intervals (first chunk claimed -> batch completed, device timer), accumulated by the
    #      kernel itself over the timed region.  Host-launched copies (sw_bulk_tma_*_kernel; resident=0, or sources
    #      the control kernel cannot resolve) are timed with CUDA events on their stream.
    if st["pull_bytes"] > 0:
        launches = max(1, st["pull_batches"])
        avg_ms = st["pull_busy_ms"] / launches
        payload_per_launch = st["pull_bytes"] / launches
        kernel = ("sw_pull_kernel (resident pull CTAs, one elected thread each: cp.async.bulk global->smem->global, "
                  "8 x 24 KiB stages; a 'launch' here is one published batch of matched messages)")
        n_launches = st["pull_batches"]
    else:
        launches = max(1, st["bulk_event_launches"])
        avg_ms = st["bulk_event_ms"] / launches
        payload_per_launch = st["bulk_event_bytes"] / launches
        kernel = ("sw_bulk_tma_jobs_kernel (<= 96 messages per launch as kernel parameters, equal byte range per CTA; "
                  "larger launches: sw_bulk_tma_kernel, same cp.async.bulk pipeline)")
        n_launches = st["bulk_event_launches"]
    if world == 1:
        algo_bytes = 2 * payload_per_launch  # loopback: read N + write N bytes of HBM (SURVEY.md 8d)
        peak, bound, peak_note = float(peaks["hbm_gbs"]), "hbm", f"HBM copy, {peaks_src}"
    else:
        algo_bytes = payload_per_launch  # N payload bytes cross NVLink in one direction
        peak, bound, peak_note = NVLINK_NOMINAL_GBS, "nvlink", "NVLink 5 per direction, nominal 900 GB/s (BASELINE.md; measured peer copy on this pool: 770 GB/s)"
    achieved = algo_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("world") == world:
            traffic = tj["dram_bytes_per_payload_byte"] * payload_per_launch
    except Exception:
        pass
    roofline = {
        "bound": bound, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
        "frac": round(achieved / peak, 4), "traffic": traffic,
        "kernel": kernel,
        "launches": n_launches, "avg_launch_us": round(avg_ms * 1e3, 2),
        "payload_bytes_per_launch": int(payload_per_launch), "peak_source": peak_note,
    }
    if st["pull_batches"]:
        # per-batch phases of the pull CTAs (device timer; averages over the life of the context)
        tot = max(1, st0_batches + st["pull_batches"])
        roofline["batch_phases_us"] = {"published_to_first_claim": round(st["pull_pickup_ms"] * 1e3 / tot, 2),
                                       "first_claim_to_last_chunk": round(st["pull_copy_ms"] * 1e3 / tot, 2),
                                       "records_and_fin_words": round(st["pull_fin_ms"] * 1e3 / tot, 2)}
    gpu_launches = int(st["put_launches"] + st["prog_launches"] + st["pull_launches"] + st["match_launches"]
                       + st["deliver_launches"] + st["bulk_tma_launches"] + st["bulk_simt_launches"])
    if rank != 0:
        sw.shutdown()
        return
    cpu = cpu_baseline_run(args.msg_bytes, args.window, budget_s=10.0) if (world == 1 and not args.no_cpu_baseline) else None
    per_gpu_peak = float(peaks["hbm_gbs"]) / 2 if world == 1 else NVLINK_NOMINAL_GBS
    for pt in sweep:
        pt["frac_of_roofline"] = round(pt.pop("_gbs") / per_gpu_peak, 4)
    if cpu is not None and sweep:
        # the reference-shaped CPU path at the same sizes (SURVEY 8d: "reference CPU path beside it")
        cpu["sweep"] = cpu_sweep([pt["bytes"] for pt in sweep])
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {
            "workload": f"configs[1]: point-to-point asend/arecv, {msg} B device buffers, tag=1 tag_mask=0xFFFF, "
                        f"window {window} msgs/step + aflush; "
                        + ("1 GPU loopback (Server+Client on cuda:0)" if world == 1 else f"ring over {world} GPUs, rank r -> r+1 over NVLink"),
            "msg_bytes": msg, "window": window,
            "l2": f"inputs larger than L2: {POOL_SETS} rotating buffer sets, {2 * POOL_SETS * window * msg >> 20} MiB footprint",
            "timing": "wall clock + CUDA events between device-wide synchronisations, max over ranks",
            "api": "public asyncio API (one Future per message, as the reference)",
            "numa": "rank bound to the GPU-local CPUs" if numa_bound else "no CPU binding applied",
            "host_cpus_rank0": len(os.sched_getaffinity(0)), "resident": int(ctx.get_option("resident")),
            "per_rank_ms_per_step_and_cpus": st.get("_per_rank"),
            "payload_check_all_ranks": payload_check,
        },
        "mmsg_per_s": round(world * window * args.steps / (ms * 1e-3) / 1e6, 4),
        "sweep": {"what": "BASELINE config 3, sampled: per size, `window` messages in flight then aflush, device buffers, "
                          "per direction per GPU" + ("" if world == 1 else f"; every rank streams to rank+1 at once ({world}-GPU ring)"),
                  "roofline_gbs_per_gpu": round(per_gpu_peak, 1),
                  "roofline": "HBM copy / 2 (loopback: every payload byte is read and written)" if world == 1 else "NVLink 5, 900 GB/s per direction (nominal)",
                  "points": sweep},
        "nvlink_roofline_frac": None if world == 1 else round(value / world / 900.0, 4),
        "clocks": clk,
        "e2e": {"value": None if args.no_e2e else round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": step_bytes, "d2h_bytes_per_step": step_bytes,
                "buffers": "page-locked host NumPy arrays through Client.asend/Server.arecv", "rank0_breakdown": e2e_diag},
        "e2e_pageable": {"value": e2e_diag.get("pageable_value"), "unit": "GB/s",
                         "buffers": "ordinary (pageable) NumPy arrays through the same calls"},
        "reference_arm_note": "the reference arm (--impl reference) is ONE in-process CPU pair on rank 0 whatever N is: compare per GPU",
        "gpu_launches": gpu_launches,
        "roofline": roofline,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    sw.shutdown()


# ----------------------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_baseline_run(msg, window, budget_s=12.0, steps=None, warmup=2):
    """Times the restated reference (oracle/cpu_engine.cpp: spinning worker thread per object,
    1-slot mailboxes, per-completion GIL + call_soon_threadsafe, single-threaded memcpy) on the
    same workload shape with host NumPy buffers."""
    import numpy as np

    from oracle import starway_cpu as cpu

    async def main():
        port = 40000 + (os.getpid() % 20000)
        s, c = cpu.make_pair(port)
        await c.aconnect("127.0.0.1", port)
        srcs = [np.random.default_rng(j).integers(0, 256, msg, dtype=np.uint8) for j in range(window)]
        dsts = [np.zeros(msg, dtype=np.uint8) for _ in range(window)]

        async def step():
            recvs = [s.arecv(d, TAG, MASK) for d in dsts]
            sends = [c.asend(x, TAG) for x in srcs]
            await asyncio.gather(*sends)
            await c.aflush()
            res = await asyncio.gather(*recvs)
            assert all(r == (TAG, msg) for r in res)

        gc.collect()
        gc.freeze()
        for _ in range(warmup):
            await step()
        assert all(np.array_equal(a, b) for a, b in zip(srcs, dsts))
        n, t0 = 0, time.perf_counter()
        while True:
            await step()
            n += 1
            el = time.perf_counter() - t0
            if (steps is not None and n >= steps) or (steps is None and el > budget_s):
                break
        await c.aclose()
        await s.aclose()
        return n, el

    n, el = new_loop_runner()(main())
    return {
        "value": round(n * window * msg / el / 1e9, 3), "unit": "GB/s", "cores": 3, "kind": "port",
        "threads": "2 spinning native worker threads (1 per Server/Client object) + 1 Python thread",
        "host_cpus_available": len(os.sched_getaffinity(0)),
        "sample": f"{n} steps of {window} x {msg} B host NumPy messages, tag=1 mask=0xFFFF, Server+Client in one process "
                  f"({el:.1f} s); restated reference (libucp absent: oracle/cpu_engine.cpp + oracle/tagmatch.c)",
        "mmsg_per_s": round(n * window / el / 1e6, 4), "ms_per_step": round(el / n * 1e3, 3),
    }


def cpu_sweep(sizes, budget_s=1.2):
    """The restated reference on host cores at the sweep sizes (host NumPy buffers, same window shape)."""
    import numpy as np

    from oracle import starway_cpu as cpu

    async def main():
        port = 41000 + (os.getpid() % 20000)
        s, c = cpu.make_pair(port)
        await c.aconnect("127.0.0.1", port)
        pool = np.random.default_rng(7).integers(0, 256, max(sizes), dtype=np.uint8)
        dpool = np.zeros(max(sizes), dtype=np.uint8)
        out = []
        for n in sizes:
            window, _ = sweep_plan(n)
            offs = [((j * n) % (len(pool) - n + 1)) & ~255 for j in range(window)]
            srcs, dsts = [pool[o:o + n] for o in offs], [dpool[o:o + n] for o in offs]

            async def one():
                recvs = [s.arecv(d, TAG, MASK) for d in dsts]
                sends = [c.asend(x, TAG) for x in srcs]
                await asyncio.gather(*sends)
                await c.aflush()
                await asyncio.gather(*recvs)

            await one()
            await one()
            gc.collect()
            it, t0 = 0, time.perf_counter()
            while True:
                await one()
                it += 1
                el = time.perf_counter() - t0
                if el > budget_s or it >= 100:
                    break
            ok = all(np.array_equal(a, b) for a, b in zip(srcs, dsts))
            out.append({"bytes": n, "window": window, "iters": it, "gbs": round(window * it * n / el / 1e9, 3),
                        "mmsg_per_s": round(window * it / el / 1e6, 4), "bit_exact": bool(ok)})
        await c.aclose()
        await s.aclose()
        return out

    return new_loop_runner()(main())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the reference arm is a host-CPU measurement: rank 0 alone runs it
    cpu = cpu_baseline_run(args.msg_bytes, args.window, steps=args.steps, warmup=max(1, min(args.warmup, 3)))
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cpu["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"configs[1] shape on host cores: {args.msg_bytes} B host NumPy buffers, tag=1 tag_mask=0xFFFF, "
                               f"window {args.window} msgs/step + aflush, Server+Client in one process",
                   "msg_bytes": args.msg_bytes, "window": args.window},
        "cpu_baseline": cpu,
        "sweep": {"what": "the same CPU pair at the sweep sizes (host NumPy buffers)",
                  "points": [] if args.no_sweep else cpu_sweep([n for n in SWEEP_SIZES if n <= args.sweep_max_bytes])},
        "e2e": {"value": cpu["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--msg-bytes", type=int, default=MSG_BYTES)
    ap.add_argument("--window", type=int, default=WINDOW)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer e2e leg (ncu launch lists of the device-resident steps)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the sampled size sweep (config 3)")
    ap.add_argument("--sweep-max-bytes", type=int, default=1 << 30)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what rank 0 received in the last one as DIR/<name>.npy (CUDA arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs is written by the CUDA arm only; run it without --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
