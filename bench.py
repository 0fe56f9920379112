#!/usr/bin/env python
"""bench.py — the rx_tools hot path on B200: I/Q Msamples/s through full_demod() / fix_fft().

A "step" = one pass of the hot path over one batch of synthetic CS16 input.

Workloads (BASELINE.json `configs`, SURVEY.md §8d):
  fm2b   (default; configs[1]) rx_fm -M wbfm -s 300k -F 9 -r 48k: 2.4 Msps capture -> 300 k (3 x fifth_order
         + droop FIR) -> fast atan -> de-emphasis a=23 -> 48 kHz, 1 GiB CS16 stream, chunk 131072 complex
  fm2a   rx_fm -M wbfm -s 2400000 -r 48000 (no decimation, de-emphasis a=181), 1 GiB
  fm1    rx_fm -M fm -s 1024000 -r 24000 (configs[0] shape, D=1, atan2), 256 MiB
  fm5a   256 NBFM channels, boxcar D=100, lut, 2.4 M complex each (channels sharded over ranks)
  power3 rx_power 1 MHz span, 1024-bin, 32768 hop buffers (1 GiB), one hop
  power4 rx_power 24-1766 MHz, 4096-bin, 871 hops x 36 sweeps (1 GiB), hops sharded over ranks + ONE all-gather

The JSON line's `value` is the --workload (default fm2b).  Unless --no-extras, the same line carries `extra.fm2a`
(the literal `-s 2400000` WBFM), `extra.fm5a` (256 channels SHARDED over the ranks, strong scaling) and
`extra.power4` (871 hops SHARDED over the ranks + the in-library NCCL all-gather, strong scaling), so that the
multi-GPU runs of this script measure the two configurations that really shard.

Multi-GPU (torchrun, one rank per GPU): a single rx_fm stream does not shard (serial carry) -> every rank runs its own
stream ("replicas only", weak scaling, no collective).  rx_fm channels and rx_power hops shard contiguously.

--impl reference times the reference's own C path (oracle/_ref, the unmodified sources compiled in the
authoring container; else the port) on the host cores of this box; it never loads librxb200.so.
"""
from __future__ import annotations

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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHUNK = 262144   # int16 per chunk = 131072 complex (MAXIMUM_BUF_LENGTH, src/rtl_fm.c:80-82)
METRIC = "I/Q Msamples/s through full_demod() & fix_fft() at 1/2/4/8 B200 vs host CPU"

# what each workload is: the reference invocation it models.  CLI-level numbers only; each arm derives the DSP
# parameters with ITS OWN code (librxb200's rxb200_fm_derive / the reference's optimal_settings in oracle/_ref).
FM_CLI = {
    "fm2b": dict(wbfm=1, rate_s=300000, rate_r=48000, use_F=1, comp_fir_size=9),
    "fm2a": dict(wbfm=1, rate_s=2400000, rate_r=48000),
    "fm1": dict(rate_s=1024000, rate_r=24000),
}
FM5A = dict(downsample=100, custom_atan=2, rate_out=24000)      # not reachable through the CLI (SURVEY §8d cfg5A)
LABEL = {
    "fm2b": "rx_fm -M wbfm -s 300k -F 9 -r 48k (2.4 Msps capture -> 48 kHz)",
    "fm2a": "rx_fm -M wbfm -s 2400000 -r 48000 (D=1)",
    "fm1": "rx_fm -M fm -s 1024000 -r 24000 (atan2)",
    "fm5a": "256 NBFM channels at 2.4 Msps, boxcar D=100, lut",
    "power3": "rx_power -f 100M:101M:1k, 1024-bin fix_fft, Hann window table, batched hop buffers",
    "power4": "rx_power -f 24M:1766M:1k -c 28.5% -w hamming, 4096-bin fix_fft, 871 hops batched",
}
POWER_ARG = {"power3": ("100M:101M:1k", 0.0, "hann"), "power4": ("24M:1766M:1k", 0.285, "hamming")}
FM5A_CHANNELS, FM5A_PER = 256, 2_400_000 - (2_400_000 % 8)


def workload_config(workload, size_mib=0):
    """The part of `config` that names the workload: identical in both arms (the driver compares it)."""
    if workload == "fm5a":
        stream = FM5A_CHANNELS * FM5A_PER * 4 if not size_mib else size_mib << 20
    elif workload.startswith("fm"):
        stream = (size_mib or (256 if workload == "fm1" else 1024)) << 20
    else:
        stream = (size_mib or 1024) << 20
    return {"workload": LABEL[workload], "chunk_complex": CHUNK // 2 if workload.startswith("fm") else None,
            "bytes_per_step": int(stream), "input": "synthetic CS16, seeded (rx_tools_b200/synth.py), period tiled"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def kernel_source_sha(workload):
    """Hash of the CUDA sources behind a workload's dominant kernel: profiles/traffic_*.json carries it, so a dram-bytes
    figure measured on an older kernel is reported as stale instead of being passed on."""
    names = ["fm_kernels.cu", "fm_rows.cuh", "common.cuh"] if workload.startswith("fm") else ["power_kernels.cu", "common.cuh"]
    h = hashlib.sha256()
    for n in names:
        with open(os.path.join(ROOT, "rx_tools_b200", "csrc", n), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(workload):
    tp = os.path.join(ROOT, "profiles", f"traffic_{workload}.json")
    if not os.path.exists(tp):
        return None, "no ncu capture for this workload"
    try:
        rec = json.load(open(tp))
    except Exception:
        return None, "unreadable"
    if rec.get("source_sha16") != kernel_source_sha(workload):
        return None, "stale: the kernel source changed after the ncu capture (tools/measure_traffic.sh refreshes it)"
    return rec.get("dram_bytes_per_launch"), rec.get("from", "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum")


def fm_params(workload):
    from rx_tools_b200 import fm
    if workload == "fm5a":
        return fm.FmParams(**FM5A)
    return fm.derive_params(**FM_CLI[workload]).params


def fm_input_period(workload, n_complex):
    from rx_tools_b200 import synth
    if workload in ("fm2b", "fm2a"):
        return synth.cfg2_iq(n_complex)
    if workload == "fm1":
        return synth.cfg1_iq(n_complex)
    return synth.cfg5_iq(n_complex, 0)


def fm_out_bytes_per_sample(p):
    d = (1 << p.downsample_passes) if p.downsample_passes else p.downsample
    r = (p.rate_out2 / p.rate_out) if p.rate_out2 > 0 else 1.0
    return 2.0 * r / d


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=2)
        sm, smax, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = max(smax, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = [v for v in sm if v > 0.5 * smax] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, local, world


def barrier_sync(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _reduce(v, world, device, op):
    import torch
    if world == 1:
        return v
    import torch.distributed as dist
    t = torch.tensor([v], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


def max_over_ranks(v, world, device):
    return _reduce(v, world, device, "MAX")


def sum_over_ranks(v, world, device):
    return _reduce(v, world, device, "SUM")


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, seed=0):
    """Write what the timed path handed its caller in its last step as out_dir/<name>.npy: 8/16-bit integers as float32,
    wider ones as float64 (both exact).  Past DUMP_LIMIT bytes in all, each array is cut to the same share of its
    elements, picked by a generator seeded with `seed`: the same shapes give the same picks, so two builds compare
    element for element."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    out = {k: v.astype(np.float32 if v.dtype.itemsize <= 2 else np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in out.values())
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        if total > DUMP_LIMIT:
            keep = max(1, int(v.size * DUMP_LIMIT // total))
            idx = np.sort(np.random.default_rng(seed).choice(v.size, size=keep, replace=False))
            v = v.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


def timed_steps(step, steps, warmup, stream, world, local, sample_clocks=True):
    """W untimed steps, then exactly K steps bracketed by barrier + synchronize, CUDA events on the launching stream,
    max over ranks.  Returns (ms for the K steps, the running clock sampler or None): the K device-resident steps last
    a few milliseconds, less than one nvidia-smi sampling period, so the caller keeps the sampler running through its
    end-to-end timed region (same workload, hundreds of milliseconds) and finishes it there."""
    import torch
    dev = torch.device("cuda", local)
    for _ in range(warmup):
        step()
    barrier_sync(world)
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier_sync(world)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    e1.synchronize()
    barrier_sync(world)
    ms = e0.elapsed_time(e1)
    return max_over_ranks(ms, world, dev), sampler


# ------------------------------------------------------------------------------------------ rx_fm arm
def run_fm(args, workload, rank, local, world, main=True):
    import torch
    from rx_tools_b200 import fm
    dev = torch.device("cuda", local)
    p = fm_params(workload)
    if workload == "fm5a":
        n_per = FM5A_PER
        if args.size_mib:
            n_ch = max(1, (args.size_mib << 20) // (n_per * 4))          # per-GPU override (testing): weak
            sharded = False
        else:
            from rx_tools_b200 import sharding
            cb, ce = sharding.unit_range(rank, world, FM5A_CHANNELS)        # channels [cb, ce) of the 256 on this rank
            n_ch = ce - cb
            sharded = True
    else:
        n_ch, sharded = 1, False
        size_mib = args.size_mib or (256 if workload == "fm1" else 1024)
        n_per = (size_mib << 20) // 4
    period = min(n_per, 1 << 24)
    period -= period % (CHUNK // 2)
    n_per = (n_per // period) * period if n_per >= period else n_per
    host_period = fm_input_period(workload, period)
    reps = n_per // period
    d_period = torch.from_numpy(host_period).to(dev)
    d_in = d_period.repeat(n_ch * reps).contiguous()
    del d_period
    demod = fm.FmDemod(p, device=local, n_channels=n_ch)
    n_int16 = 2 * n_per
    cap = demod.max_output(n_int16, CHUNK) + 8
    d_out = torch.empty(n_ch * cap, dtype=torch.int16, device=dev)
    stream = torch.cuda.ExternalStream(demod.stream, device=dev)
    n_pcm = [0]

    def step():
        n_pcm[0] = demod.process_device(d_in.data_ptr(), n_int16, CHUNK, d_out.data_ptr(), cap, sync=False)

    steps = args.steps if main else max(3, min(args.steps, 10))
    ms, sampler = timed_steps(step, steps, args.warmup, stream, world, local, sample_clocks=main)
    if main and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pcm": d_out.view(n_ch, cap)[:, :n_pcm[0]].cpu().numpy()})
    stats = demod.stats()
    # dominant-kernel duration, CUDA events recorded around the fused kernel on its own stream
    kms = []
    for _ in range(max(3, min(steps, 10))):
        step()
        kms.append(demod.kernel_ms())
    kernel_ms = float(np.mean(kms))
    samples_rank = n_ch * n_per
    samples_all = sum_over_ranks(float(samples_rank), world, dev)
    value = samples_all * steps / (ms * 1e-3) / 1e6

    # end to end through the public host API: pinned host buffers, H2D + kernel + D2H inside the timed region
    e2e = None
    if main and not args.no_e2e:
        h_in = torch.empty(n_ch * n_int16, dtype=torch.int16).pin_memory()
        h_in.view(n_ch * reps, -1)[:] = torch.from_numpy(host_period)
        h_out = torch.empty(n_ch * cap, dtype=torch.int16).pin_memory()
        import ctypes as C
        from rx_tools_b200 import _lib
        npcm = C.c_size_t(0)
        demod.reset()

        def e2e_step():
            _lib.check(_lib.lib().rxb200_fm_process(demod._h, h_in.data_ptr(), n_int16, CHUNK, h_out.data_ptr(), cap,
                                                    C.byref(npcm), None))
        e2e_step()
        barrier_sync(world)
        t0 = time.perf_counter()
        k2 = max(2, min(steps, 5))
        for _ in range(k2):
            e2e_step()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        e2e = {"value": samples_all * k2 / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(n_ch * n_int16 * 2), "d2h_bytes_per_step": int(n_ch * npcm.value * 2),
               "steps": k2}
        del h_in, h_out
    if sampler is not None and len(sampler.rows) < 3:
        for _ in range(200):                      # nothing sampled yet (nvidia-smi starts slowly): keep the GPU on this workload
            step()
        torch.cuda.synchronize()
    clocks = sampler.finish() if sampler is not None else None

    peak, peak_src = peaks()
    bytes_per_sample = 4.0 + fm_out_bytes_per_sample(p)
    achieved = samples_rank * bytes_per_sample / (kernel_ms * 1e-3) / 1e9 if samples_rank else 0.0
    traffic, traffic_src = measured_traffic(workload)
    cfg = workload_config(workload, args.size_mib)
    cfg.update({"stream_bytes_per_gpu": int(n_ch * n_int16 * 2), "channels_per_gpu": n_ch,
                "l2": f"input ({n_ch * n_int16 * 2 / 2**20:.0f} MiB per step per GPU) is larger than the 126 MB L2",
                "parallelism": (f"channels sharded x{world}" if sharded else f"replicas x{world}")})
    res = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong" if sharded else "weak",
        "vs_baseline": None, "dtype": "int16/int32 (fp64 atan2 on first sample of each chunk)", "data": "synthetic",
        "config": cfg,
        "detail": {"segment_len": stats["segment_len"], "warmup_len": stats["warmup_len"],
                   "fixup_segments": stats["fixup_segments"], "launches_per_step": stats["launches"]},
        "gpu_launches": stats["launches"] * steps,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": stats.get("kernel", "fm_fused_kernel"), "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_sample": bytes_per_sample},
        "e2e": e2e,
    }
    demod.close()
    del d_in, d_out
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------ rx_power arm
def run_power(args, workload, rank, local, world, comm, main=True):
    import torch
    from rx_tools_b200 import power, synth
    dev = torch.device("cuda", local)
    arg, crop, wname = POWER_ARG[workload]
    plan = power.plan_range(arg, crop)
    window = power.window_table(wname, 1 << plan.bin_e)
    if workload == "power3":
        n_pass = ((args.size_mib or 1024) << 20) // (plan.buf_len * 2)
    else:
        n_pass = max(1, ((args.size_mib or 1024) << 20) // (plan.n_hops * plan.buf_len * 2))
    n_hops = plan.n_hops
    # hops shard contiguously over ranks (rxb200_power_shard, SURVEY §8e); one hop: the passes are split instead
    if n_hops == 1:
        hb, he = 0, 1
        my_pass = n_pass // world
    else:
        hb, he = power.shard(n_hops, world, rank)
        my_pass = n_pass
    nh = he - hb
    # every hop gets its own seeded buffers (seed = 4000 + hop, SURVEY §8d cfg4) so a mis-ordered gather would show
    base = np.concatenate([synth.power_hops(2, 1, plan.buf_len, seed=4000 + hb + i) for i in range(min(max(nh, 1), 16))], axis=1)
    d_base = torch.from_numpy(np.ascontiguousarray(base)).to(dev)            # [2][<=16][buf_len]
    reps_h = -(-max(nh, 1) // d_base.shape[1])
    d_in = d_base.repeat(-(-my_pass // 2), reps_h, 1)[:my_pass, :max(nh, 1)].contiguous().view(-1)
    sc = power.PowerScanner(plan, window, device=local)
    stream = torch.cuda.ExternalStream(sc.stream, device=dev)
    N = 1 << plan.bin_e
    do_gather = world > 1 and n_hops > 1

    def step():
        if nh > 0:
            sc.scanner_device(d_in.data_ptr(), my_pass, hb, he, sync=False)
        if do_gather:
            sc.gather(comm, sync=False)        # ONE in-place NCCL all-gather inside librxb200, on the handle's stream

    steps = args.steps if main else max(3, min(args.steps, 10))
    ms, sampler = timed_steps(step, steps, args.warmup, stream, world, local, sample_clocks=main)
    if main and args.dump_outputs and rank == 0:
        avg, smp = sc.read()
        dump_outputs(args.dump_outputs, {"avg": avg, "samples": smp})
    kms = []
    for _ in range(max(3, min(steps, 10))):
        if nh > 0:
            sc.scanner_device(d_in.data_ptr(), my_pass, hb, he, sync=False)
            kms.append(sc.kernel_ms())
    kernel_ms = float(np.mean(kms)) if kms else 0.0
    kernel_ms_max = max_over_ranks(kernel_ms, world, dev)
    gather_ms = None
    if do_gather:
        g_ms, _ = timed_steps(lambda: sc.gather(comm, sync=False), 5, 2, stream, world, local, sample_clocks=False)
        gather_ms = g_ms / 5
    samples_rank = my_pass * nh * (plan.buf_len // 2)
    samples_all = sum_over_ranks(float(samples_rank), world, dev)
    value = samples_all * steps / (ms * 1e-3) / 1e6
    e2e = None
    if main and not args.no_e2e and nh > 0:
        h_in = torch.empty(d_in.numel(), dtype=torch.int16).pin_memory()
        h_in.copy_(d_in.cpu())
        k2 = max(2, min(steps, 5))
        sc.reset()
        sc.scanner(h_in.numpy(), my_pass, hb, he)
        barrier_sync(world)
        t0 = time.perf_counter()
        for _ in range(k2):
            sc.scanner(h_in.numpy(), my_pass, hb, he)
            if do_gather:
                sc.gather(comm, sync=True)
            avg, smp = sc.read()
        dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        e2e = {"value": samples_all * k2 / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(d_in.numel() * 2), "d2h_bytes_per_step": int(avg.nbytes), "steps": k2}
    if sampler is not None and len(sampler.rows) < 3 and nh > 0:
        for _ in range(100):                      # kernel only: no collective here, ranks may disagree on the sample count
            sc.scanner_device(d_in.data_ptr(), my_pass, hb, he, sync=False)
        torch.cuda.synchronize()
    clocks = sampler.finish() if sampler is not None else None
    peak, peak_src = peaks()
    achieved = samples_rank * 4.0 / (kernel_ms * 1e-3) / 1e9 if kernel_ms else 0.0
    traffic, traffic_src = measured_traffic(workload) if world == 1 else (None, "single-GPU capture only")
    fft8 = (plan.downsample == 1 and plan.buf_len == 16384 and 3 <= plan.bin_e <= 13
            and not os.environ.get("RXB200_POWER_V1"))
    cfg = workload_config(workload, args.size_mib)
    cfg.update({"hops": n_hops, "passes": n_pass, "bins": N, "buf_len_int16": plan.buf_len,
                "hops_this_rank": nh,
                "l2": "hop buffers per step (~1 GiB over all GPUs) are larger than the 126 MB L2" if world == 1 else
                      f"{d_in.numel() * 2 / 2**20:.0f} MiB of hop buffers per GPU per step",
                "parallelism": (f"hops sharded x{world} + ONE in-place ncclAllGather of {-(-n_hops // world) * world}x{N} int64 rows"
                                " inside rxb200_power_gather" if n_hops > 1 else f"passes sharded x{world}")})
    res = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int16 FFT, int64 accumulate", "data": "synthetic",
        "config": cfg, "gpu_launches": steps, "clocks": clocks,
        "allgather_ms": gather_ms, "kernel_ms_max_over_ranks": kernel_ms_max,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": "power_fft8_kernel" if fft8 else "power_fft_kernel", "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_sample": 4.0},
        "e2e": e2e,
    }
    sc.close()
    del d_in
    torch.cuda.empty_cache()
    return res


def compact(res):
    """An extra workload inside the main line: the numbers, without repeating the boilerplate."""
    keep = ("value", "unit", "n_gpus", "steps", "ms_per_step", "scaling", "allgather_ms", "kernel_ms_max_over_ranks")
    out = {k: res[k] for k in keep if k in res and res[k] is not None}
    out["workload"] = res["config"]["workload"]
    out["parallelism"] = res["config"]["parallelism"]
    out["roofline"] = {k: res["roofline"][k] for k in ("achieved", "peak", "frac", "kernel", "kernel_ms", "traffic")}
    return out


# ------------------------------------------------------------------------------------------ CPU legs
def usable_cores():
    """Host threads this process may really use: the affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:            # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def _cpu_worker(job):
    """One host process = one copy of the reference's globals.  Imports oracle/ and the numpy generators only: the
    reference arm never maps librxb200.so."""
    kind_pref, workload, n_complex, repeats = job
    import oracle
    from rx_tools_b200 import synth      # pure numpy generators (the package __init__ loads nothing native)
    use_ref = kind_pref == "reference" and oracle.have_ref()
    if workload.startswith("fm"):
        if workload == "fm5a":
            op = oracle.FmParams(**FM5A)
        elif use_ref:
            op = oracle.RefFm().derive(**FM_CLI[workload])[0]        # the reference's own main() + optimal_settings()
        else:
            from rx_tools_b200 import fm                                # port only (no _ref on this box): host derive
            op = oracle.FmParams(**fm.derive_params(**FM_CLI[workload]).params.reference_fields())
        if workload in ("fm2b", "fm2a"):
            x = synth.cfg2_iq(n_complex)
        elif workload == "fm1":
            x = synth.cfg1_iq(n_complex)
        else:
            x = synth.cfg5_iq(n_complex, 0)
        if use_ref:
            return oracle.RefFm().time(op, x, CHUNK, repeats), n_complex * repeats, "reference"
        return oracle.port().fm_time(op, x, CHUNK, repeats), n_complex * repeats, "port"
    arg, crop, wname = POWER_ARG[workload]
    if use_ref:
        rp = oracle.RefPower()
        with open(os.devnull, "w") as dn:          # frequency_range() prints its plan to stderr
            saved = os.dup(2)
            os.dup2(dn.fileno(), 2)
            try:
                plan = rp.setup(arg, crop, 1, 0, 0, "rectangle", oracle.port().window_table(wname, 4096 if workload == "power4" else 1024))
            finally:
                os.dup2(saved, 2)
                os.close(saved)
        n_hops, buf_len = plan.tune_count, plan.buf_len
    else:
        from rx_tools_b200 import power
        pl = power.plan_range(arg, crop)
        n_hops, buf_len, bin_e = pl.n_hops, pl.buf_len, pl.bin_e
    n_pass = max(1, n_complex // (n_hops * (buf_len // 2)))
    hb = synth.power_hops(min(n_pass, 2), n_hops, buf_len, seed=777)
    hb = np.ascontiguousarray(np.tile(hb, (-(-n_pass // hb.shape[0]), 1, 1))[:n_pass])
    if use_ref:
        return rp.time(hb, n_pass, repeats), n_pass * n_hops * (buf_len // 2) * repeats, "reference"
    win = oracle.port().window_table(wname, 1 << bin_e)
    pp = oracle.PowerParams(bin_e=bin_e, buf_len=buf_len)
    return oracle.port().power_time(pp, win, hb, n_pass, n_hops, repeats), n_pass * n_hops * (buf_len // 2) * repeats, "port"


def _run_pool(ctx, procs, job):
    if procs == 1:
        return [_cpu_worker(job)]
    with ctx.Pool(procs) as pool:
        return pool.map(_cpu_worker, [job] * procs)


def cpu_leg(workload, cores, target_seconds=12.0, pick_procs=False):
    """Time the reference C path on `cores` host processes (each its own copy of the globals).  With pick_procs the
    process count is chosen by a short calibration among cores, cores/2, cores/4 (a box may expose more logical CPUs
    than it lets a container use)."""
    import multiprocessing as mp
    import oracle
    oracle.build()
    kind = "reference" if oracle.have_ref() else "port"
    n_complex = 1 << 23 if workload.startswith("fm") else 1 << 22
    t1, n1, kind = _cpu_worker((kind, workload, n_complex, 1))     # one repeat on one core: the unit of work
    ctx = mp.get_context("spawn")
    procs, tried = cores, {}
    if pick_procs and cores > 1:
        r_cal = max(1, int(1.5 / max(t1, 1e-3)))
        for c in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
            rs = _run_pool(ctx, c, (kind, workload, n_complex, r_cal))
            tried[c] = sum(r[1] for r in rs) / max(r[0] for r in rs) / 1e6
        procs = max(tried, key=tried.get)
    repeats = max(1, int(target_seconds / max(t1, 1e-3)))
    t0 = time.perf_counter()
    results = _run_pool(ctx, procs, (kind, workload, n_complex, repeats))
    wall = time.perf_counter() - t0
    total = sum(r[1] for r in results)
    slowest = max(r[0] for r in results)
    leg = {"value": total / slowest / 1e6, "unit": "Msamples/s", "cores": procs, "kind": kind,
           "sample": f"{repeats} x {n1} complex samples of the same workload per process, chunk {CHUNK // 2}; "
                     f"timed inside the C loop (slowest process {slowest:.2f} s, wall {wall:.1f} s)",
           "usable_cores_detected": cores}
    if tried:
        leg["calibration_msamples_by_procs"] = {str(k): round(v, 1) for k, v in tried.items()}
    return leg


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cores = usable_cores()
    t0 = time.perf_counter()
    # a step = every process runs the bounded sample once; K+W of them are sized to end within ~a minute
    leg = cpu_leg(args.workload, cores, target_seconds=min(45.0, max(6.0, 1.5 * (args.steps + args.warmup))), pick_procs=True)
    res = {"impl": "reference", "metric": METRIC,
           "value": leg["value"], "unit": "Msamples/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": (time.perf_counter() - t0) * 1e3 / max(args.steps, 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16/int32 C (gcc -O2)",
           "data": "synthetic", "config": workload_config(args.workload, args.size_mib),
           "detail": {"threads": leg["cores"], "usable_cores_detected": cores},
           "gpu_launches": 0, "cpu_baseline": leg,
           "e2e": {"value": leg["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="fm2b", choices=["fm2b", "fm2a", "fm1", "fm5a", "power3", "power4"])
    ap.add_argument("--size-mib", type=int, default=0, help="override the per-GPU input size (testing)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the --workload, no extra.* records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the --workload's outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        res = run_reference(args)
        if res is not None:
            print(json.dumps(res))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (librxb200 has no CPU fallback)")
    rank, local, world = dist_setup(args.gpus)
    comm = None
    if world > 1:
        from rx_tools_b200 import sharding
        comm = sharding.make_comm(rank, world, local)       # librxb200's own NCCL communicator (rx_power collation)

    def run(workload, main):
        if workload.startswith("fm"):
            return run_fm(args, workload, rank, local, world, main)
        return run_power(args, workload, rank, local, world, comm, main)

    res = run(args.workload, True)
    if not args.no_extras and not args.size_mib:
        res["extra"] = {}
        for w in ("fm2a", "fm5a", "power4"):
            if w == args.workload:
                continue
            if world > 1:
                res["extra"][w] = compact(run(w, False))     # collectives inside: a rank must not skip one on its own
                continue
            try:
                res["extra"][w] = compact(run(w, False))
            except Exception as e:       # single GPU: an extra must never take the headline down with it
                res["extra"][w] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        if world == 1 and not args.no_cpu:
            res["cpu_baseline"] = cpu_leg(args.workload, 1, target_seconds=12.0)
        else:
            res["cpu_baseline"] = None
        print(json.dumps(res))
    if comm is not None:
        comm.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
