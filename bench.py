#!/usr/bin/env python
"""bench.py - Msamples/s of the Mode S receive hot path (IQ demod + preamble detect + slice + CRC).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n 28] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): synthetic 1090 MHz IQ at 4 Msps, 2^28 complex samples (2 GiB) per GPU,
1000 DF11/DF17 bursts at mixed SNR on complex Gaussian noise. A step = one pass of the whole receive
chain over that buffer (fresh stream each step). At N > 1 every rank owns an independent channel of the
same size (weak scaling, no data-path collective; NCCL only fans the buffers out from rank 0).

  value        whole-job Msamples/s with the input resident in HBM (max-over-ranks device time, CUDA events)
  e2e          same through the public API from PINNED HOST memory: H2D of the IQ + D2H of the frames inside
  roofline     scan kernel: 8 algorithmic bytes/sample / its measured duration vs the measured HBM peak
  cpu_baseline the reference's own C++ (oracle/_ref: unmodified preamble_impl/slicer_impl/modes_crc behind the
               restated GNU Radio front end) on a bounded sample, all host threads

--dump-outputs DIR writes the frames the headline's last timed step delivered (see dump_outputs). The input is seeded,
so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RATE = 4e6
THRESHOLD_DB = 7.0
N_BURSTS = 1000
NOISE_SIGMA = 0.01
DUMP_LIMIT_BYTES = 64 << 20


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        top = sorted(sm)[len(sm) // 2:] if sm else []          # under-load half
        return {"sm_mhz": float(np.median(top)) if top else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- BASELINE.json configs (SURVEY.md 8d). "c1" is the N = 1 headline, "c2" the N > 1 headline -----------------------
CONFIGS = {
    "c1": dict(rate=4e6, seed=0, dense=False,
               what="synthetic 1090 MHz IQ @ 4 Msps, 1000 DF11/DF17 bursts at mixed SNR (BASELINE configs[1])"),
    "c2": dict(rate=10e6, seed=30, dense=False,
               what="one synthetic 10 Msps channel per GPU, seeds 30+rank, 1000 DF11/DF17 bursts each (BASELINE configs[2])"),
    "c3": dict(rate=20e6, seed=4, dense=False,
               what="20 Msps oversampled input, 10 samples/chip, 1000 DF11/DF17 bursts (BASELINE configs[3])"),
    "c4": dict(rate=4e6, seed=5, dense=True,
               what="dense-traffic stress @ 4 Msps: 10 000 overlapping squitters/s, 20 % with 1-5 flipped bits, plus "
                    "Mode A/C-like FRUIT pulse pairs (BASELINE configs[4])"),
}


def scene_args(cfg, n):
    if cfg["dense"]:
        nb = int(10_000 * n / cfg["rate"])
        return dict(n_bursts=nb, garble_frac=0.2, fruit=nb // 4, snr_db=(4.0, 30.0))
    return dict(n_bursts=N_BURSTS)


def make_device_scene(cfg, n, channel, device, out=None):
    """(iq float32[2n] on `device`, hex payloads sent or None). Seeded; noise from torch's device generator."""
    from gr_air_modes_b200 import synth
    iq, hexs, _ = synth.make_scene_device(cfg["rate"], n, seed=cfg["seed"] + channel, device=device,
                                          noise_sigma=NOISE_SIGMA, out=out, **scene_args(cfg, n))
    return iq, hexs


# ---- the checker: the reference's arithmetic on the very buffer that was timed (oracle/, test infrastructure) ----------
def oracle_full(iq_np, rate, threads):
    """Every detection and message the reference produces for this recording. Front end = the canonical restatement
    (oracle/modes_oracle.c, fp64 ascending window sums) evaluated in parallel over cuts with 49*spc samples of
    context (each output only depends on that many inputs); scan + slicer + CRC = oracle/_ref (the unmodified
    preamble_impl.cc / slicer_impl.cc / modes_crc.cc) when it was built, else the C port."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cpu_oracle as co
    port = co.Port()
    n = iq_np.size // 2
    spc = int(rate / 2e6)
    h = 49 * spc
    bb = np.empty(n, np.float32)
    avg = np.empty(n, np.float32)
    chunk = 1 << 20

    def work(a):
        b = min(a + chunk, n)
        a0 = max(0, a - h)
        x, y = port.frontend(iq_np[2 * a0: 2 * b], rate, True, co.MA_CANONICAL)
        bb[a:b] = x[a - a0:]
        avg[a:b] = y[a - a0:]

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(work, range(0, n, chunk)))
    kind = "reference" if co.ref_available() else "port"
    eng = co.Ref() if kind == "reference" else port
    return eng.run_streams(bb, avg, rate, THRESHOLD_DB), kind


def parity_check(rx, q, iq, rate, threads):
    """Run the CUDA chain once more over `iq` (device tensor) collecting everything, D2H the recording, run the
    oracle over it and compare every detection index and every message string."""
    from collections import Counter
    t0 = time.perf_counter()
    rx.reset()
    rx._slicer._first = True            # a fresh slicer's first message has 6 digits (slicer_impl.cc:192)
    q.flush()
    rx.process(iq, flush=True)
    ours_idx = np.array([f.sample_index for f in rx.frames], dtype=np.uint64)
    ours_msgs = q.strings()
    q.flush()
    host = iq.cpu().numpy()
    want, kind = oracle_full(host, rate, threads)
    del host
    if ours_msgs == want.msgs:
        m = dict(matched=len(ours_msgs), missing=0, extra=0)
    else:
        a, b = Counter(ours_msgs), Counter(want.msgs)
        m = dict(matched=sum((a & b).values()), missing=sum((b - a).values()), extra=sum((a - b).values()))
    wi = want.index.astype(np.uint64)
    if ours_idx.size == wi.size and np.array_equal(ours_idx, wi):
        d = dict(matched=int(wi.size), missing=0, extra=0)
    else:
        both = np.intersect1d(ours_idx, wi).size
        d = dict(matched=int(both), missing=int(wi.size - both), extra=int(ours_idx.size - both))
    return {"matched": m["matched"], "missing": m["missing"], "extra": m["extra"], "compared": "every message string "
            "(payload, CRC syndrome, level, timestamp) and every detection index of the timed recording, full size",
            "detections": d, "oracle": kind, "seconds": round(time.perf_counter() - t0, 1)}


def dump_outputs(out_dir, frames):
    """What a caller of the timed path receives: its frames (struct amb_frame, stream order), one float64 array per
    field as out_dir/<field>.npy; lowconfbits and data are [n, 24] and [n, 14]. Beyond DUMP_LIMIT_BYTES in all, a fixed
    seeded sample of the frames (kept in stream order) is written instead."""
    from gr_air_modes_b200._lib import Frame
    rec = np.frombuffer(b"".join(bytes(f) for f in frames), dtype=np.dtype(Frame))
    names = [name for name, _ in Frame._fields_ if name != "pad_"]
    per_frame = 8 * sum(int(np.prod(rec.dtype[name].shape)) for name in names)
    if rec.size * per_frame > DUMP_LIMIT_BYTES:
        rec = rec[np.sort(np.random.default_rng(0).choice(rec.size, DUMP_LIMIT_BYTES // per_frame, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name in names:
        np.save(os.path.join(out_dir, name + ".npy"), rec[name].astype(np.float64))


def run_config(key, n, args, rank, local_rank, world, device, fan=None, steps=None, dump_dir=None):
    """Device-resident timing + full-size parity of one BASELINE config. Returns (result dict, iq, rx, q)."""
    import torch
    import torch.distributed as dist
    import gr_air_modes_b200 as am
    from gr_air_modes_b200 import shard
    cfg = CONFIGS[key]
    rate = cfg["rate"]
    steps = steps or args.steps
    t_f0 = time.perf_counter()
    timing = {}
    iq, sent = shard.fan_out(lambda ch: make_device_scene(cfg, n, ch, device), rank, world, device, 2 * n, timing)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_f0
    q = am.msg_queue()
    rx = am.rx_path(rate, THRESHOLD_DB, q, use_pmf=True, device=local_rank)
    rx._ctx.use_stream(torch.cuda.current_stream().cuda_stream)
    rx._ctx.call("amb_enable_timing", 1)

    def step():
        rx.reset()
        rx.process(iq, flush=True, collect=False)

    for _ in range(args.warmup):
        step()
    nmsg = rx.drain()
    q.flush()
    launches0 = rx.stats().kernel_launches
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    rx._ctx.join()                 # the sparse kernels of the last step run on the library's second stream
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    scan_ms = rx._ctx.scan_times_ms(min(steps, 64))
    st = rx.stats()
    launches = st.kernel_launches - launches0
    rx.drain()                     # the last timed step's frames: reset() dropped the earlier steps' results
    if dump_dir:
        dump_outputs(dump_dir, rx.frames)
    q.flush()
    ms_max = shard.max_over_ranks(ms, world, device)
    scan_avg = shard.max_over_ranks(float(np.mean(scan_ms)), world, device)
    peak, peak_src = measured_peak_gbs()
    res = {"config": key, "workload": cfg["what"], "rate_sps": rate, "samples_per_gpu": n,
           "value": world * n * steps / (ms_max * 1e-3) / 1e6, "unit": "Msamples/s", "steps": steps,
           "ms_per_step": ms_max / steps, "scan_ms": scan_avg,
           "frac": 8.0 * n / (scan_avg * 1e-3) / 1e9 / peak, "step_frac": 8.0 * n / (ms_max / steps * 1e-3) / 1e9 / peak,
           "msgs_per_step": nmsg, "candidates": int(st.candidates), "detections": int(st.detections),
           "gpu_launches": int(launches), "setup_s": round(setup_s, 2)}
    if sent is not None:
        res["bursts_sent"] = len(sent)
    if timing.get("bytes"):
        res["fanout_gbps"] = timing["bytes"] / (timing["send_ms"] * 1e-3) / 1e9
        res["fanout_ms"] = timing["send_ms"]
    if not args.no_parity:
        threads = max(1, len(os.sched_getaffinity(0)) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
        par = parity_check(rx, q, iq, rate, threads)
        if world > 1:       # sum over ranks
            t = torch.tensor([par["matched"], par["missing"], par["extra"], par["detections"]["matched"],
                              par["detections"]["missing"], par["detections"]["extra"]], dtype=torch.int64, device=device)
            dist.all_reduce(t)
            v = [int(x) for x in t.tolist()]
            par.update(matched=v[0], missing=v[1], extra=v[2], detections=dict(matched=v[3], missing=v[4], extra=v[5]))
        res["parity"] = par
    return res, iq, rx, q


def bind_near_gpu(index):
    """Pin this process to the CPUs next to GPU `index` (NVML's ideal affinity) so that the pinned staging buffer of
    the end-to-end leg lands on the NUMA node the GPU's PCIe root hangs off. Returns a note for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:                                    # CUDA's device order need not be NVML's: go through the PCI address
            import torch
            pr = torch.cuda.get_device_properties(index)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
        except Exception:                       # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (int(v) >> b) & 1} & os.sched_getaffinity(0)
        if not cpus:
            return "nvml gave no usable cpu set"
        os.sched_setaffinity(0, cpus)
        return "%d cpus near gpu %d" % (len(cpus), index)
    except Exception as e:                      # noqa: BLE001 - optional tuning only
        return "not bound (%s)" % type(e).__name__


def _tame_malloc():
    """Keep multi-MB buffers on the heap instead of mmap/munmap per call: the per-call allocations are an artefact
    of the oracle's whole-buffer driver (GNU Radio keeps persistent ring buffers), and first-touch page faults
    would otherwise dominate the CPU arm."""
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6")
        libc.mallopt(-3, 1 << 30)            # M_MMAP_THRESHOLD
        libc.mallopt(-1, (1 << 31) - 1)      # M_TRIM_THRESHOLD
    except Exception:
        pass


def _cpu_arm_setup(cfg, log2n):
    """Shared by the reference arm and the cpu_baseline leg: engine, thread count, one DISTINCT cut per thread."""
    from oracle import cpu_oracle as co
    from gr_air_modes_b200 import synth
    _tame_malloc()
    port = co.Port()
    kind = "reference" if co.ref_available() else "port"
    ref = co.Ref() if kind == "reference" else None
    cores = max(1, min(len(os.sched_getaffinity(0)), 256))       # every host thread we are allowed to use
    n_slice = 1 << (23 if cores <= 64 else 22)
    rate = cfg["rate"]
    n_full = 1 << log2n
    sa = scene_args(cfg, n_slice)
    if not cfg["dense"]:
        sa["n_bursts"] = max(1, int(N_BURSTS * n_slice / n_full))
    sc = synth.make_scene(rate, n_slice, sa.pop("n_bursts"), 7, noise_sigma=NOISE_SIGMA, **sa)
    # one private copy per thread: 128 threads re-reading ONE 32 MB cut would run out of the L3, a stream does not
    slices = [sc.iq.copy() for _ in range(cores)]

    def work(iq):
        bb, avg = port.frontend(iq, rate, True, co.MA_GR_FLOAT, 4096)     # GNU Radio's fp32 running-sum schedule
        r = (ref.run_streams(bb, avg, rate, THRESHOLD_DB) if ref else port.run_streams(bb, avg, rate, THRESHOLD_DB))
        return len(r.msgs)

    what = "%d threads, each over its own 2^%d-sample cut of the same scene type (the full 2^%d-sample recording does " \
           "not fit a bounded CPU step): GR fp32 moving averages + %s preamble/slicer/CRC" % (
               cores, int(np.log2(n_slice)), log2n, "the unmodified reference's" if ref else "the oracle port's")
    return work, slices, cores, n_slice, kind, what


def reference_arm(args, rank, world, key):
    """The reference's own CPU implementation of the path, all host threads, bounded sample per step."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    cfg = CONFIGS[key]
    work, slices, cores, n_slice, kind, what = _cpu_arm_setup(cfg, args.log2n)
    with ThreadPoolExecutor(cores) as ex:
        for _ in range(max(args.warmup, 2)):
            list(ex.map(work, slices))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            msgs = list(ex.map(work, slices))
        dt = time.perf_counter() - t0
    total = args.steps * cores * n_slice
    val = total / dt / 1e6
    line = {"impl": "reference", "metric": "Msamples/s IQ demod+slice+CRC", "value": val, "unit": "Msamples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["what"] + "; CPU arm = bounded sample of that workload", "config_key": key,
                       "rate_sps": cfg["rate"], "threshold_db": THRESHOLD_DB, "use_pmf": True,
                       "same_config_note": "same scene type, rate, threshold and burst density as the GPU arm; per step "
                                           "the CPU processes cores x 2^%d samples instead of 2^%d" % (int(np.log2(n_slice)), args.log2n)},
            "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": what},
            "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "msgs_per_step": int(sum(msgs))}
    print(json.dumps(line))


def cpu_baseline_leg(key, log2n):
    from concurrent.futures import ThreadPoolExecutor
    work, slices, cores, n_slice, kind, what = _cpu_arm_setup(CONFIGS[key], log2n)
    reps = max(1, int(round(2 * (1 << 29) / (cores * n_slice))))  # ~2^30 samples in total: 10-30 s of CPU work
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(work, slices))
        list(ex.map(work, slices))
        t0 = time.perf_counter()
        for _ in range(reps):
            list(ex.map(work, slices))
        dt = time.perf_counter() - t0
    val = reps * cores * n_slice / dt / 1e6
    return {"value": val, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": "%d passes x %s" % (reps, what)}


def time_shard_arm(args, rank, local_rank, world, device):
    """Secondary multi-GPU mode (SURVEY.md 8e): one recording, `world` time spans with halos, the scan-loop state
    (16 bytes) handed down the ranks between the dense and the sparse stages. Strong scaling; not the headline."""
    import torch
    import torch.distributed as dist
    import gr_air_modes_b200 as am
    from gr_air_modes_b200 import shard
    n = 1 << args.log2n
    plan = shard.time_shard_plan(n, world, am.query_geometry(RATE, THRESHOLD_DB, True))
    active = rank < len(plan)
    sp = plan[rank] if active else None
    t_f0 = time.perf_counter()
    whole = sent = None
    if rank == 0:
        whole, sent = make_device_scene(CONFIGS['c1'], n, 0, device)
        for r in range(1, len(plan)):
            dist.send(whole[2 * plan[r].first_sample: 2 * plan[r].end].contiguous(), dst=r)
        iq = whole[: 2 * sp.end]
    elif active:
        iq = torch.empty(2 * (sp.end - sp.first_sample), dtype=torch.float32, device=device)
        dist.recv(iq, src=0)
    torch.cuda.synchronize()
    fanout_s = time.perf_counter() - t_f0
    q = am.msg_queue()
    rx = am.rx_path(RATE, THRESHOLD_DB, q, use_pmf=True, device=local_rank)
    rx._ctx.use_stream(torch.cuda.current_stream().cuda_stream)
    recv, send = shard.dist_state_exchange(rank, device)

    gather = shard.dist_all_gather6(world, device) if world > 1 else (lambda v: [list(v)])
    last = len(plan) - 1
    fallbacks = [0]

    scratch = (shard.AsyncPass(world, len(plan), device, steps=args.warmup + args.steps + 1, side=torch.cuda.Stream(device))
               if args.ts_mode == "async" and not args.chain else None)
    counter = [0]

    def step():
        if scratch is not None:                          # device-side hand-over: a fixed sequence of enqueues
            shard.time_shard_pass_async(rx, iq if active else None, plan, rank, scratch, counter[0])
            counter[0] += 1
            return
        if args.chain:
            if not active:
                return
            rx.seek(sp.first_sample, sp.first_decision)
            rx.process(iq, flush=sp.flush, collect=False)
            entry = recv()[:2] if rank else (0, 0)
            rx.resolve(entry)
            if not sp.flush:
                send(rx.walk_state() + (0,))
            return
        mine = [0] * 6                                   # speculative resolution: one all-gather, no chain
        if active:
            rx.seek(sp.first_sample, sp.first_decision)
            rx.process(iq, flush=sp.flush, collect=False)
            if rank < last:
                rx.resolve(None)
                s = rx.walk_summary()
                mine = [s.pos, s.p, s.first_real, s.first_packet, s.exact_span, s.frames_passed]
        entries, _, bad = shard.compose_entries(plan, gather(mine))
        fallbacks[0] += bad < last
        if active and rank >= bad:
            rx.resolve(entries[rank] if rank == bad else recv()[:2])
            if not sp.flush:
                send(rx.walk_state() + (0,))

    rx.defer_resolve(True)
    for _ in range(args.warmup):
        step()
    launches0 = rx.stats().kernel_launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    rx._ctx.join()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0)
    if world > 1:
        dist.barrier()
    launches = rx.stats().kernel_launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_max = shard.max_over_ranks(ms, world, device)
    if scratch is not None:                              # passes whose speculation did not hold would have to be redone
        fallbacks[0] = int((scratch.out[args.warmup: args.warmup + args.steps, 0] < last).sum().item())
    # ---- check: the spans' messages, concatenated in rank order, are the one-shot run's
    if args.chain:
        mine = shard.process_time_sharded(rx, iq, sp, recv, send) if active else 0
    else:
        mine = shard.process_time_sharded_speculative(rx, iq if active else None, plan, rank, gather, recv, send)
    msgs = q.strings()
    q.flush()
    allm = [None] * world
    if world > 1:
        dist.all_gather_object(allm, msgs)
    else:
        allm = [msgs]
    if rank == 0:
        rx.defer_resolve(False)
        rx.reset()
        rx._slicer._first = True                  # a fresh slicer's first message has 6 digits (slicer_impl.cc:192)
        rx.process(whole, flush=True)
        ref_msgs = q.strings()
        joined = [m for part in allm for m in part]
        line = {"metric": "Msamples/s IQ demod+slice+CRC", "value": n * args.steps / (ms_max * 1e-3) / 1e6,
                "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "mode": "time-shard/" + ("async (device-side hand-over)" if scratch is not None else "chain" if args.chain else "speculative (host-driven)"),
                "fallback_steps": fallbacks[0],
                "config": {"workload": "ONE synthetic 4 Msps recording of 2^%d samples cut into %d time spans with halos"
                                       % (args.log2n, len(plan)), "parallelism": "time-shard x%d" % len(plan),
                           "fanout_s": round(fanout_s, 3), "timing": "host clock between barrier+synchronize (the state "
                           "hand-over is host-driven)", "spans": [repr(x) for x in plan]},
                "identical_to_one_shot": joined == ref_msgs, "msgs": len(ref_msgs),
                "gpu_launches": int(launches), "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def e2e_legs(rx, q, iq, n, args, local_rank, world, device):
    """End to end through the public API (rx_path.process): the step's IQ starts in HOST memory, the H2D copy, the
    whole chain and the read-back of the frames are inside the timed region. Headline: pinned float32 (gr_complex,
    the reference's boundary). Extras: pageable host memory, 16-bit IQ, small process() calls as GNU Radio makes them."""
    import torch
    import torch.distributed as dist
    from gr_air_modes_b200 import shard
    numa = bind_near_gpu(local_rank)          # the pinned buffer is first-touched on the GPU's NUMA node
    host = torch.empty(2 * n, dtype=torch.float32, pin_memory=True)
    host.copy_(iq)
    torch.cuda.synchronize()

    def timed(fn, reps):
        fn()
        q.flush()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0) / reps
        q.flush()
        return shard.max_over_ranks(ms, world, device)

    d2h = [0]

    def pinned():
        rx.reset()
        rx.process(host, flush=True)          # H2D copy + kernels + frame read-back (drain) inside
        d2h[0] = len(rx.frames) * 80 + 32

    ms = timed(pinned, args.e2e_steps)
    out = {"value": world * n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 8 * n,
           "d2h_bytes_per_step": d2h[0], "ms_per_step": ms, "h2d_gbps": 8 * n / (ms * 1e-3) / 1e9,
           "host_numa_binding": numa, "input": "pinned host float32 I/Q (gr_complex)"}
    extras = {}
    if not args.no_e2e_extras:
        extras = e2e_extra_legs(rx, q, host, n, args, world, timed)
    del host
    return out, extras


def e2e_extra_legs(rx, q, host, n, args, world, timed):
    """Further end-to-end figures through the same public call (not the headline):
      e2e_pageable    the recording in ordinary pageable memory (np.fromfile, GNU Radio buffers): the library gathers it
                      into its pinned ring with a few copy threads while earlier chunks are in flight
      e2e_sc16        16-bit IQ (the receivers' wire format) from pinned memory, widened on the device: half the bytes
      e2e_small_call  process() calls of 8 k / 32 k / 256 k samples + a non-blocking poll each, the way a GNU Radio
                      sink block's work() drives the library; x real time at the config's sample rate"""
    import torch
    out = {}
    rate = rx._rate
    # ---- pageable
    page = np.empty(2 * n, dtype=np.float32)
    page[:] = host.numpy()

    def pageable():
        rx.reset()
        rx.process(page, flush=True)

    ms = timed(pageable, max(1, args.e2e_steps - 1))
    out["e2e_pageable"] = {"value": world * n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms,
                           "h2d_bytes_per_step": 8 * n, "input": "pageable host float32 I/Q"}
    del page
    # ---- 16-bit IQ
    i16 = torch.empty(2 * n, dtype=torch.int16, pin_memory=True)
    step = 1 << 26
    for a in range(0, 2 * n, step):
        i16[a:a + step] = torch.clamp(torch.round(host[a:a + step] * 32768.0), -32768, 32767).to(torch.int16)

    def sc16():
        rx.reset()
        rx.process(i16, flush=True)

    ms = timed(sc16, args.e2e_steps)
    out["e2e_sc16"] = {"value": world * n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms,
                       "h2d_bytes_per_step": 4 * n, "input": "pinned host int16 I/Q, widened x*2^-15 on the device",
                       "msgs_per_step": len([f for f in rx.frames if f.passed])}
    del i16
    # ---- small calls (bounded stretch of the stream)
    small = {}
    hv = host.numpy()
    for call in (8192, 32768, 262144):
        total = min(n, call * 512)

        def run():
            rx.reset()
            got = 0
            for a in range(0, total, call):
                rx.process(hv[2 * a: 2 * (a + call)], flush=False, collect=False)
                got += rx.poll_ready()
            rx.process(hv[:0], flush=True)
            return got

        ms = timed(run, 2)
        small[str(call)] = {"Msamples/s": total / (ms * 1e-3) / 1e6, "x_real_time": total / (ms * 1e-3) / rate,
                            "us_per_call": 1e3 * ms / (total // call)}
    out["e2e_small_call"] = {"calls_of_samples": small, "how": "rx_path.process(chunk, collect=False) + rx_path.poll_ready() per "
                             "call over 512 calls of pinned-host float32, then a closing flush; input gathered by the library "
                             "(option coalesce = 2^18 samples)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS), help="headline workload (default: c1 on one GPU, "
                    "c2 = one 10 Msps channel per GPU on several)")
    ap.add_argument("--rate", type=float, default=None, help="shorthand: 4e6 -> c1, 10e6 -> c2, 20e6 -> c3")
    ap.add_argument("--dense", action="store_true", help="shorthand for --config c4")
    ap.add_argument("--extra-configs", default=None, help="comma list of further configs measured into configs[] "
                    "(default: the other three on one GPU, c1 on several; 'none' to skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-e2e-extras", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the end-to-end legs (the line then has no e2e)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the frames of the headline's last timed "
                    "step as DIR/<field>.npy (rank 0)")
    ap.add_argument("--time-shard", action="store_true",
                    help="secondary mode: ONE 2^log2n-sample recording cut into --gpus spans (strong scaling)")
    ap.add_argument("--chain", action="store_true", help="--time-shard: plain hand-over chain instead of speculative resolution")
    ap.add_argument("--ts-mode", default="async", choices=["async", "host"], help="--time-shard: speculative resolution with the "
                    "device-side hand-over (default) or driven by the host (round 1)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    key = args.config
    if key is None and args.dense:
        key = "c4"
    if key is None and args.rate is not None:
        key = {4e6: "c1", 10e6: "c2", 20e6: "c3"}.get(args.rate)
        if key is None:
            raise SystemExit("bench.py: --rate must be 4e6, 10e6 or 20e6 (the BASELINE configs)")
    if key is None:
        key = "c1" if max(world, args.gpus) == 1 else "c2"

    if args.impl == "reference":
        reference_arm(args, rank, world, key)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - this framework has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    n = 1 << args.log2n
    if args.time_shard:
        time_shard_arm(args, rank, local_rank, world, device)
        return

    if args.extra_configs is None:
        extra = [k for k in ("c2", "c3", "c4") if k != key] if world == 1 else [k for k in ("c1",) if k != key]
        if world == 1 and key != "c1":
            extra = ["c1"] + extra
    else:
        extra = [k for k in args.extra_configs.split(",") if k and k != "none"]

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    all_cpus = os.sched_getaffinity(0)
    head, iq, rx, q = run_config(key, n, args, rank, local_rank, world, device,
                                 dump_dir=args.dump_outputs if rank == 0 else None)
    e2e, e2e_extras = (None, {}) if args.no_e2e else e2e_legs(rx, q, iq, n, args, local_rank, world, device)
    clocks = sampler.stop() if rank == 0 else None     # sampled across the headline's timed regions (device + end to end)
    os.sched_setaffinity(0, all_cpus)                  # the CPU legs below get every host thread back
    rx.close()
    del iq, rx
    torch.cuda.empty_cache()

    others = []
    for k in extra:
        r, iq2, rx2, _ = run_config(k, n, args, rank, local_rank, world, device)
        rx2.close()
        del iq2, rx2
        torch.cuda.empty_cache()
        others.append(r)

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        cfg = CONFIGS[key]
        ach = 8.0 * n / (head["scan_ms"] * 1e-3) / 1e9
        scan_name = "amb_scan_kernel<%d,true,%d>" % (int(cfg["rate"] / 2e6), 2 if cfg["rate"] <= 6e6 else 1)
        line = {
            "metric": "Msamples/s IQ demod+slice+CRC", "value": head["value"],
            "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s; 2^%d complex samples per GPU; one independent channel per GPU" % (cfg["what"], args.log2n),
                       "config_key": key, "rate_sps": cfg["rate"], "threshold_db": THRESHOLD_DB, "use_pmf": True,
                       "samples_per_gpu": n,
                       "l2": "input (%.1f GiB per GPU) is larger than L2, no flush needed" % (8 * n / 2 ** 30),
                       "parallelism": "channel-per-gpu x%d" % world, "setup_s": head["setup_s"],
                       "e2e_steps": args.e2e_steps, "msgs_per_step": head["msgs_per_step"],
                       "candidates_per_step": head["candidates"], "detections_per_step": head["detections"]},
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": None, "kernel": scan_name, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": 8 * n, "scan_ms": head["scan_ms"],
                         "whole_step_frac": head["step_frac"]},
            "e2e": e2e,
            "gpu_launches": head["gpu_launches"], "clocks": clocks,
        }
        if "fanout_gbps" in head:
            line["config"]["fanout_gbps"] = head["fanout_gbps"]
            line["config"]["fanout_ms"] = head["fanout_ms"]
        if "parity" in head:
            line["parity"] = head["parity"]
        line.update(e2e_extras)
        line["configs"] = others
        line["roofline"].update(scan_traffic(key, args.log2n))
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_leg(key, args.log2n)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def scan_traffic(key, log2n):
    """dram bytes per scan launch from the committed ncu capture - only if that capture was taken of the kernel
    source that is built now (profiles/scan_traffic.json records the sha256 of csrc/amb_kernels.cu)."""
    import hashlib
    tr = os.path.join(ROOT, "profiles", "scan_traffic.json")
    try:
        rec = json.load(open(tr))
        src = os.path.join(ROOT, "gr_air_modes_b200", "csrc", "amb_kernels.cu")
        sha = hashlib.sha256(open(src, "rb").read()).hexdigest()
        ent = rec.get("%s_2p%d" % (key, log2n))
        if not ent:
            return {"traffic": None, "traffic_note": "no ncu capture of this config committed"}
        if ent.get("kernels_sha256") != sha:
            return {"traffic": None, "traffic_note": "committed ncu capture is of another revision of amb_kernels.cu"}
        return {"traffic": ent["dram_bytes_per_launch"], "traffic_source": ent.get("source")}
    except Exception as e:      # noqa: BLE001
        return {"traffic": None, "traffic_note": "profiles/scan_traffic.json unreadable (%s)" % type(e).__name__}


if __name__ == "__main__":
    main()
