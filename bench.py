#!/usr/bin/env python
"""bench.py -- RX unpack + TX pack throughput of the SoapySX IQ sample path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one RX block (S32_LE I2S frames -> CF32) and one TX block (CF32 -> I2S frames
with clamp/truncate/flag bits) of 2^27 frames each per GPU: 1 GiB in and 1 GiB out per
conversion, the 1 GiB point of BASELINE config 5's sweep (1 MB - 4 GB per block) and ~8x the
L2, so every byte comes from and goes to HBM.  (Measured: back-to-back launches at the 4 GiB
point sustain the same GB/s within 1 %; --log2-frames 29 selects it.)  Blocks are independent, so ranks shard them with no collective
on the data path ("weak" scaling); NCCL only gathers the output checksums afterwards.

The JSON line carries
  value     Msamples/s, whole job, inputs resident in HBM (CUDA events, max over ranks)
  e2e       the same metric through the host-buffer C-ABI entry points (pinned host in,
            pinned host out, both PCIe copies inside the timed region)
  roofline  achieved HBM GB/s of the dominant kernel vs MEASURED_PEAKS.json
  cpu_baseline  the reference's own converters (oracle/_ref) timed on this box's host cores

`--impl reference` times only the reference's CPU converters, on all host threads.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "rx_unpack+tx_pack throughput"
UNIT = "Msamples/s"
SEED = 0x53581255
THR2 = 1.0e-6  # (1e-3)^2, the driver's default TX-enable threshold (SoapySX.cpp:767-773)
BYTES_PER_FRAME = 16  # 8 read + 8 written, RX and TX alike (SURVEY.md section 8(d))


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ---------------------------------------------------------------------------------------------
# The plugin call: readStream + timed writeStream through the flat sxh_* harness.  The same
# function drives the product module (SoapySXB200, CUDA converters) and -- for the CPU arm, the
# only place bench.py touches oracle/ -- the unmodified reference driver built in oracle/_ref.
# ---------------------------------------------------------------------------------------------
RATE = 600000.0            # the SX1255's highest sample rate (SoapySX.cpp:196-206)
RING = 65536               # frames in the I2S DMA ring (SoapySX.cpp:464)
REF_PLUGIN = ROOT / "oracle" / "_ref" / "libsx_ref.so"


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def capture_table(seed):
    """One ring of synthetic I2S frames: the stand-in's capture signal is this table, repeated
    (snd_pcm_readi is then one copy out of the ring, as it is on a sound card)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    return rng.integers(-2**31, 2**31, size=2 * RING, dtype=np.int64).astype(np.int32)


class PluginStreams:
    """D independent driver=sx devices, one caller thread each; a step is readStream(n) followed by
    writeStream(n, HAS_TIME, that block's time + 3n frames) on every device (the repeater
    iteration of example/linear_repeater.py:50-71 with an identity process()), n = frames / D.
    `kind`: "pageable" (a numpy array, what the reference's callers pass), "pin" (the same with the
    stream argument pin=1) or "pinned" (memory from sxgpu_malloc_host; product only)."""

    def __init__(self, harness, frames, nstreams, kind="pageable", dev_args="", ctx=None, seed=SEED):
        import numpy as np
        from sxxcvr_b200 import plugin
        self.plugin, self.h, self.kind, self.ctx = plugin, harness, kind, ctx
        self.n = max(1, frames // nstreams)
        self.devs, self.rx, self.tx, self.bufs, self.addrs, self.pinned = [], [], [], [], [], []
        table = capture_table(seed)
        period = min(self.n, RING)
        pin = ", pin=1" if kind == "pin" else ""
        for k in range(nstreams):
            d = harness.device("driver=sx" + dev_args)
            d.set_rate(RATE)
            rx = d.setup(plugin.RX, args=f"period={period}{pin}")
            tx = d.setup(plugin.TX, args=f"period={period}{pin}")
            d.activate(rx), d.activate(tx)
            d.sink_limit(0)                         # the played frames are not kept: only timing matters
            d.capture_table(table.ctypes.data, RING)
            if kind == "pinned":
                addr = ctx.malloc_host(8 * self.n)
                self.pinned.append(addr)
                buf = None
            else:
                buf = np.ones(2 * self.n, np.float32)   # written once, so every page exists
                addr = buf.ctypes.data
            self.devs.append(d), self.rx.append(rx), self.tx.append(tx), self.bufs.append(buf), self.addrs.append(addr)
        self.lat_ns = int(round(3 * self.n * 1e9 / RATE))

    def run(self, iters, warmup=1):
        """Seconds per step: every stream thread times its own `iters` pairs natively; the step time
        is the slowest thread's."""
        secs = [0.0] * len(self.devs)
        gate = threading.Barrier(len(self.devs))

        def work(k):
            d = self.devs[k]
            if warmup:
                d.bench_pairs(self.rx[k], self.tx[k], self.addrs[k], self.n, warmup, self.lat_ns)
            gate.wait()
            secs[k] = d.bench_pairs(self.rx[k], self.tx[k], self.addrs[k], self.n, iters, self.lat_ns)

        if len(self.devs) == 1:
            work(0)
        else:
            ts = [threading.Thread(target=work, args=(k,)) for k in range(len(self.devs))]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        return max(secs) / iters

    def close(self):
        for d in self.devs:
            d.close()
        for addr in self.pinned:
            self.ctx.free_host(addr)
        self.devs, self.bufs = [], []


def reference_harness():
    """The unmodified reference driver (oracle/_ref), or None where it was never built."""
    from sxxcvr_b200 import plugin
    return plugin.Harness(REF_PLUGIN) if REF_PLUGIN.exists() else None


def load_cpu_converters():
    """(kind, rx, tx) bare converters: oracle/_ref (the unmodified reference, kind 'reference') if it
    was built, else the plain-C restatement (kind 'port')."""
    P, S = C.c_void_p, C.c_size_t
    if REF_PLUGIN.exists():
        lib = C.CDLL(str(REF_PLUGIN))
        rx, tx, kind = lib.sxref_convert_rx_buffer, lib.sxref_convert_tx_buffer, "reference"
    else:
        port = ROOT / "oracle" / "libsx_oracle.so"
        if not port.exists():
            subprocess.run(["make", "-C", str(ROOT / "oracle"), "libsx_oracle.so"], check=True, capture_output=True)
        lib = C.CDLL(str(port))
        rx, tx, kind = lib.sxo_convert_rx_buffer, lib.sxo_convert_tx_buffer, "port"
    rx.argtypes, rx.restype = [P, S, P, S, S], None
    tx.argtypes, tx.restype = [P, S, P, S, S, C.c_float], None
    return kind, rx, tx


class CpuConverters:
    """The bare converter loops split across host threads (ctypes releases the GIL): used when the
    reference driver itself could not be built, and as an extra row beside the plugin figure."""

    def __init__(self, frames: int, threads: int):
        import numpy as np
        self.kind, self.rx, self.tx = load_cpu_converters()
        self.frames, self.threads = frames, threads
        rng = np.random.default_rng(SEED)
        self.i2s = rng.integers(-2**31, 2**31, size=2 * frames, dtype=np.int64).astype(np.int32)
        self.cf = np.empty(2 * frames, np.float32)
        self.txin = (rng.random(2 * frames, dtype=np.float32) * 1.98 - 0.99).astype(np.float32)
        self.out = np.empty(2 * frames, np.int32)
        per = (frames + threads - 1) // threads
        self.slices = [(t * per, min(per, frames - t * per)) for t in range(threads) if t * per < frames]

    def _run(self, fn):
        if len(self.slices) == 1:
            fn(*self.slices[0])
            return
        ts = [threading.Thread(target=fn, args=s) for s in self.slices]
        for t in ts:
            t.start()
        for t in ts:
            t.join()

    def step(self):
        a, b, c, d = self.i2s.ctypes.data, self.cf.ctypes.data, self.txin.ctypes.data, self.out.ctypes.data
        self._run(lambda off, n: self.rx(a, off, b, off, n))
        self._run(lambda off, n: self.tx(c, off, d, off, n, THR2))

    def time_steps(self, steps: int, warmup: int):
        for _ in range(warmup):
            self.step()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        return (time.perf_counter() - t0) / steps


def cpu_plugin_arm(frames, threads, steps, warmup):
    """The reference driver's readStream + writeStream on `threads` host threads (one device per
    thread: a SoapySX device converts on its caller's thread, so this is how it uses them all),
    `frames` per direction per step in total.  Returns (kind, seconds per step, description)."""
    h = reference_harness()
    if h is None:
        arm = CpuConverters(frames, threads)
        return arm.kind, arm.time_steps(steps, warmup), "bare converter loops (the reference driver was not built here)"
    streams = PluginStreams(h, frames, threads)
    try:
        sec = streams.run(steps, warmup)
    finally:
        streams.close()
    return "reference", sec, (f"unmodified SoapySX readStream + timed writeStream over the ALSA stand-in, {threads} device(s) on "
                              f"{threads} thread(s), {streams.n} frames per call, pageable caller buffers")


def run_reference_arm(args, rank: int):
    if rank != 0:
        return
    threads = host_threads()
    frames = 1 << args.log2_frames
    kind, sec, what = cpu_plugin_arm(frames, threads, args.steps, args.warmup)
    value = 2 * frames / sec / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
        "config": workload_config(args, per_gpu_frames=frames),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"RX 2^{args.log2_frames} + TX 2^{args.log2_frames} frames per step: {what}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


def workload_config(args, per_gpu_frames):
    return {
        "workload": "SoapySX RX convert (S32_LE I2S -> CF32) + TX convert (CF32 -> S32_LE I2S, clamp/trunc/flag bits), "
                    f"one block each per step per GPU (BASELINE config 5, {8 * per_gpu_frames / 2**30:g} GiB-per-block point)",
        "frames_per_block": per_gpu_frames, "blocks_per_step_per_gpu": 2,
        "bytes_per_frame": BYTES_PER_FRAME, "tx_threshold2": THR2,
        "cache": f"each buffer is {8 * per_gpu_frames / 2**20:g} MiB, inputs >> 126 MB L2, so no flush is needed",
        "parallelism": f"independent blocks sharded over {args.gpus} GPU(s), no data-path collective",
    }


# ---------------------------------------------------------------------------------------------
# Clock sampling during the timed region
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and throttle reasons of one GPU, sampled in-process through NVML every
    few milliseconds between start() and stop() (the timed region lasts tens of milliseconds,
    too short for `nvidia-smi -lms`, which is kept as the fallback)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
    SMI_FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                  "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                  "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, pci_bus_id: str | None = None, period_s: float = 0.002):
        self.gpu_index, self.period_s = gpu_index, period_s
        self.samples, self.power, self.mask = [], [], 0
        self.stop_flag = threading.Event()
        self.thread = self.proc = self.nvml = self.handle = None
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(pci_bus_id.encode()) if pci_bus_id else None
            except Exception:
                self.handle = None
            if self.handle is None:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.power.append(n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
                self.mask |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass
            self.stop_flag.wait(self.period_s)

    def start(self):
        if self.nvml:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.lines = []
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.SMI_FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l.strip()) for l in self.proc.stdout], daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            reasons = sorted(name for bit, name in self.REASONS.items() if self.mask & bit)
            return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.sm_max,
                    "sm_min_mhz": min(self.samples) if self.samples else None,
                    "power_w_max": max(self.power) if self.power else None, "samples": len(self.samples),
                    "reasons": reasons, "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvml, no nvidia-smi"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, state in zip(names, parts[4:8]):
                if state.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi"}


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def measured_peak():
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


DUMP_FRAMES = 1 << 21  # frames kept per output: 16 MiB of CF32 + 32 MiB of I2S words as float64


def dump_frames(frames: int):
    """The frames --dump-outputs keeps of a block: all of them (None) up to DUMP_FRAMES, else the
    same seeded, sorted sample on every run, so that two builds can be compared element for element."""
    import numpy as np
    if frames <= DUMP_FRAMES:
        return None
    return np.sort(np.random.default_rng(SEED).choice(frames, DUMP_FRAMES, replace=False))


def dump_outputs(out_dir: Path, frames: int, cf, i2s_out):
    """Write what the RX and TX conversions hand back to their caller, at the frames dump_frames()
    picks: rx_cf32.npy (float32 I/Q samples) and tx_i2s.npy (the int32 I2S words as float64,
    which holds every int32 exactly)."""
    import numpy as np
    import torch
    pick = dump_frames(frames)
    if pick is not None:
        words = torch.from_numpy(np.stack([2 * pick, 2 * pick + 1], axis=1).ravel()).to(cf.device)
        cf, i2s_out = cf.index_select(0, words), i2s_out.index_select(0, words)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "rx_cf32.npy", cf.cpu().numpy().astype(np.float32))
    np.save(out_dir / "tx_i2s.npy", i2s_out.cpu().numpy().astype(np.float64))


def run_gpu_arm(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist
    from sxxcvr_b200 import Context

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sample path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    # stdout carries exactly one JSON line: keep NCCL's version/debug banner off it.
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x: float):
        if world == 1:
            return [x]
        mine = torch.tensor([x], dtype=torch.float64, device="cuda")
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        return [float(t.item()) for t in every]

    ctx = Context(local_rank)
    frames = 1 << args.log2_frames
    side = torch.cuda.Stream()  # a real stream handle: 0 would mean "the context's own stream"
    torch.cuda.set_stream(side)
    st = side.cuda_stream

    i2s_in = torch.empty(2 * frames, dtype=torch.int32, device="cuda")
    cf = torch.empty(2 * frames, dtype=torch.float32, device="cuda")
    i2s_out = torch.empty(2 * frames, dtype=torch.int32, device="cuda")
    ctx.synth_frames(i2s_in.data_ptr(), 0, frames, SEED + rank, st)  # the stubbed ADC, per-rank seed

    def rx():
        ctx.convert_rx_buffer(i2s_in.data_ptr(), 0, cf.data_ptr(), 0, frames, st)

    def tx():
        ctx.convert_tx_buffer(cf.data_ptr(), 0, i2s_out.data_ptr(), 0, frames, THR2, st)

    for _ in range(max(args.warmup, 3)):
        rx()
        tx()
    barrier()

    # ---- timed region: K steps, an event between every launch ---------------------------------
    props = torch.cuda.get_device_properties(local_rank)
    bus = None
    if all(hasattr(props, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
        bus = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
    sampler = ClockSampler(local_rank, bus)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    launches0 = ctx.counter("launches")
    barrier()
    ev[0].record(side)
    for k in range(args.steps):
        rx()
        ev[2 * k + 1].record(side)
        tx()
        ev[2 * k + 2].record(side)
    barrier()
    launches = ctx.counter("launches") - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), frames, cf, i2s_out)

    total_ms = ev[0].elapsed_time(ev[-1])
    rx_ms = [ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(args.steps)]
    tx_ms = [ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(args.steps)]
    step_ms = max_over_ranks(total_ms / args.steps)
    value = world * 2 * frames / (step_ms * 1e-3) / 1e6

    peak, peak_src = measured_peak()

    def roof(ms_list, name):
        avg = sum(ms_list) / len(ms_list)
        achieved = frames * BYTES_PER_FRAME / (avg * 1e-3) / 1e9
        return {"kernel": name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "avg_launch_ms": avg, "best_launch_ms": min(ms_list),
                "algorithmic_bytes_per_launch": frames * BYTES_PER_FRAME, "peak_source": peak_src}

    roof_rx = roof(rx_ms, "stream_convert_kernel<RxCf32, 2, 2, 256>, one tile per CTA")
    roof_tx = roof(tx_ms, "stream_convert_kernel<TxCf32, 2, 2, 256>, one tile per CTA")
    dominant = roof_tx if sum(tx_ms) >= sum(rx_ms) else roof_rx
    # DRAM bytes per launch come from an `ncu --set full` capture, which cannot run inside a timed
    # bench: the committed capture of this same launch (same kernel, same frames per launch) is
    # quoted, with its file named, and only when its launch size matches this run's.
    for name in ("r02_traffic.json", "r01_traffic.json"):
        traffic_file = ROOT / "profiles" / name
        if not traffic_file.exists():
            continue
        try:
            t = json.loads(traffic_file.read_text())
            if t.get("frames_per_launch") == frames:
                roof_rx["traffic"], roof_tx["traffic"] = t.get("rx_bytes_per_launch"), t.get("tx_bytes_per_launch")
                roof_rx["traffic_source"] = roof_tx["traffic_source"] = f"profiles/{name} (ncu --set full, one launch)"
                break
        except ValueError:
            pass

    # ---- checksums of what the timed kernels produced, gathered over NCCL ----------------------
    from sxxcvr_b200 import sharding
    stats = ctx.stats_words(i2s_out.data_ptr(), 2 * frames, 0, st)
    checks = [list(c) for c in sharding.gather_stats(stats, device="cuda")]

    # ---- sustained figure: the same step for at least --min-seconds ----------------------------
    sustained = None
    if args.min_seconds > 0:
        per_step = max(step_ms, 1e-3) * 1e-3
        batch = max(args.steps, int(0.25 * args.min_seconds / per_step) + 1)
        sampler2 = ClockSampler(local_rank, bus)
        barrier()
        sampler2.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(side)
        nsus, t_start = 0, time.perf_counter()
        while True:                      # whole batches until the wall clock says enough
            for _ in range(batch):
                rx()
                tx()
            nsus += batch
            side.synchronize()
            enough = max_over_ranks(1.0 if time.perf_counter() - t_start >= args.min_seconds else 0.0)
            if enough > 0:               # every rank runs the same number of batches
                break
        s1.record(side)
        barrier()
        sus_ms = max_over_ranks(s0.elapsed_time(s1) / nsus)
        sustained = {"value": world * 2 * frames / (sus_ms * 1e-3) / 1e6, "unit": UNIT, "steps": nsus,
                     "seconds": sus_ms * nsus * 1e-3, "ms_per_step": sus_ms,
                     "hbm_gbs_per_gpu": 2 * frames * BYTES_PER_FRAME / (sus_ms * 1e-3) / 1e9,
                     "clocks": sampler2.stop()}

    # ---- raw link: copy engines only, both directions loaded, every rank at once ----------------
    # The ceiling for anything that takes host buffers: 8 B/frame must cross each way.
    link_bytes = 256 << 20
    h_up = torch.empty(link_bytes, dtype=torch.uint8, pin_memory=True)
    h_down = torch.empty(link_bytes, dtype=torch.uint8, pin_memory=True)
    d_up = torch.empty(link_bytes, dtype=torch.uint8, device="cuda")
    d_down = torch.empty(link_bytes, dtype=torch.uint8, device="cuda")
    s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()

    def link_pass(up: bool, down: bool, reps=4):
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s_up):
                    d_up.copy_(h_up, non_blocking=True)
            if down:
                with torch.cuda.stream(s_down):
                    h_down.copy_(d_down, non_blocking=True)
        s_up.synchronize(), s_down.synchronize()
        return reps * link_bytes / (time.perf_counter() - t0) / 1e9

    link_pass(True, True, 1)
    link = {"h2d_alone_gbs": all_ranks(link_pass(True, False)), "d2h_alone_gbs": all_ranks(link_pass(False, True)),
            "both_each_way_gbs": all_ranks(link_pass(True, True))}
    del h_up, h_down, d_up, d_down

    # ---- end to end: the plugin call.  SoapySXB200::readStream + timed writeStream on host buffers,
    # the ALSA stand-in underneath, both PCIe copies and the stand-in's own copies inside the timed
    # region.  D devices on D caller threads share this rank's GPU, as D SX1255 front-ends would. ---
    from sxxcvr_b200 import plugin
    product = plugin.Harness()
    threads_here = max(1, host_threads() // max(1, env_int("LOCAL_WORLD_SIZE", world)))
    e2e_streams = args.e2e_streams or max(1, min(8, threads_here // 2))
    e2e_frames = min(1 << args.e2e_log2_frames, frames)
    bounce = max(1, threads_here // e2e_streams - 1)
    dev_args = f", gpu={local_rank}, sxgpu.bounce_threads={bounce}" + (args.e2e_dev_args and ", " + args.e2e_dev_args)
    def plugin_leg(kind):
        streams = PluginStreams(product, e2e_frames, e2e_streams, kind, dev_args, ctx, SEED + rank)
        try:
            streams.run(max(args.warmup, 3), 0)   # warm-up as a pass of its own: every rank enters the timed one together
            barrier()
            sec = streams.run(args.steps, 0)
            barrier()
            nlaunch = sum(d.counter("launches") for d in streams.devs)
        finally:
            streams.close()
        per_rank = [2 * e2e_frames / t / 1e6 for t in all_ranks(sec)]
        sec = max_over_ranks(sec)
        return {"value": world * 2 * e2e_frames / sec / 1e6, "sec": sec, "per_rank": per_rank, "launches": nlaunch}

    legs = {args.e2e_buffers: plugin_leg(args.e2e_buffers)}
    if not args.no_rows:                 # the other kinds of caller memory, same workload
        for kind in ("pinned", "pin", "pageable"):
            if kind not in legs:
                legs[kind] = plugin_leg(kind)
    head = legs[args.e2e_buffers]
    e2e_sec, e2e_value, e2e_per_rank, e2e_launches = head["sec"], head["value"], head["per_rank"], head["launches"]
    # bytes that crossed the link each way per second on this rank, against what the link carries
    e2e_link_gbs = [v * 1e6 * 8 / 1e9 for v in e2e_per_rank]
    frac_of_link = [a / b if b else None for a, b in zip(e2e_link_gbs, link["both_each_way_gbs"])]

    # ---- the same bytes through the C ABI alone (no plugin, no ALSA stand-in): D threads, each with
    # a context of its own, alternate sxgpu_convert_rx_buffer_host / _tx_buffer_host on pinned
    # buffers.  What separates this figure from the plugin leg is the stand-in's own copies (the
    # "hardware" side of the I/O model, which the reference arm pays too), not the library.
    c_abi = None
    if world == 1 and not args.no_rows:
        from sxxcvr_b200 import Context
        D, n_call, iters = e2e_streams, e2e_frames // e2e_streams, 6
        ctxs = [Context(local_rank) for _ in range(D)]
        bufs = [[c.malloc_host(8 * n_call) for _ in range(3)] for c in ctxs]
        secs, gate = [0.0] * D, threading.Barrier(D)

        def abi_work(k):
            c, (a, b, d) = ctxs[k], bufs[k]
            c.convert_rx_buffer_host(a, 0, b, 0, n_call)
            c.convert_tx_buffer_host(b, 0, d, 0, n_call, THR2)
            gate.wait()
            t0 = time.perf_counter()
            for _ in range(iters):
                c.convert_rx_buffer_host(a, 0, b, 0, n_call)
                c.convert_tx_buffer_host(b, 0, d, 0, n_call, THR2)
            secs[k] = time.perf_counter() - t0

        ts = [threading.Thread(target=abi_work, args=(k,)) for k in range(D)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for c, three in zip(ctxs, bufs):
            for ptr in three:
                c.free_host(ptr)
            c.close()
        abi_msps = D * iters * 2 * n_call / max(secs) / 1e6
        c_abi = {"value": round(abi_msps, 1), "unit": UNIT, "threads": D, "frames_per_call": n_call,
                 "frac_of_link": round(abi_msps * 1e6 * 8 / 1e9 / link["both_each_way_gbs"][0], 3),
                 "api": "sxgpu_convert_rx_buffer_host + sxgpu_convert_tx_buffer_host on sxgpu_malloc_host memory, one context per thread"}

    # ---- one stream at a time: frames per call x caller buffer, product beside the reference -----
    rows = []
    if rank == 0 and not args.no_rows:
        ref = reference_harness() if world == 1 else None
        sizes = [(256, 4000), (4096, 2000), (65536, 200), (1 << 20, 20), (min(frames, 1 << 27), 2)]
        for n, iters in sizes:
            row = {"frames_per_call": n}

            def pair_us(h, kind, extra=""):
                st_ = PluginStreams(h, n, 1, kind, extra, ctx, SEED)
                try:
                    return st_.run(iters, 1 if n > (1 << 22) else 5) * 1e6
                finally:
                    st_.close()

            one = f", gpu={local_rank}"
            row["product_pageable_us"] = pair_us(product, "pageable", one)
            row["product_pin1_us"] = pair_us(product, "pin", one)
            row["product_library_pinned_us"] = pair_us(product, "pinned", one)
            if n <= 4096:
                row["product_lowlatency1_us"] = pair_us(product, "pageable", one + ", lowlatency=1")
                row["product_lowlatency0_us"] = pair_us(product, "pageable", one + ", lowlatency=0")
            if ref is not None:
                row["reference_us"] = pair_us(ref, "pageable")
            for k in list(row):
                if k.endswith("_us"):
                    row[k.replace("_us", "_msps")] = round(2 * n / row[k], 1)
                    row[k] = round(row[k], 2)
            rows.append(row)

    # ---- small-block latency through the C ABI (period-sized calls, the reference's native regime)
    pinned = []

    def pinned_words(nwords, dtype):
        import ctypes
        addr = ctx.malloc_host(4 * nwords)
        pinned.append(addr)
        return torch.frombuffer((ctypes.c_char * (4 * nwords)).from_address(addr), dtype=dtype)

    h_i2s = pinned_words(2 * 65536, torch.int32)
    h_cf_out = pinned_words(2 * 65536, torch.float32)
    h_i2s.copy_(i2s_in[: 2 * 65536].cpu())
    small = {}
    for mode, label in ((2, "flag"), (1, "stream_sync")):
        ctx.set_option("small_mode", mode)
        for nf in (256, 4096, 65536):
            for _ in range(5):
                ctx.convert_rx_buffer_host(h_i2s.data_ptr(), 0, h_cf_out.data_ptr(), 0, nf)
            reps = 300
            a_, b_ = h_i2s.data_ptr(), h_cf_out.data_ptr()
            t0 = time.perf_counter()
            for _ in range(reps):
                ctx.convert_rx_buffer_host(a_, 0, b_, 0, nf)
            small[f"rx_host_{nf}_frames_us_per_call_{label}"] = (time.perf_counter() - t0) / reps * 1e6
    ctx.set_option("small_mode", 0)
    ctx.set_option("resident_max_frames", 4096)
    for nf in (256, 4096):
        for _ in range(5):
            ctx.convert_rx_buffer_host(h_i2s.data_ptr(), 0, h_cf_out.data_ptr(), 0, nf)
        reps = 500
        a_, b_ = h_i2s.data_ptr(), h_cf_out.data_ptr()
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.convert_rx_buffer_host(a_, 0, b_, 0, nf)
        small[f"rx_host_{nf}_frames_us_per_call_resident"] = (time.perf_counter() - t0) / reps * 1e6
    ctx.set_option("resident_max_frames", 0)

    # ---- the same workload from ONE process (sxgpu_multi_*): rank 0 alone drives every GPU of the
    # job for a few steps while the other ranks wait, so that the scaling record also holds the
    # one-process-G-contexts way of sharding (SURVEY.md section 8(e)) ------------------------------
    single = None
    if world > 1 and not args.no_rows:
        barrier()
        # The other ranks must wait on the HOST: a rank parked in an NCCL barrier keeps a kernel
        # spinning on its GPU, which is one of the GPUs being measured.
        try:
            store = dist.distributed_c10d._get_default_store()
        except Exception:
            store = None
        if rank == 0:
            if torch.cuda.device_count() >= world and store is not None:
                try:
                    sp_steps = min(args.steps, 20)
                    sec_sp, launches_sp, checks_sp = measure_single_process(world, frames, sp_steps, 3)
                    single = {"value": world * 2 * frames / sec_sp / 1e6, "unit": UNIT, "ms_per_step": sec_sp * 1e3,
                              "steps": sp_steps, "gpu_launches": launches_sp,
                              "hbm_gbs_per_gpu": 2 * frames * BYTES_PER_FRAME / sec_sp / 1e9,
                              "how": f"one process, {world} contexts and host threads (sxgpu_multi_*), wall clock with every GPU "
                                     "synchronised on both sides; the other ranks wait on the host meanwhile",
                              "checksums_match_ranks": [c[:3] for c in checks_sp] == [list(c[:3]) for c in checks]}
                except Exception as ex:          # evidence only: never take the judged line down with it
                    single = {"error": str(ex)[:200]}
            if store is not None:
                store.set("sx_single_process_leg_done", "1")
        elif store is not None:
            store.wait(["sx_single_process_leg_done"])
        barrier()

    # ---- CPU baseline beside it (rank 0, N=1 only): the reference driver on this box's cores ------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        cpu_frames = 1 << args.cpu_log2_frames
        kind, sec_all, what = cpu_plugin_arm(cpu_frames, threads, 3, 1)
        _, sec_one, what_one = cpu_plugin_arm(cpu_frames >> 2, 1, 2, 1)
        conv = CpuConverters(cpu_frames, threads)
        sec_conv = conv.time_steps(3, 1)
        cpu = {"value": 2 * cpu_frames / sec_all / 1e6, "unit": UNIT, "cores": threads, "kind": kind,
               "sample": f"3 steps of RX 2^{args.cpu_log2_frames} + TX 2^{args.cpu_log2_frames} frames: {what}",
               "single_thread": {"value": 2 * (cpu_frames >> 2) / sec_one / 1e6, "cores": 1,
                                 "sample": f"2 steps of RX+TX 2^{args.cpu_log2_frames - 2} frames: {what_one} "
                                           f"(how the reference runs: it converts on the calling thread)"},
               "bare_converters": {"value": 2 * cpu_frames / sec_conv / 1e6, "cores": threads, "kind": conv.kind,
                                   "sample": "convert_rx_buffer + convert_tx_buffer alone, no stream calls, "
                                             f"2^{args.cpu_log2_frames} frames split over {threads} threads"}}

    if rank == 0:
        info = ctx.info()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
            "config": workload_config(args, frames),
            "roofline": dominant, "roofline_rx": roof_rx, "roofline_tx": roof_tx, "sustained": sustained,
            "single_process": single,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * 8 * e2e_frames,
                    "d2h_bytes_per_step": 2 * 8 * e2e_frames, "frames_per_block": e2e_frames,
                    "ms_per_step": e2e_sec * 1e3, "gpu_launches": e2e_launches,
                    "api": "SoapySXB200::readStream + writeStream(HAS_TIME) through the sxh_* harness "
                           "(csrc/host/harness_capi.cpp), ALSA stand-in underneath",
                    "caller_buffers": {"pageable": "pageable numpy arrays, default stream arguments",
                                       "pin": "pageable numpy arrays, stream argument pin=1",
                                       "pinned": "sxgpu_malloc_host memory"}[args.e2e_buffers],
                    "streams_per_gpu": e2e_streams, "frames_per_call": e2e_frames // e2e_streams,
                    "bounce_threads_per_stream": bounce,
                    "bound": "PCIe: 8 B/frame cross the link each way per conversion",
                    "per_rank": [round(v, 1) for v in e2e_per_rank],
                    "raw_link_gbs_per_rank": {k: [round(x, 2) for x in v] for k, v in link.items()},
                    "link_gbs_each_way_per_rank": [round(v, 2) for v in e2e_link_gbs],
                    "frac_of_link": [round(v, 3) if v is not None else None for v in frac_of_link],
                    "by_caller_memory": {k: {"value": round(v["value"], 1), "ms_per_step": round(v["sec"] * 1e3, 3),
                                             "frac_of_link": [round(x * 1e6 * 8 / 1e9 / l, 3) if l else None
                                                              for x, l in zip(v["per_rank"], link["both_each_way_gbs"])]}
                                         for k, v in legs.items()},
                    "c_abi_host_calls": c_abi,
                    "plugin_rows": rows},
            "gpu_launches": launches, "clocks": clocks, "cpu_baseline": cpu, "small_blocks": small,
            "checksums": {"fields": list(sharding.STATS_FIELDS), "per_rank": checks,
                          "combined": list(sharding.combine_stats(checks)),
                          "gathered_with": "nccl all_gather" if world > 1 else "local"},
            "device": info.name.decode(), "sm_count": info.sm_count, "host_threads": host_threads(),
        }
        emit(json.dumps(line))

    del h_i2s, h_cf_out
    for addr in pinned:
        ctx.free_host(addr)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_bank_arm(args, rank: int, local_rank: int, world: int):
    """--workload bank: BASELINE config 4.  S HBM-resident stream pairs per GPU (streams sharded
    over the ranks in contiguous ranges), one step = readStream(256) on every stream followed by
    writeStream(256, HAS_TIME, rx time + 768 frames) on every stream.  Same JSON contract; there is
    no host-buffer leg because the bank exists to keep the samples off PCIe."""
    import torch
    import torch.distributed as dist
    from sxxcvr_b200 import Bank, Context, sharding

    torch.cuda.set_device(local_rank)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = Context(local_rank)
    S, P, rate = args.streams, 256, 75000.0
    lat_ns = int(round(768 * 1e9 / rate))
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    st = side.cuda_stream
    if args.repeat_variant is not None:
        ctx.set_option("bank_repeat_variant", args.repeat_variant)
    if args.ctas_per_sm is not None:
        ctx.set_option("ctas_per_sm", args.ctas_per_sm)
    bank = Bank(ctx, S, P, rate, 0.0, SEED + rank * S)          # this rank's streams: ids rank*S .. rank*S+S-1
    if args.external:
        # frames from outside: one period per stream handed in through sxgpu_bank_ingest (here once,
        # from device memory); every iteration then converts what the capture slots hold
        ext = torch.empty(S * P * 2, dtype=torch.int32, device="cuda")
        ctx.synth_frames(ext.data_ptr(), 0, S * P, SEED + rank, st)
        bank.ingest(0, S, ext.data_ptr(), st)
    cf = torch.empty(S * P * 2, dtype=torch.float32, device="cuda")

    def step():
        if args.fused:
            bank.repeat(cf.data_ptr(), lat_ns, st)      # the same iteration as one launch
        else:
            bank.read(cf.data_ptr(), st)
            bank.write(cf.data_ptr(), 4, None, lat_ns, st)

    for _ in range(max(args.warmup, 3)):
        step()
    run = step
    if args.graph:
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            step()
        run = g.replay
        run()
    barrier()
    launches0 = ctx.counter("launches")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record(side)
    for _ in range(args.steps):
        run()
    b.record(side)
    barrier()
    ms = a.elapsed_time(b) / args.steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = ctx.counter("launches") - launches0
    _, rxp, txp = bank.positions(st)
    ok = bool(((txp - rxp) == 768).all())
    ring = bank.playback(0, int(txp[0]) - P, P, st)
    stats = ctx.stats_words(cf.data_ptr(), 2 * S * P, 0, st)
    checks = [list(c) for c in sharding.gather_stats(stats, device="cuda")]
    peak, peak_src = measured_peak()
    value = world * 2 * S * P / (ms * 1e-3) / 1e6
    # separate calls on a large bank (plan + data kernels per half): the read half writes slot and CF32
    # block from registers (16 W), the write half reads the block and writes the ring (8 R + 8 W);
    # the warp-per-stream kernels of smaller banks re-read the slot too (40 B/frame)
    large_bank = S >= 16384 and S * P >= (1 << 21)      # sx::bank_is_large
    hbm_bytes = 24 if args.fused else (32 if large_bank else 40)
    traffic = None      # DRAM bytes per launch from the committed ncu capture, when it is of this shape
    traffic_source = None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.loads((ROOT / "profiles" / name).read_text()).get("bank_repeat", {})
            if args.fused and not args.external and t.get("streams") == S and t.get("frames_per_block") == P:
                traffic, traffic_source = t.get("bytes_per_launch"), f"profiles/{name} (ncu --set full, one launch)"
                break
        except (OSError, ValueError):
            pass
    if rank == 0:
        emit(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
            "config": {"workload": "BASELINE config 4: bank of HBM-resident stream pairs, per step readStream(256) + "
                                   "writeStream(256, HAS_TIME, rx time + 768 frames) on every stream",
                       "streams_per_gpu": S, "frames_per_block": P, "sample_rate": rate,
                       "cuda_graph_replay": bool(args.graph),
                       "capture": "frames handed in through sxgpu_bank_ingest" if args.external else
                                  "synthetic generator inside the kernel (stand-in for the I2S DMA)",
                       "bank_repeat_variant": ctx.get_option("bank_repeat_variant") if args.fused else None,
                       "ctas_per_sm": ctx.get_option("ctas_per_sm"),
                       "calls_per_step": "sxgpu_bank_repeat (one launch)" if args.fused
                                         else "sxgpu_bank_read + sxgpu_bank_write",
                       "parallelism": f"streams sharded over {world} GPU(s) in contiguous ranges, no data-path collective"},
            # One call: nothing is read back (the capture frames, their CF32 and I2S forms stay in
            # registers between the stages), so what must cross HBM is the three writes, 24 B/frame --
            # or 8 read + 16 written when the capture frames come from outside; the roofline is taken
            # against those.  Separate read and write calls move all 40 B/frame through HBM.
            "roofline": {"kernel": ("bank_plan_repeat_kernel + bank_repeat_data_kernel (decisions by a thread per stream, then "
                                    "capture -> RX -> TX in registers, three stores per vector; "
                                    + ("8 R + 16 W" if args.external else "24 W") + " per frame reach HBM)")
                                   if args.fused else
                                   "bank iteration, separate calls: plan + data kernels per call (read: capture and CF32 block "
                                   "written from registers, 16 W; write: 8 R + 8 W per frame)",
                         "hbm_bytes_per_frame": hbm_bytes, "bytes_moved_per_frame": 40 if args.fused or not large_bank else 32,
                         "bound": "hbm", "achieved": hbm_bytes * S * P / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": hbm_bytes * S * P / (ms * 1e-3) / 1e9 / peak,
                         "moved_gbs": (40 if args.fused or not large_bank else 32) * S * P / (ms * 1e-3) / 1e9,
                         "algorithmic_bytes_per_launch": hbm_bytes * S * P,
                         "traffic": traffic, "traffic_source": traffic_source, "peak_source": peak_src,
                         "frac_of_write_only_ceiling": hbm_bytes * S * P / (ms * 1e-3) / 1e9 / 7139.0,
                         "write_only_ceiling": "7 139 GB/s: cudaMemset of 1 GiB on this part (profiles/r01_hbm_limits.json)"},
            "e2e": None, "gpu_launches": launches if not args.graph else None, "cpu_baseline": None,
            "constant_latency_holds": ok, "last_block_nonzero": bool(ring.any()),
            "checksums": {"fields": list(sharding.STATS_FIELDS), "per_rank": checks,
                          "combined": list(sharding.combine_stats(checks))},
        }))
    bank.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_sweep_arm(args, rank: int, local_rank: int, world: int):
    """--workload sweep: BASELINE config 5's small end.  1 GiB of RX and 1 GiB of TX work per GPU
    per step as N independent blocks in ONE launch each (sxgpu_convert_*_batch, device-resident
    descriptor lists), N x size from 1024 x 1 MiB to 1 x 1 GiB.  `value` is the whole sweep's
    aggregate; `sweep` has one row per shape with its fraction of the measured HBM peak."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from sxxcvr_b200 import Context
    from sxxcvr_b200.capi import Block

    torch.cuda.set_device(local_rank)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = Context(local_rank)
    total = 1 << args.log2_frames
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    st = side.cuda_stream
    src = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    cf = torch.empty(2 * total, dtype=torch.float32, device="cuda")
    dst = torch.empty(2 * total, dtype=torch.int32, device="cuda")
    ctx.synth_frames(src.data_ptr(), 0, total, SEED + rank, st)
    peak, peak_src = measured_peak()
    rows, all_ms, launches0 = [], 0.0, ctx.counter("launches")
    for log2n in (17, 19, 21, 23, args.log2_frames):
        n = 1 << log2n
        nb = total // n
        lists = []
        for a, b, thr in ((src, cf, 0.0), (cf, dst, THR2)):
            arr = (Block * nb)(*[Block(a.data_ptr() + 8 * n * k, b.data_ptr() + 8 * n * k, n, thr, 0) for k in range(nb)])
            lists.append(torch.from_numpy(np.frombuffer(bytes(arr), dtype=np.uint8).copy()).cuda())

        def step():
            ctx.convert_batch("rx", lists[0].data_ptr(), on_device=True, max_length=n, stream=st, nblocks=nb)
            ctx.convert_batch("tx", lists[1].data_ptr(), on_device=True, max_length=n, stream=st, nblocks=nb)

        for _ in range(max(args.warmup, 3)):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for _ in range(args.steps):
            step()
        e1.record(side)
        barrier()
        ms = e0.elapsed_time(e1) / args.steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        all_ms += ms
        gbs = 2 * total * BYTES_PER_FRAME / (ms * 1e-3) / 1e9
        rows.append({"blocks_per_launch": nb, "block_bytes": 8 * n, "frames_per_block": n, "ms_per_step": ms,
                     "msamples_per_s": world * 2 * total / (ms * 1e-3) / 1e6, "hbm_gbs_per_gpu": gbs, "frac": gbs / peak})
    launches = ctx.counter("launches") - launches0
    worst = min(rows, key=lambda r: r["frac"])
    if rank == 0:
        emit(json.dumps({
            "metric": METRIC, "value": world * 2 * total * len(rows) / (all_ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": all_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
            "config": {"workload": "BASELINE config 5, small end: 1 GiB of RX + 1 GiB of TX per GPU per step as N blocks in one "
                                   "launch each (sxgpu_convert_rx_batch / _tx_batch), N x size swept; a step here = all shapes once",
                       "frames_per_step_per_gpu": 2 * total * len(rows), "bytes_per_frame": BYTES_PER_FRAME,
                       "cache": "buffers of 1 GiB >> 126 MB L2",
                       "parallelism": f"blocks sharded over {world} GPU(s), no data-path collective"},
            "roofline": {"kernel": "batch_direct_kernel (worst shape of the sweep)", "bound": "hbm",
                         "achieved": worst["hbm_gbs_per_gpu"], "peak": peak, "unit": "GB/s", "frac": worst["frac"],
                         "traffic": None, "peak_source": peak_src, "shape": f"{worst['blocks_per_launch']} x {worst['block_bytes'] >> 20} MiB"},
            "sweep": rows, "e2e": None, "gpu_launches": launches, "cpu_baseline": None}))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_group_arm(args, rank: int, local_rank: int, world: int):
    """--workload group: BASELINE config 4 with frames that come from N host-side ALSA stand-ins.
    S front-ends per GPU behind ONE group device (SoapySXB200Group): a step is readStream(256) on
    every member + writeStream(256, HAS_TIME, rx time + 768 frames) on every member, all members'
    conversions in one launch; the reference beside it is S unmodified SoapySX devices stepped
    one after the other on one thread (how one process would serve them)."""
    import torch
    import torch.distributed as dist
    from sxxcvr_b200 import plugin

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    product = plugin.Harness()
    P, rate = 256, 75000.0
    lat = int(round(768 * 1e9 / rate))
    rows = []
    for S in (64, 1024, 4096):
        with plugin.Group(product, S, f"gpu={local_rank}, threshold=0") as g:
            g.set_rate(rate)
            g.activate()
            for i in range(S):
                product.lib.sx_alsa_set_sink_limit(g.pcm(i, False), 0)
            g.bench_repeat(P, lat, 5)
            iters = max(20, min(500, 200000 // S))
            sec = g.bench_repeat(P, lat, iters) / iters
            rc, rx, tx, t = g.repeat_all(0, P, lat)
            ok = rc == 0 and bool((rx == P).all() and (tx == P).all())
            launches = 0
        row = {"members": S, "us_per_iteration": sec * 1e6, "us_per_member": sec / S * 1e6,
               "msamples_per_s": 2 * S * P / sec / 1e6, "all_members_returned_full_blocks": ok}
        rows.append(row)
    # The reference beside it: one unmodified SoapySX device's read+write pair, timed natively; a
    # process serving S front-ends with it pays that per member per period (its converters run on
    # the calling thread).
    ref_pair_us = None
    ref = reference_harness() if (rank == 0 and world == 1) else None
    if ref is not None:
        one = PluginStreams(ref, P, 1)
        try:
            ref_pair_us = one.run(5000, 50) * 1e6
        finally:
            one.close()
        for row in rows:
            row["reference_us_per_member"] = ref_pair_us
            row["reference_us_per_iteration_one_thread"] = ref_pair_us * row["members"]
    if world > 1:
        vals = [None] * world
        dist.all_gather_object(vals, rows[-1]["us_per_iteration"])
        worst_us = max(vals)
    else:
        worst_us = rows[-1]["us_per_iteration"]
    if rank == 0:
        S = rows[-1]["members"]
        emit(json.dumps({
            "metric": METRIC, "value": world * 2 * S * P / (worst_us * 1e-6) / 1e6, "unit": UNIT, "n_gpus": world,
            "steps": None, "warmup": 5, "ms_per_step": worst_us * 1e-3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
            "config": {"workload": "BASELINE config 4 through the group device: S front-ends (each its own ALSA stand-in pair) per GPU, "
                                   "per step readStream(256) + writeStream(256, HAS_TIME, +768 frames) on every member, one launch for all",
                       "members_per_gpu": S, "frames_per_block": P, "sample_rate": rate,
                       "parallelism": f"members sharded over {world} GPU(s), no data-path collective"},
            "group": rows, "e2e": {"value": world * 2 * S * P / (worst_us * 1e-6) / 1e6, "unit": UNIT,
                                   "h2d_bytes_per_step": 8 * S * P, "d2h_bytes_per_step": 16 * S * P},
            "roofline": None, "gpu_launches": None, "cpu_baseline": None}))
    if world > 1:
        dist.destroy_process_group()


def measure_single_process(G, frames, steps, warmup):
    """K steps of one RX + one TX block per GPU driven from this ONE process through
    sxgpu_multi_* (a context and a host thread per GPU).  Wall clock, every GPU synchronised on
    both sides.  Returns (seconds per step, launches, per-GPU output checksums)."""
    import torch
    from sxxcvr_b200 import Multi
    from sxxcvr_b200.capi import Block

    with Multi(list(range(G))) as m:
        bufs = []
        for g in range(G):
            dev = f"cuda:{g}"
            i2s = torch.empty(2 * frames, dtype=torch.int32, device=dev)
            cf = torch.empty(2 * frames, dtype=torch.float32, device=dev)
            out = torch.empty(2 * frames, dtype=torch.int32, device=dev)
            m.context(g).synth_frames(i2s.data_ptr(), 0, frames, SEED + g)
            bufs.append((i2s, cf, out))
        m.sync()
        rx = [Block(b[0].data_ptr(), b[1].data_ptr(), frames, 0.0, 0) for b in bufs]
        tx = [Block(b[1].data_ptr(), b[2].data_ptr(), frames, THR2, 0) for b in bufs]
        for _ in range(max(warmup, 3)):
            m.convert_rx_batch(rx)
            m.convert_tx_batch(tx)
        m.sync()
        l0 = sum(m.context(g).counter("launches") for g in range(G))
        t0 = time.perf_counter()
        for _ in range(steps):
            m.convert_rx_batch(rx)
            m.convert_tx_batch(tx)
        m.sync()
        sec = (time.perf_counter() - t0) / steps
        launches = sum(m.context(g).counter("launches") for g in range(G)) - l0
        checks = [list(m.context(g).stats_words(bufs[g][2].data_ptr(), 2 * frames, 0)) for g in range(G)]
        del bufs
    return sec, launches, checks


def run_single_process_arm(args):
    """--single-process --gpus N: the device-resident workload driven from ONE process through
    sxgpu_multi_* (one context and one host thread per GPU, SURVEY.md section 8(e)) instead of one
    rank per GPU.  Wall clock around K steps, every GPU synchronised on both sides."""
    import torch

    G = args.gpus
    if torch.cuda.device_count() < G:
        raise SystemExit(f"bench.py --single-process: {G} GPUs requested, {torch.cuda.device_count()} visible")
    frames = 1 << args.log2_frames
    sec, launches, checks = measure_single_process(G, frames, args.steps, args.warmup)
    peak, peak_src = measured_peak()
    gbs = 2 * frames * BYTES_PER_FRAME / sec / 1e9
    emit(json.dumps({
        "metric": METRIC, "value": G * 2 * frames / sec / 1e6, "unit": UNIT, "n_gpus": G, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "s32<->f32", "data": "synthetic",
        "config": dict(workload_config(args, frames),
                       parallelism=f"ONE process, {G} contexts and host threads (sxgpu_multi_*), one block per GPU per launch, no collective",
                       timing="wall clock around the timed steps, every GPU synchronised on both sides"),
        "roofline": {"kernel": "batch_direct_kernel, one 1 GiB block per GPU", "bound": "hbm", "achieved": gbs, "peak": peak,
                     "unit": "GB/s", "frac": gbs / peak, "traffic": None, "peak_source": peak_src,
                     "note": "per-GPU average over the RX+TX step, launch gaps included"},
        "e2e": None, "gpu_launches": launches, "cpu_baseline": None,
        "checksums": {"per_gpu": checks}}))


class QuietStdout:
    """stdout must carry exactly one JSON line.  Native libraries write banners to file descriptor 1
    (NCCL prints its version there when NCCL_DEBUG is set), so for the duration of the run fd 1
    points at stderr; emit() restores it for the one line that matters."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line: str):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


OUT = None


def emit(line: str):
    if OUT is not None:
        OUT.emit(line)
    else:
        print(line, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-frames", type=int, default=27, help="frames per block per GPU (2^27 = 1 GiB in)")
    ap.add_argument("--e2e-log2-frames", type=int, default=27, help="frames per block of the plugin leg (capped at --log2-frames)")
    ap.add_argument("--e2e-dev-args", default="", help="extra device arguments of the plugin leg, e.g. sxgpu.host_chunk_frames=1048576")
    ap.add_argument("--e2e-streams", type=int, default=0, help="devices (caller threads) per GPU in the plugin leg; 0 = auto")
    ap.add_argument("--e2e-buffers", default="pinned", choices=["pageable", "pin", "pinned"],
                    help="caller buffers of the headline plugin leg: sxgpu_malloc_host memory (default: the contract's "
                         "'host->device copy from pinned host memory'), pageable numpy arrays with pin=1, or plain pageable "
                         "numpy arrays (what the reference's callers pass); the other two are reported beside it")
    ap.add_argument("--min-seconds", type=float, default=1.0,
                    help="also report the device-resident figure sustained over at least this long (0 = skip)")
    ap.add_argument("--no-rows", action="store_true", help="skip the one-stream frames-per-call x buffer-kind table")
    ap.add_argument("--cpu-log2-frames", type=int, default=27, help="frames per step of the cpu_baseline sample inside the GPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="blocks", choices=["blocks", "bank", "sweep", "group"],
                    help="blocks: the judged RX+TX block workload (default); bank: BASELINE config 4 (HBM-resident streams); "
                         "sweep: config 5's block-size sweep, many blocks per launch; group: config 4 through the group "
                         "device, frames from N host ALSA stand-ins")
    ap.add_argument("--single-process", action="store_true",
                    help="drive --gpus N from ONE process (sxgpu_multi_*: a context and a host thread per GPU) instead of one rank per GPU")
    ap.add_argument("--streams", type=int, default=65536, help="--workload bank: stream pairs per GPU")
    ap.add_argument("--graph", action="store_true", help="--workload bank: replay the step from a CUDA graph")
    ap.add_argument("--repeat-variant", type=int, default=None, help="--fused: option bank_repeat_variant")
    ap.add_argument("--ctas-per-sm", type=int, default=None, help="option ctas_per_sm (persistent grids)")
    ap.add_argument("--external", action="store_true",
                    help="--workload bank: capture frames come from sxgpu_bank_ingest instead of the synthetic generator")
    ap.add_argument("--fused", action="store_true",
                    help="--workload bank: the iteration as one sxgpu_bank_repeat launch instead of read + write")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="default workload: after the timed steps, write the last step's RX and TX outputs (rank 0's, "
                         f"a fixed seeded sample of {DUMP_FRAMES} frames of larger blocks) as DIR/rx_cf32.npy and DIR/tx_i2s.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "blocks" or args.single_process):
        ap.error("--dump-outputs is implemented for the default workload only (--impl b200 --workload blocks, one rank per GPU)")

    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.single_process and args.impl != "reference":
        global OUT
        with QuietStdout() as OUT:
            run_single_process_arm(args)
        return
    if world == 1 and args.gpus > 1:
        # Launched without torchrun: re-exec under it so there is one process per GPU.
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))

    with QuietStdout() as OUT:
        if args.impl == "reference":
            run_reference_arm(args, rank)
        elif args.workload == "bank":
            run_bank_arm(args, rank, local_rank, world)
        elif args.workload == "sweep":
            run_sweep_arm(args, rank, local_rank, world)
        elif args.workload == "group":
            run_group_arm(args, rank, local_rank, world)
        else:
            run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
