#!/usr/bin/env python
"""bench.py -- QuantizedSAE forward hot path on N B200s: tokens/s, roofline, CPU baseline.

    python bench.py --gpus 1 --steps 20 --warmup 5              # headline + every BASELINE.json config (extra keys)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 5 --warmup 1       # CPU arm (oracle port of the reference, rank 0 only)
    python bench.py --config 3                                   # one config as the headline line (1..5)
    python bench.py --steps 20 --dump-outputs DIR                # also write config 1's last timed step to DIR/*.npy

Headline = BASELINE.json configs[0]: b_sae 512->32768 n_bits=4 gamma=4 k=32 forward at batch 4096 per GPU.
A "step" is one forward of the hot path over one batch of synthetic activations: x [B,512] fp32 (resident in HBM) ->
(cast + sample pre-pass + prior) -> fused tcgen05 encoder sweep + top-k -> merge + packed int4 decode ->
(values, indices) [B,k] + reconstruction [B,512], behind ONE C-ABI call (qsae_bsae_forward). Weights are pre-packed
(one-time cost, not in the step). Rows are independent, so N GPUs shard the batch with replicated weights and no
collective on the data path ("scaling": "weak"). The default run also measures the other BASELINE configs and attaches
them under "configs" (config 5, the dictionary-sharded 2^20 variant, when N > 1). Prints ONE JSON line on rank 0.
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

D, H, N_BITS, GAMMA = 512, 32768, 4, 4.0
E2E_CHUNK = int(os.environ.get("QSAE_E2E_CHUNK", "8192"))   # largest row chunk of the host-buffer pipeline
METRIC = "b_sae 512->32768 4-bit fwd tokens/s"
UNIT = "tokens/s"
L2_BYTES = 126 * 1024 * 1024


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="all", choices=["all", "1", "2", "3", "4", "5"],
                    help="all (default): config 1 is the headline line and configs 2-4 (5 when --gpus > 1) are attached "
                         "under 'configs'; N: only that BASELINE.json config, as the headline line")
    ap.add_argument("--batch", type=int, default=4096, help="rows per GPU per step of config 1 (BASELINE configs[0]: 4096)")
    ap.add_argument("--k", type=int, default=32, help="latents kept per row (model.k = k / 32768)")
    ap.add_argument("--cpu-batch", type=int, default=4096, help="rows per step of the CPU arm / cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch the kernels directly instead of replaying the step from CUDA graphs (default: graphs for "
                         "batches up to 16384 rows, where launch gaps are a visible share of the step)")
    ap.add_argument("--streams", type=int, default=2,
                    help="batches in flight: consecutive steps alternate between this many CUDA streams, so the small kernels "
                         "around one batch's sweep (prior, merge + decode, tail) overlap the neighbouring batches' (1 = one "
                         "stream, every step strictly after the previous one; reported beside the headline either way)")
    ap.add_argument("--quick", action="store_true", help="config 1 only: skip the attached configs")
    ap.add_argument("--heavy-tail", action="store_true",
                    help="SURVEY 8d heavy-tail variant of the inputs: 8 of the 512 dimensions scaled by 20")
    ap.add_argument("--hidden", type=int, default=2 ** 20, help="dictionary size of config 5 (dictionary-sharded)")
    ap.add_argument("--transport", default="p2p", choices=["nccl", "p2p"],
                    help="config 5: candidate / partial exchange through NCCL collectives or CUDA IPC peer memory")
    # accepted for compatibility with round-1 command lines
    ap.add_argument("--variant", default=None, choices=[None, "batch-sharded", "dict-sharded"])
    ap.add_argument("--graph", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of config 1, write what its last step returned (latent values and indices, "
                         "reconstruction) as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.variant == "dict-sharded":
        a.config = "5"
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.config not in ("all", "1")):
        ap.error("--dump-outputs writes the outputs of config 1 on the B200 (--impl b200, --config all or 1)")
    return a


HEAVY_TAIL = False   # set from --heavy-tail


def workload_name(batch, k):
    return (f"b_sae input_dim=512 hidden_dim=32768 n_bits=4 gamma=4.0 k={k} forward, "
            f"synthetic Pythia-70m-shaped activations{' (heavy-tail variant: 8 dims x 20)' if HEAVY_TAIL else ''}, "
            f"batch {batch} per GPU")


# ---------------------------------------------------------------------------------------------
# synthetic weights / inputs (SURVEY.md 8d config 1): xavier encoder rounded to bf16-representable
# fp32, polarised (+-110) decoder logits, N(0,1) decoder bias, N(0,1) x rounded to bf16-representable
# ---------------------------------------------------------------------------------------------
def make_weights(torch, device, seed=0, hidden=H):
    g = torch.Generator(device=device).manual_seed(seed)
    bound = (6.0 / (hidden + D)) ** 0.5
    We = ((torch.rand((hidden, D), device=device, generator=g) * 2 - 1) * bound).bfloat16().float()
    be = torch.zeros(hidden, device=device)
    logits = torch.where(torch.rand((hidden, D * N_BITS), device=device, generator=g) < 0.5, 110.0, -110.0)
    bd = torch.randn(D, device=device, generator=g)
    return We, be, logits.float().contiguous(), bd


def make_x(torch, device, batch, seed):
    g = torch.Generator(device=device).manual_seed(1000 + seed)
    x = torch.randn((batch, D), device=device, generator=g)
    if HEAVY_TAIL:       # a few outlier channels, like the residual stream of a transformer
        x[:, torch.arange(8, device=device) * 61 + 5] *= 20.0
    return x.bfloat16().float()


def n_rotating(batch):
    """Distinct input buffers so that the inputs of consecutive steps exceed the L2 (x always comes from HBM; the
    weights stay L2-resident, as they do in a steady-state serving loop)."""
    per = batch * D * 4
    return max(3, min(64, -(-int(1.1 * L2_BYTES) // per)))


# ---------------------------------------------------------------------------------------------
# clocks sampler (NVML / nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every 2 ms from a thread (a timed
    region is only tens of milliseconds long), nvidia-smi -lms as the fallback when pynvml is unavailable."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.index])
            except (ValueError, IndexError):
                pass
        return self.index

    def start(self):
        try:
            import pynvml as N

            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.sm_max = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            bits = {"hw_slowdown": N.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": N.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": N.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": N.nvmlClocksThrottleReasonSwPowerCap}

            def poll():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                        r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for name, bit in bits.items():
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                    time.sleep(0.002)

            self._nvml = N
            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self._nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self._physical_index())], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self._nvml is not None:
            self._stop.set()
            self._thread.join(timeout=1.0)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml, 2 ms polling"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            p = [t.strip() for t in s.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(self.NAMES, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


# ---------------------------------------------------------------------------------------------
# CPU arm: op-for-op port of the reference forward (oracle/), torch CPU, all host threads
# ---------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and the pinned host buffers it allocates afterwards) to the CPUs next to its GPU: the
    local_cpulist of the GPU's PCI device. Returns a description for the JSON line."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = Path(f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0")
        cpus = (path / "local_cpulist").read_text().strip()
        node = (path / "numa_node").read_text().strip()
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        allowed = os.sched_getaffinity(0)
        use = ids & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
        return {"numa_node": node, "local_cpulist": cpus, "bound": bool(use and use != allowed)}
    except Exception as e:  # no sysfs entry in this container, single-node host, ...
        return {"numa_node": None, "bound": False, "note": f"{type(e).__name__}"}


def cpu_forward_times(batch, k, steps, warmup):
    import torch

    from oracle import qsae_oracle as O

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cpu = torch.device("cpu")
    We, be, logits, bd = make_weights(torch, cpu)
    x = make_x(torch, cpu, batch, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.bsae_forward_dense_port_torch(x, We, be, logits, bd, n_bits=N_BITS, gamma=GAMMA, k=k)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times, torch.get_num_threads()


def cpu_baseline_block(batch, k, steps, warmup):
    times, cores = cpu_forward_times(batch, k, steps, warmup)
    med, best = statistics.median(times), min(times)
    return {"value": batch / med, "unit": UNIT, "cores": cores, "kind": "port",
            "best": batch / best, "median_s_per_forward": med, "best_s_per_forward": best,
            "sample": f"{batch} rows x {len(times)} timed forwards ({warmup} warm-up) of the same workload, median; "
                      f"oracle/qsae_oracle.bsae_forward_dense_port_torch == the reference's op sequence "
                      f"(sae/binary.py:91-103), pinned to the reference's stored outputs by tests/test_oracle_golden.py; "
                      f"torch CPU, {cores} threads"}, times


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, min(args.warmup, 3))
    cb, times = cpu_baseline_block(args.cpu_batch, args.k, steps, warmup)
    mean_s = sum(times) / len(times)
    rate = args.cpu_batch / mean_s
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": warmup, "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.cpu_batch, args.k), "cpu_rows_per_step": args.cpu_batch,
                   "note": (f"every step is one full forward of {args.cpu_batch} rows"
                            + (" (the configs[0] batch, the same rows per step as the B200 arm)" if args.cpu_batch == 4096 else
                               " (a bounded sample: the B200 arm's step has 4096 rows; the metric is a per-token rate)")
                            + "; value = mean over the timed steps, cpu_baseline carries median and best")},
        "cpu_baseline": dict(cb, value=rate),
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ---------------------------------------------------------------------------------------------
# timing helpers
# ---------------------------------------------------------------------------------------------
def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return {"burst": float(j.get("bf16_tflops", 1590.0)), "sustained": float(j.get("bf16_tflops_sustained", j.get("bf16_tflops", 1400.0))),
                "hbm_gbs": float(j["hbm_gbs"]), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md; of fallback)"}


def pick_peak(peaks, region_ms, clocks):
    """Burst figure for a timed region of well under a second at full SM clock with no power cap (the regime
    MEASURED_PEAKS.json's best-of-10 GEMM was taken in), the sustained figure otherwise; both fractions are printed."""
    full_clock = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and clocks["sm_mhz"] >= 0.97 * clocks["sm_max_mhz"])
    capped = bool(clocks and "sw_power_cap" in (clocks.get("reasons") or []))
    if region_ms < 1000.0 and full_clock and not capped:
        return "burst", ("bf16_tflops (burst): the timed region is %.0f ms at the full SM clock with no power cap; the sustained "
                         "figure (1327 MHz under the power cap) is printed beside it" % region_ms)
    return "sustained", "bf16_tflops_sustained: long or power-capped timed region"


class Timer:
    def __init__(self, torch, dist, device):
        self.torch, self.dist, self.device = torch, dist, device

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], device=self.device, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def streams(self, n, always=False):
        """The timer's worker streams (created once: the library keeps one workspace per stream)."""
        if n <= 1 and not always:
            return []
        pool = self.__dict__.setdefault("_workers", [])
        while len(pool) < n:
            pool.append(self.torch.cuda.Stream(device=self.device))
        return pool[:n]

    def on_streams(self, fn, streams):
        """fn(i) issued on streams[i % S] (S batches in flight); no streams: fn itself."""
        if not streams:
            return fn
        torch = self.torch

        def run(i):
            with torch.cuda.stream(streams[i % len(streams)]):
                return fn(i)
        return run

    def fork(self, streams):
        """Event on the current stream that every worker stream waits for (start of a timed region)."""
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        for st in streams:
            st.wait_event(e)
        return e

    def join(self, streams):
        """The current stream waits for everything issued on the worker streams; -> event behind it."""
        cur = self.torch.cuda.current_stream()
        for st in streams:
            ev = self.torch.cuda.Event()
            ev.record(st)
            cur.wait_event(ev)
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def time(self, fn, steps, warmup, streams=()):
        """fn(i) enqueues step i (on its own stream when `streams` are in use: see on_streams / graphs). -> ms per step:
        CUDA events on the launching stream around the fork / join of the worker streams, barrier + synchronize on both
        sides, max over ranks."""
        for i in range(warmup):
            fn(i)
        self.join(streams)
        self.barrier()
        e0 = self.fork(streams)
        for i in range(steps):
            fn(i)
        e1 = self.join(streams)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def graphs(self, fn, n, n_streams=1):
        """One CUDA graph per rotating input: fn(i) captured for i in [0, n) (ctypes launches go to torch's current
        stream; outputs and the library's per-(device, stream) workspaces live in the graphs' pool). With n_streams > 1
        graph i is captured on, and always replayed on, stream i % n_streams (n is trimmed to a multiple of it), so
        consecutive steps are in flight together on different streams.
        -> (replay(i), launches per step counted by the library during capture, graphs, worker streams)"""
        torch = self.torch
        from quantizedsae_b200 import _lib as L

        gs = []
        per_step = 0
        pool = torch.cuda.graph_pool_handle()
        S = max(1, n_streams)
        caps = self.streams(S, always=True)
        n = max(S, n - n % S)
        for i in range(n):
            g = torch.cuda.CUDAGraph()
            c0 = L.launch_count()
            with torch.cuda.graph(g, pool=pool, stream=caps[i % S]):
                out = fn(i)
            per_step = L.launch_count() - c0
            gs.append((g, out))
        if S == 1:
            return (lambda i: gs[i % n][0].replay()), per_step, gs, []

        def replay(i):
            j = i % n
            with torch.cuda.stream(caps[j % S]):
                gs[j][0].replay()
        return replay, per_step, gs, caps


def oracle_rows_check(O, np, x_rows, We, be, k, vals, idx):
    """In-run parity spot check: top-k indices of a few rows against the numpy oracle (bit-exact index sets, order
    included, values to 1e-5)."""
    z = O.encode_pre(x_rows, We, be)
    rv, ri = O.topk_rows(z, k)
    return bool(np.array_equal(idx, ri) and np.all(np.abs(vals - rv) <= 1e-5 * np.maximum(1.0, np.abs(rv))))


# ---------------------------------------------------------------------------------------------
# config 1: b_sae (headline)
# ---------------------------------------------------------------------------------------------
def bench_bsae(args, T, rank, world, device, B, k, steps, warmup, want_e2e=True, want_roofline=True, exact_too=True,
               graph=True, keep_last=False):
    import numpy as np
    import torch

    from quantizedsae_b200 import _lib as L

    lib = L.load()
    We, be, logits, bd = make_weights(torch, device)
    w_bf16 = L.cast_bf16(We)
    sample = L.prepare_sample(w_bf16, be)
    packed, _, gap = L.pack_bitplanes(logits, D, N_BITS)
    assert gap == 0.0
    del logits
    qstep = GAMMA / 2 ** (N_BITS - 1)
    n_in = n_rotating(B)
    xs = [make_x(torch, device, B, s + 100 * rank) for s in range(n_in)]

    def step(i, exact=False):
        x = xs[i % n_in]
        vals, idx, _, recon = L.bsae_forward(x, w_bf16, We if exact else None, be, k, packed, N_BITS, qstep, bd, exact=exact,
                                             sample=sample)
        return vals, idx, recon

    for i in range(max(3, warmup)):
        step(i)
    T.barrier()

    # ---- parity spot check against the numpy oracle (64 rows of input 0)
    from oracle import qsae_oracle as O

    rows = np.arange(0, B, max(1, B // 64))[:64]
    v, ix, rec = step(0)
    torch.cuda.synchronize()
    parity = oracle_rows_check(O, np, xs[0][rows].cpu().numpy(), We.cpu().numpy(), be.cpu().numpy(), k,
                               v[rows].cpu().numpy(), ix[rows].cpu().numpy())

    # ---- headline: device-resident steps, graph replay for small batches, args.streams batches in flight
    use_graph = graph and not args.no_graph and B <= 16384
    S = max(1, args.streams)
    launches_per_step = None
    sampler = ClockSampler(device.index)
    if use_graph:
        run, launches_per_step, keep, streams = T.graphs(step, n_in, S)
    else:
        streams = T.streams(S)
        run = T.on_streams(step, streams)
    for i in range(warmup):
        run(i)
    T.join(streams)
    T.barrier()
    if rank == 0:
        sampler.start()
    c0 = L.launch_count()
    T.barrier()
    e0 = T.fork(streams)
    for i in range(steps):
        last = run(i)
    e1 = T.join(streams)
    T.barrier()
    elapsed_ms = T.max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    if keep_last:
        # a graph replay returns nothing: the last step's outputs are the ones its graph was captured with
        last_step = [t.cpu().numpy() for t in (keep[(steps - 1) % len(keep)][1] if use_graph else last)]
    launches = launches_per_step * steps if use_graph else L.launch_count() - c0
    ms = elapsed_ms / steps
    out = {"value": world * B / (ms * 1e-3), "ms_per_step": ms, "elapsed_ms": elapsed_ms, "clocks": clocks, "gpu_launches": int(launches),
           "launch": ("CUDA graph replay, one graph per rotating input" if use_graph else "direct launches") +
                     (f"; {S} batches in flight: consecutive steps alternate between {S} streams, every step's kernels are inside "
                      f"the timed region (fork / join events on the timing stream)" if S > 1 else "; one stream"),
           "parity_checked": parity, "n_inputs": n_in, "batch": B, "k": k, "streams": S}
    if keep_last:
        out["last_step"] = last_step
    if S > 1:
        # the pipelined steps produce the same bits as a lone step, and the strictly serial number is reported beside it
        if use_graph:
            torch.cuda.synchronize()
            same = all(torch.equal(a, b) for a, b in zip((v, ix, rec), keep[0][1]))
            one, _, keep1, _ = T.graphs(step, n_in, 1)
        else:
            with torch.cuda.stream(streams[0]):
                o2 = step(0)
            torch.cuda.synchronize()
            same = all(torch.equal(a, b) for a, b in zip((v, ix, rec), o2))
            one = step
        ms1 = T.time(one, steps, warmup)
        out["pipelined_results_identical"] = bool(same)
        out["single_stream"] = {"value": world * B / (ms1 * 1e-3), "unit": UNIT, "ms_per_step": ms1,
                                "note": "the same steps on one stream: each batch's first kernel starts after the previous batch's last"}
        if use_graph:
            del keep1

    # ---- the same step launched directly (no graph), and in exact mode
    if use_graph:
        out["direct_launch_ms"] = T.time(step, max(5, min(steps, 50)), 3)
    if exact_too:
        ems1 = T.time(lambda i: step(i, True), max(5, min(steps, 20)), 3)
        st2 = T.streams(S)
        ems = T.time(T.on_streams(lambda i: step(i, True), st2), max(5, min(steps, 20)), 3, st2) if st2 else ems1
        out["exact_mode"] = {"value": world * B / (ems * 1e-3), "unit": UNIT, "ms_per_step": ems, "single_stream_ms": ems1,
                             "note": "fp32 re-scoring of k + 16 tensor-core candidates from the fp32 weights (module default; valid for "
                                     f"arbitrary fp32 operands); direct launches, {S} batches in flight"}

    # ---- roofline of the dominant kernel: CUDA events around the sweep launch only, direct launches
    if want_roofline:
        n_k = max(5, min(steps, 50))
        k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_k)]
        stage_ms = None
        for i in range(n_k):
            k_ev[i][0].record(); k_ev[i][1].record()           # materialise the handles before handing them over
            L.check(lib.qsae_set_encode_kernel_events(k_ev[i][0].cuda_event, k_ev[i][1].cuda_event))
            step(i)
        L.check(lib.qsae_set_encode_kernel_events(None, None))
        torch.cuda.synchronize()
        out["kernel_ms"] = statistics.median(a.elapsed_time(b) for a, b in k_ev)

    # ---- e2e: the reference-facing C-ABI call with HOST buffers (H2D + kernels + D2H inside)
    if want_e2e:
        out["e2e"] = e2e_bsae(args, T, world, device, B, k, We, be, bd, xs)
    return out


def e2e_bsae(args, T, world, device, B, k, We, be, bd, xs):
    import torch

    from quantizedsae_b200 import _lib as L

    lib = L.load()
    plan = C.c_void_p()
    g = torch.Generator(device=device).manual_seed(5)
    logits2 = torch.where(torch.rand((H, D * N_BITS), device=device, generator=g) < 0.5, 110.0, -110.0).float()
    L.check(lib.qsae_bsae_plan_create(We.data_ptr(), be.data_ptr(), logits2.data_ptr(), bd.data_ptr(), H, D, N_BITS,
                                      C.c_float(GAMMA), k, min(E2E_CHUNK, B), C.byref(plan)))
    del logits2
    try:
        depth = 4   # steps in flight: step i + 1's H2D copy overlaps step i's kernels and step i - 1's D2H copy
        hx = [xs[j % len(xs)].cpu().pin_memory() for j in range(depth)]
        hv = [torch.empty((B, k), dtype=torch.float32).pin_memory() for _ in range(depth)]
        hi = [torch.empty((B, k), dtype=torch.int32).pin_memory() for _ in range(depth)]
        hr = [torch.empty((B, D), dtype=torch.float32).pin_memory() for _ in range(depth)]
        # steady-state throughput of a stream of host batches: the pipeline's fill and drain (one H2D + one step of kernels
        # + one D2H, ~0.5 ms) are inside the timed region, so it is timed over at least 100 steps (reported as "steps")
        n = max(100, args.steps)

        def sync_call(i):
            j = i % depth
            L.check(lib.qsae_bsae_forward_host(plan, hx[j].data_ptr(), B, hv[j].data_ptr(), hi[j].data_ptr(), hr[j].data_ptr()))

        for i in range(3):
            sync_call(i)
        T.barrier()
        t0 = time.perf_counter()
        for i in range(n):
            sync_call(i)
        sync_s = T.max_over_ranks(time.perf_counter() - t0)
        res = {"unit": UNIT, "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": B * k * 8 + B * D * 4, "steps": n,
               "synchronous": {"value": world * B * n / sync_s, "ms_per_step": sync_s / n * 1e3,
                               "api": "qsae_bsae_forward_host: returns when the step's results are in host memory"}}
        if hasattr(lib, "qsae_bsae_submit_host"):
            tickets = [None] * depth

            def wait(j):
                if tickets[j] is not None:
                    L.check(lib.qsae_bsae_wait_host(plan, tickets[j]))
                    tickets[j] = None

            def submit(i):
                j = i % depth
                wait(j)                                    # the slot's previous step has landed in its host buffers
                t = C.c_int(0)
                L.check(lib.qsae_bsae_submit_host(plan, hx[j].data_ptr(), B, hv[j].data_ptr(), hi[j].data_ptr(),
                                                  hr[j].data_ptr(), C.byref(t)))
                tickets[j] = t.value

            for i in range(depth):
                submit(i)
            for j in range(depth):
                wait(j)
            T.barrier()
            t0 = time.perf_counter()
            for i in range(n):
                submit(i)
            for j in range(depth):
                wait(j)
            pipe_s = T.max_over_ranks(time.perf_counter() - t0)
            res["value"] = world * B * n / pipe_s
            res["ms_per_step"] = pipe_s / n * 1e3
            res["api"] = (f"qsae_bsae_submit_host / qsae_bsae_wait_host: {depth} steps in flight (pinned host x in; values, indices, "
                          f"reconstruction to pinned host); every step's H2D and D2H copies are inside the timed region")
            # opt-in narrow host formats: bf16 x in (exact here: x is bf16-representable), bf16 reconstruction out
            L.check(lib.qsae_bsae_plan_set_io(plan, 1, 1))
            hxb = [h.bfloat16().pin_memory() for h in hx]
            hrb = [torch.empty((B, D), dtype=torch.bfloat16).pin_memory() for _ in range(depth)]

            def submit16(i):
                j = i % depth
                wait(j)
                t = C.c_int(0)
                L.check(lib.qsae_bsae_submit_host(plan, hxb[j].data_ptr(), B, hv[j].data_ptr(), hi[j].data_ptr(),
                                                  hrb[j].data_ptr(), C.byref(t)))
                tickets[j] = t.value

            for i in range(depth):
                submit16(i)
            for j in range(depth):
                wait(j)
            T.barrier()
            t0 = time.perf_counter()
            for i in range(n):
                submit16(i)
            for j in range(depth):
                wait(j)
            s16 = T.max_over_ranks(time.perf_counter() - t0)
            res["bf16_io"] = {"value": world * B * n / s16, "ms_per_step": s16 / n * 1e3, "h2d_bytes_per_step": B * D * 2,
                              "d2h_bytes_per_step": B * k * 8 + B * D * 2,
                              "note": "qsae_bsae_plan_set_io(x bf16, recon bf16): opt-in, halves the PCIe bytes of x and of the reconstruction"}
            L.check(lib.qsae_bsae_plan_set_io(plan, 0, 0))
        else:
            res["value"] = res["synchronous"]["value"]
            res["ms_per_step"] = res["synchronous"]["ms_per_step"]
            res["api"] = res["synchronous"]["api"]
        return res
    finally:
        lib.qsae_bsae_plan_destroy(plan)


def roofline_block(peaks, flops_per_launch, kernel_ms, step_flops, step_ms, region_ms, clocks, kernel, traffic_key=None):
    which, why = pick_peak(peaks, region_ms, clocks)
    achieved = flops_per_launch / (kernel_ms * 1e-3) / 1e12
    step_tf = step_flops / (step_ms * 1e-3) / 1e12
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists() and traffic_key:
        traffic = json.loads(tp.read_text()).get(traffic_key)
    return {"bound": "tensor", "kernel": kernel, "achieved": achieved, "peak": peaks[which], "unit": "TFLOP/s",
            "frac": achieved / peaks[which], "frac_burst": achieved / peaks["burst"], "frac_sustained": achieved / peaks["sustained"],
            "traffic": traffic, "algorithmic_flops_per_launch": flops_per_launch, "kernel_ms": kernel_ms,
            "step": {"achieved": step_tf, "frac_burst": step_tf / peaks["burst"], "frac_sustained": step_tf / peaks["sustained"],
                     "note": "whole step (all launches) against the same peaks: algorithmic encoder flops / step time"},
            "peak_source": f"{peaks['source']}; denominator rule: {why}"}


# ---------------------------------------------------------------------------------------------
# configs 2-4 through the drop-in modules (the public API), device-resident
# ---------------------------------------------------------------------------------------------
def module_e2e(torch, T, world, model_fn, xs, B, out_bytes):
    """Module-level end-to-end: pinned host x -> device -> forward -> reconstruction back to pinned host."""
    hx = [x.cpu().pin_memory() for x in xs[:2]]
    dst = None
    n = 5
    for it in range(2 + n):
        if it == 2:
            T.barrier()
            t0 = time.perf_counter()
        xd = hx[it % 2].to(xs[0].device, non_blocking=True)
        recon = model_fn(xd)
        if dst is None:
            dst = torch.empty(recon.shape, dtype=recon.dtype).pin_memory()
        dst.copy_(recon, non_blocking=True)
        torch.cuda.synchronize()
    s = T.max_over_ranks(time.perf_counter() - t0)
    return {"value": world * B * n / s, "unit": UNIT, "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": out_bytes, "steps": n,
            "api": "nn.Module forward: pinned host x -> .to(device) -> model(x) -> reconstruction copied to pinned host"}


def bench_baseline(args, T, rank, world, device, peaks, steps, warmup, B=65536):
    import numpy as np
    import torch

    import quantizedsae_b200 as Q
    from oracle import qsae_oracle as O

    torch.manual_seed(0)
    with torch.device(device):
        m = Q.BaselineSparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
    m.eval()
    m.return_dense, m.exact = False, False
    n_in = n_rotating(B)
    xs = [make_x(torch, device, B, 50 + s + 100 * rank) for s in range(n_in)]
    streams = T.streams(args.streams)
    with torch.no_grad():
        ms1 = T.time(lambda i: m(xs[i % n_in]), steps, max(3, warmup))
        ms = T.time(T.on_streams(lambda i: m(xs[i % n_in]), streams), steps, max(3, warmup), streams) if streams else ms1
        lat, recon = m(xs[0])
        rows = np.arange(0, B, B // 32)[:32]
        parity = oracle_rows_check(O, np, xs[0][rows].cpu().numpy(), m.encoder[0].weight.detach().cpu().numpy(),
                                   m.encoder[0].bias.detach().cpu().numpy(), 32, lat.values[rows].cpu().numpy(),
                                   lat.indices[rows].cpu().numpy())
        m.exact = True
        ems = T.time(lambda i: m(xs[i % n_in]), max(3, steps // 2), 2)
        m.exact = False
        e2e = module_e2e(torch, T, world, lambda xd: m(xd)[1], xs, B, B * D * 4)
    flops = 2.0 * B * H * D
    tf = flops / (ms * 1e-3) / 1e12
    return {"workload": f"baseline_sae 512->32768 top_k=32 forward, bf16-representable operands, batch {B} per GPU (BASELINE configs[1])",
            "value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": B,
            "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                         "frac_sustained": tf / peaks["sustained"], "algorithmic_flops_per_step": flops,
                         "note": "whole forward (encoder sweep + merge + fp32 row-gather decode) against the encoder's 2 B D H flops"},
            "launch": f"direct launches, {max(1, args.streams)} batches in flight on as many streams", "single_stream_ms": ms1,
            "exact_mode": {"value": world * B / (ems * 1e-3), "ms_per_step": ems},
            "e2e": e2e, "parity_checked": parity, "latents_out": "sparse (values, indices); dense [B,H] not written"}


def bench_tsae(args, T, rank, world, device, peaks, steps, warmup, B=4096):
    import numpy as np
    import torch

    import quantizedsae_b200 as Q
    from oracle import qsae_oracle as O

    torch.manual_seed(0)
    with torch.device(device):
        m = Q.TernarySparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
        # kaiming init gives an all-zero ternary matrix (SURVEY 8d config 3): N(0, 0.4824^2) => 30 % non-zeros
        m.decoder.weight.copy_(0.4824 * torch.randn(m.decoder.weight.shape, device=device,
                                                    generator=torch.Generator(device=device).manual_seed(3)))
    m.eval()
    m.exact = False
    n_in = n_rotating(B)
    xs = [make_x(torch, device, B, 70 + s + 100 * rank) for s in range(n_in)]
    launch = "direct launches"
    with torch.no_grad():
        ms = T.time(lambda i: m(xs[i % n_in]), steps, max(3, warmup))
        if B <= 16384 and not args.no_graph:
            n_g = min(n_in, 4)        # every graph keeps its own dense h [B, H] (0.5 GB at B = 4096): 4 inputs rotate = 34 MB of x + 2 GB of h > L2
            replay, _, keep, _ = T.graphs(lambda i: m(xs[i % n_g]), n_g)
            ms_direct, ms = ms, T.time(replay, steps, max(3, warmup))
            launch = f"CUDA graph replay of model(x), {n_g} graphs rotating (direct launches: {ms_direct:.4f} ms)"
            del keep
            if args.streams > 1:
                replay, _, keep, streams = T.graphs(lambda i: m(xs[i % n_g]), n_g, args.streams)
                ms_one, ms = ms, T.time(replay, steps, max(3, warmup), streams)
                launch += f"; {args.streams} batches in flight on as many streams (one stream: {ms_one:.4f} ms)"
                del keep
        h, recon = m(xs[0])
        rows = np.arange(0, B, B // 16)[:16]
        We, be = m.encoder[0].weight.detach().cpu().numpy(), m.encoder[0].bias.detach().cpu().numpy()
        href, rref = O.tsae_forward(xs[0][rows].cpu().numpy(), We, be, m.decoder.weight.detach().cpu().numpy())
        rms = float(np.sqrt(np.mean(rref.astype(np.float64) ** 2))) + 1e-30
        parity = bool(np.allclose(h[rows].cpu().numpy(), href, rtol=1e-4, atol=1e-5) and
                      np.allclose(recon[rows].cpu().numpy(), rref, rtol=8e-3, atol=8e-3 * rms))
        m.exact = True
        ems = T.time(lambda i: m(xs[i % n_in]), max(3, steps // 4), 2)
        m.exact = False
        e2e = module_e2e(torch, T, world, lambda xd: m(xd)[1], xs, B, B * D * 4)
    flops = 4.0 * B * H * D
    tf = flops / (ms * 1e-3) / 1e12
    return {"workload": f"t_sae 512->32768 dense ReLU latents + dense ternary decoder (30 % non-zero), batch {B} per GPU, batch-sharded (BASELINE configs[2])",
            "value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": B, "launch": launch,
            "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                         "frac_sustained": tf / peaks["sustained"], "algorithmic_flops_per_step": flops,
                         "note": "two chained GEMMs, 4 B D H flops; the dense fp32 h [B,H] (a return value) is written to HBM"},
            "exact_mode": {"value": world * B / (ems * 1e-3), "ms_per_step": ems},
            "e2e": e2e, "parity_checked": parity,
            "parity_tolerance": "h 1e-4; recon 8e-3 (fast mode: one bf16 rounding of h before the decoder GEMM)"}


def bench_qsae(args, T, rank, world, device, peaks, steps, warmup):
    import numpy as np
    import torch

    import quantizedsae_b200 as Q
    from oracle import qsae_oracle as O

    out = {}
    torch.manual_seed(0)
    with torch.device(device):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
        m.encoder[0].bias.fill_(-0.543)          # mean total L0 ~ 33.6 (SURVEY 8d config 4)
        for w in (m.decoder.weight, m.decoder.weight_mirror):
            # sigmoid(w) >= 0.5 in fp32 depends on the expf implementation for |w| < ~1e-7 (DESIGN.md 3, edge (a)):
            # keep the synthetic decoder logits away from that band so the in-run oracle check is meaningful
            w.copy_(torch.where(w.abs() < 1e-6, torch.full_like(w, 1e-6), w))
    m.eval()
    m.exact = False
    for B in (4096, 65536):
        n_in = n_rotating(B)
        xs = [make_x(torch, device, B, 90 + s + 100 * rank) for s in range(n_in)]
        with torch.no_grad():
            ms = T.time(lambda i: m(xs[i % n_in]), steps, max(3, warmup))
            groups, levels = m(xs[0])
            entry = {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": B, "path": m.last_path,
                     "mean_l0": float(sum(float(g) for g in groups)), "launch": "direct launches"}
            if B <= 16384 and not args.no_graph and m.last_path == "sparse":
                # steady state has no host synchronisation (regime known, overflow flag lazy): the forward is capturable
                replay, _, keep, _ = T.graphs(lambda i: m(xs[i % n_in]), n_in)
                gms = T.time(replay, steps, max(3, warmup))
                entry["direct_launch_ms"] = ms
                entry.update({"value": world * B / (gms * 1e-3), "ms_per_step": gms,
                              "launch": "CUDA graph replay of model(x), one graph per rotating input"})
                ms = gms
                del keep
                if args.streams > 1:
                    sq = args.streams + 1      # measured: q_sae's longer tail (cast + level decoder) fills a third stream (149 -> 142 us)
                    replay, _, keep, streams = T.graphs(lambda i: m(xs[i % n_in]), n_in, sq)
                    gms = T.time(replay, steps, max(3, warmup), streams)
                    entry.update({"value": world * B / (gms * 1e-3), "ms_per_step": gms, "single_stream_ms": ms,
                                  "launch": entry["launch"] + f"; {sq} batches in flight on as many streams"})
                    ms = gms
                    del keep
            elif args.streams > 1 and m.last_path == "sparse":
                streams = T.streams(args.streams)
                pms = T.time(T.on_streams(lambda i: m(xs[i % n_in]), streams), steps, max(3, warmup), streams)
                entry.update({"value": world * B / (pms * 1e-3), "ms_per_step": pms, "single_stream_ms": ms,
                              "launch": f"direct launches, {args.streams} batches in flight on as many streams"})
                ms = pms
            if B == 4096:
                rows = np.arange(0, B, B // 16)[:16]
                lg, res, _act = O.qsae_forward(xs[0][rows].cpu().numpy(), m.encoder[0].weight.detach().cpu().numpy(),
                                         m.encoder[0].bias.detach().cpu().numpy(), m.decoder.weight.detach().cpu().numpy(),
                                         m.decoder.weight_mirror.detach().cpu().numpy(), m.decoder.bias.detach().cpu().numpy(),
                                         n_bits=4, abs_range=4.0)
                ok = True
                for i in range(4):
                    rms = float(np.sqrt(np.mean(np.asarray(res[i], dtype=np.float64) ** 2))) + 1e-30
                    ok = ok and bool(np.allclose(levels[i][rows].cpu().numpy(), res[i], rtol=1e-4, atol=1e-4 * rms))
                entry["parity_checked"] = ok
                entry["e2e"] = module_e2e(torch, T, world, lambda xd: m(xd)[1][-1], xs, B, B * D * 4)
            tf = 2.0 * B * H * D / (ms * 1e-3) / 1e12
            entry["roofline"] = {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                                 "frac_sustained": tf / peaks["sustained"]}
        out[f"sparse_b{B}"] = entry
        del xs
    # untrained encoder (~50 % active): the dense level-GEMM path
    with torch.no_grad():
        m.encoder[0].bias.zero_()
        B = 4096
        xs = [make_x(torch, device, B, 95 + s + 100 * rank) for s in range(3)]
        m.dense_mode = "always"
        ms = T.time(lambda i: m(xs[i % 3]), max(3, steps // 2), 2)
        tf = 4.0 * B * H * D / (ms * 1e-3) / 1e12
        out["dense_untrained_b4096"] = {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": B, "path": m.last_path,
                                        "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                                                     "frac_sustained": tf / peaks["sustained"],
                                                     "note": "encoder GEMM + per-level decoder GEMMs = 4 B D H flops"}}
    out["workload"] = ("q_sae Matryoshka 512->32768 top_k=32 n_bits=4 abs_range=4 forward (BASELINE configs[3]): encoder bias -0.543 "
                       "(mean L0 ~ 34, sparse level decoder) and untrained / ~50 % active (dense level GEMMs)")
    return out


def bench_soft_decode(args, T, device, peaks, B=4096, k=65):
    """The reference's actual b_sae forward semantics: soft bits sigmoid(w) (sae/binary.py:26-38) -> fp32 soft rows."""
    import torch

    from quantizedsae_b200 import _lib as L

    g = torch.Generator(device=device).manual_seed(11)
    rows = torch.randn((H, D), device=device, generator=g)
    vals = torch.randn((B, k), device=device, generator=g)
    idx = torch.randint(0, H, (B, k), device=device, generator=g, dtype=torch.int32)   # every row its own k dictionary rows
    bd = torch.randn(D, device=device, generator=g)
    ms = T.time(lambda i: L.decode_rows_f32(vals, idx, rows, H, D, 0.5, bd), 20, 3)
    nbytes = B * (k * (D * 4 + 8) + D * 4)
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"workload": f"soft-bit decode (decode_rows_f32 over the cached fp32 soft dictionary, 67 MB), B={B}, k={k}",
            "ms": ms, "algorithmic_bytes_per_token": k * (D * 4 + 8) + D * 4,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                         "note": "algorithmic bytes; the 67 MB dictionary is largely L2-resident, so values above the HBM peak are L2 hits"}}


def bench_bsae_soft(args, T, rank, world, device, peaks, steps, warmup, B=4096):
    """The reference's literal b_sae forward semantics (SURVEY D4): soft bits sigmoid(w) on NON-polarised logits,
    reference-default k = 65, through the nn.Module API (decode_mode 'auto' resolves to the fp32 soft dictionary)."""
    import numpy as np
    import torch

    import quantizedsae_b200 as Q
    from oracle import qsae_oracle as O

    torch.manual_seed(0)
    with torch.device(device):
        m = Q.BinarySAE(D, H, GAMMA, N_BITS)
    g = torch.Generator(device=device).manual_seed(31)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
        m.decoder.weight.copy_(torch.randn(m.decoder.weight.shape, device=device, generator=g) * 1.5)
        m.decoder.bias.copy_(torch.randn(D, device=device, generator=g))
    m.eval()
    m.return_dense = False
    n_in = n_rotating(B)
    xs = [make_x(torch, device, B, 40 + s + 100 * rank) for s in range(n_in)]
    out = {}
    with torch.no_grad():
        for exact in (False, True):
            m.exact = exact
            m(xs[0])
            assert m.decoder.resolved_mode() == "soft"
            ms1 = T.time(lambda i: m(xs[i % n_in]), steps, max(3, warmup))
            streams = T.streams(args.streams)
            ms = T.time(T.on_streams(lambda i: m(xs[i % n_in]), streams), steps, max(3, warmup), streams) if streams else ms1
            out["exact" if exact else "fast"] = {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "single_stream_ms": ms1}
        m.exact = False
        lat, recon, pol = m(xs[0])
        rows = np.arange(0, B, B // 16)[:16]
        k = lat.indices.shape[1]
        rv, ri, rr, rp = O.bsae_forward(xs[0][rows].cpu().numpy(), m.encoder[0].weight.detach().cpu().numpy(),
                                        m.encoder[0].bias.detach().cpu().numpy(), m.decoder.weight.detach().cpu().numpy(),
                                        m.decoder.bias.detach().cpu().numpy(), n_bits=N_BITS, gamma=GAMMA, k=k, mode="soft")
        rms = float(np.sqrt(np.mean(rr.astype(np.float64) ** 2))) + 1e-30
        parity = bool(np.array_equal(lat.indices[rows].cpu().numpy(), ri) and
                      np.allclose(recon[rows].cpu().numpy(), rr, rtol=1e-4, atol=1e-4 * rms) and abs(float(pol) / rp - 1) < 1e-5)
    tf = 2.0 * B * H * D / (out["fast"]["ms_per_step"] * 1e-3) / 1e12
    return {"workload": f"b_sae 512->32768 n_bits=4 forward with SOFT bits (non-polarised logits, fp32 soft dictionary 67 MB), "
                        f"reference-default k={k}, batch {B}, nn.Module API", "value": out["fast"]["value"], "unit": UNIT,
            "ms_per_step": out["fast"]["ms_per_step"], "single_stream_ms": out["fast"]["single_stream_ms"], "batch": B,
            "exact_mode": out["exact"], "parity_checked": parity,
            "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                         "frac_sustained": tf / peaks["sustained"]}}


def bench_training_side(args, T, device, peaks, B=4096):
    """SURVEY 8f-4: the training-side kernels at the config-1 shape (soft logits, reference-default k = 65): one b_sae
    trainer step (forward + loss + backward through the sparse autograd node, training/trainer.py:143-151), its
    HBM-bound logit-gradient pass, and one RigL update_mask over the [512, 32768] ternary decoder."""
    import torch

    import quantizedsae_b200 as Q
    from quantizedsae_b200 import _lib as L

    g = torch.Generator(device=device).manual_seed(21)
    m = Q.BinarySAE(D, H, 4.0, 4).to(device)
    with torch.no_grad():
        m.decoder.weight.copy_(torch.randn((H, D * 4), device=device, generator=g) * 1.5)
    m.autograd, m.return_dense, m.exact = True, False, True
    xs = [torch.randn((B, D), device=device, generator=g) for _ in range(4)]

    def step(i):
        x = xs[i % len(xs)]
        m.zero_grad(set_to_none=True)
        _, recon, pol = m(x)
        (0.5 * torch.nn.functional.mse_loss(recon, x) + 0.1 * pol).backward()

    step_ms = T.time(step, 10, 3)
    logits = m.decoder.weight.detach()
    G = torch.randn((H, D), device=device, generator=g)
    grad = torch.empty_like(logits)
    lg_ms = T.time(lambda i: L.bsae_logit_grad(logits, G, D, 4, 0.1, grad, False), 20, 3)
    lg_bytes = H * D * 4 * (4 + 1 + 4)            # logits in, G in, gradient out
    k = 65
    vals = torch.randn((B, k), device=device, generator=g)
    idx = torch.randint(0, H, (B, k), device=device, generator=g, dtype=torch.int32)
    gr = torch.randn((B, D), device=device, generator=g)
    dst = torch.zeros((H, D), device=device)
    sc_ms = T.time(lambda i: L.rows_scatter_add(vals, idx, gr, dst, 0.5), 20, 3)
    sc_bytes = B * k * D * 4                      # one 16-byte reduction per 4 gradient entries
    w = torch.randn((D, H), device=device, generator=g) * 0.4824
    mask = torch.ones_like(w)
    L.rigl_init_mask(w, mask, int(0.7 * w.numel()))
    a_mean = torch.rand(H, device=device, generator=g) + 1e-3
    d_mean = torch.randn(D, device=device, generator=g)
    n = int(0.1 * 0.3 * w.numel())
    rg_ms = T.time(lambda i: L.rigl_update_mask(w, mask, a_mean, d_mean, n, n), 10, 3)
    rg_bytes = w.numel() * 4 * (6 * 2 + 2 + 2 + 4)   # 6 histogram passes + drop apply + tie count over (w, mask); apply reads both, writes both
    hbm = peaks["hbm_gbs"]

    def rl(nbytes, ms, note):
        gbs = nbytes / (ms * 1e-3) / 1e9
        return {"ms": ms, "algorithmic_bytes": nbytes, "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                                                                      "frac": gbs / hbm, "note": note}}

    return {"workload": f"training-side kernels (SURVEY 8f-4) at 512->32768 n_bits=4, soft logits, k={k}, B={B}",
            "bsae_trainer_step": {"ms": step_ms, "tokens_per_s": B / (step_ms * 1e-3),
                                  "what": "forward (exact encoder + top-k, soft-row decode, pack for polarize_loss) + 0.5 mse + 0.1 polarize "
                                          "+ backward to all four parameter gradients"},
            "bsae_logit_grad_kernel": rl(lg_bytes, lg_ms, "streams logits + d/d int_w in, gradient out: 604 MB"),
            "rows_scatter_add_kernel": rl(sc_bytes, sc_ms, "atomic traffic B k D 4 bytes into a 67 MB matrix (L2-resident)"),
            "rigl_update_mask": rl(rg_bytes, rg_ms, "17 launches: two 3-pass radix selects over 16.7 M entries + apply passes")}


# ---------------------------------------------------------------------------------------------
# config 5: b_sae 512 -> 2^20, dictionary split over the ranks (strong scaling)
# ---------------------------------------------------------------------------------------------
def dict_sharded_parity(m, x, latents, rows, rank, world, dist, k, n_rows=8):
    """In-run oracle check of the dictionary-sharded forward (config 5): for a few rows of rank 0's row block every rank
    scores ITS shard with the numpy oracle (fp32 pre-activations, local top-k, hard int4 rows of the winners it owns),
    rank 0 merges the candidates (value desc, global index asc), sums the partial reconstructions and compares with what
    the CUDA path returned. -> bool on rank 0 (None elsewhere)."""
    import numpy as np

    from oracle import qsae_oracle as O

    plan = m.plan
    R = list(range(0, min(n_rows, rows.shape[0])))                    # rank 0 owns the first rows of the batch
    xr = x[R].cpu().numpy()
    lin = m.encoder[0]
    z = O.encode_pre(xr, lin.weight.detach().cpu().numpy(), lin.bias.detach().cpu().numpy())
    lv, li = O.topk_rows(z, min(k, z.shape[1]))
    a, b = plan.latent_range()
    gi = latents.indices[R].cpu().numpy().astype(np.int64)            # the CUDA path's global winners (same on all ranks)
    gv = latents.values[R].cpu().numpy()
    mine = (gi >= a) & (gi < b)
    loc = np.where(mine, gi - a, 0)
    need = np.unique(loc[mine])
    logit_rows = m.decoder.weight.detach()[need.tolist() if len(need) else [0]].cpu().numpy()
    iw = np.zeros((b - a, m.input_dim), dtype=np.float32)
    if len(need):
        iw[need] = O.dequant_hard(logit_rows, m.n_bits).astype(np.float32)
    q = m.decoder.quantization_step if hasattr(m.decoder, "quantization_step") else m.quantization_step
    partial = O.decode_rows(np.where(mine, gv, np.float32(0)), loc, iw, q, None).astype(np.float64)
    payload = (lv, li.astype(np.int64) + a, partial)
    gathered = [None] * world
    if world > 1:
        dist.all_gather_object(gathered, payload)
    else:
        gathered = [payload]
    if rank != 0:
        return None
    v = np.concatenate([g[0] for g in gathered], axis=1)
    i = np.concatenate([g[1] for g in gathered], axis=1)
    order = np.lexsort((i, -v.astype(np.float64)), axis=1)[:, :k]
    ri = np.take_along_axis(i, order, 1)
    rv = np.take_along_axis(v, order, 1)
    ok = bool(np.array_equal(gi, ri) and np.all(np.abs(gv - rv) <= 1e-5 * np.maximum(1.0, np.abs(rv))))
    recon = sum(g[2] for g in gathered) + m.decoder.bias.detach().cpu().numpy().astype(np.float64)
    got = rows[R].cpu().numpy()
    rms = float(np.sqrt(np.mean(recon ** 2))) + 1e-30
    return ok and bool(np.allclose(got, recon, rtol=1e-4, atol=1e-4 * rms))


def bench_dict_sharded(args, T, rank, world, device, peaks, steps, warmup, ks=(32, 2097), B=4096):
    import torch

    from quantizedsae_b200.sharded import DictionaryShardedBinarySAE

    Hh = args.hidden
    dist = T.dist
    with torch.device(device):
        m = DictionaryShardedBinarySAE(D, Hh, GAMMA, N_BITS, rank=rank, world_size=world)
    g = torch.Generator(device=device).manual_seed(100 + rank)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
        hs = m.plan.shard_latents
        for a in range(0, hs, 65536):          # polarised logits, generated in slices
            b = min(hs, a + 65536)
            m.decoder.weight[a:b] = torch.where(torch.rand((b - a, D * N_BITS), device=device, generator=g) < 0.5, 110.0, -110.0)
        m.decoder.bias.copy_(torch.randn(D, device=device, generator=torch.Generator(device=device).manual_seed(7)))
    m.eval()
    m.exact = False
    gx = torch.Generator(device=device).manual_seed(1000)     # the same x on every rank (replicated input)
    xs = [torch.randn((B, D), device=device, generator=gx).bfloat16().float() for _ in range(3)]
    out = {"workload": f"b_sae input_dim=512 hidden_dim={Hh} n_bits=4 gamma=4.0 forward, batch {B} replicated, dictionary split over "
                       f"{world} GPU(s) (BASELINE configs[4]); strong scaling", "hidden": Hh, "batch": B, "n_gpus": world}
    flops_per_gpu = 2.0 * B * (Hh // world) * D
    for transport in ([args.transport] if world == 1 else sorted({args.transport, "nccl"})):
        m.transport = transport
        for k in ks:
            m.k = k / Hh
            with torch.no_grad():
                ms = T.time(lambda i: m(xs[i % 3]), steps, max(3, warmup))
                # compute-only share: the same step with the exchanges skipped is not expressible (the merge needs the
                # gathered lists), so time the local stage alone -- encoder sweep + local top-k of this shard
                local_ms = T.time(lambda i: m.local_candidates(xs[i % 3]), max(3, steps // 2), 2) if hasattr(m, "local_candidates") else None
            if getattr(m, "_peer", None) is not None:
                m._peer.check()
            parity = None
            if k <= 64:      # oracle spot check of this transport (the k = 2097 variant shares every kernel but the large-k select, covered by the tests)
                with torch.no_grad():
                    lat, rws, _ = m(xs[0])
                torch.cuda.synchronize()
                parity = dict_sharded_parity(m, xs[0], lat, rws, rank, world, dist, k)
            tf = flops_per_gpu / (ms * 1e-3) / 1e12
            k_send = getattr(m, "last_k_send", None)
            entry = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "k": k, "transport": transport,
                     "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "frac_burst": tf / peaks["burst"],
                                  "frac_sustained": tf / peaks["sustained"],
                                  "note": "per-GPU sweep flops over the WHOLE step time (exchange + merge + decode included): lower bound of the kernel's fraction"}}
            if parity is not None:
                entry["parity_checked"] = parity
            if local_ms is not None:
                entry["local_ms"] = local_ms
                entry["comm_ms"] = max(0.0, ms - local_ms)
                entry["comm_note"] = "comm_ms = step - (local sweep + local top-k): exchange of candidates, global merge, owner decode, reduce of partials"
            if k_send:
                entry["k_send"] = k_send
                entry["nvlink_bytes_per_step_per_gpu"] = B * k_send * 8 * (world - 1) + (B // max(world, 1)) * D * 4 * (world - 1)
            out[f"{transport}_k{k}"] = entry
            if k > 224:
                # the same step with the winners returned as a set (ordered_latents = False): the sort of 2097 winners per
                # row is most of the large-k selection's instructions and the reference only uses the set (sae/binary.py:96-99)
                m.ordered_latents = False
                with torch.no_grad():
                    ums = T.time(lambda i: m(xs[i % 3]), steps, max(3, warmup))
                m.ordered_latents = True
                if getattr(m, "_peer", None) is not None:
                    m._peer.check()
                out[f"{transport}_k{k}_unordered"] = {"value": B / (ums * 1e-3), "unit": UNIT, "ms_per_step": ums, "k": k,
                                                      "transport": transport, "note": "SparseLatents hold each row's k winners as a set"}
    return out


# ---------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch

    from quantizedsae_b200 import _lib as L

    dist = None
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=device)
    lib = L.load()
    L.check(lib.qsae_check_device())
    T = Timer(torch, dist, device)
    peaks = load_peaks()
    steps, warmup = args.steps, max(3, args.warmup)
    cfg = args.config
    out = None

    if cfg in ("all", "1"):
        B, k = args.batch, args.k
        r = bench_bsae(args, T, rank, world, device, B, k, steps, warmup, keep_last=bool(args.dump_outputs))
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, *r.pop("last_step"))
        flops = 2.0 * B * H * D
        out = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(B, k), "baseline_config": "BASELINE.json configs[0]",
                       "launch": r["launch"],
                       "latents_out": "sparse (values, indices) [B,k]; dense [B,H] not written",
                       "l2": f"{r['n_inputs']} rotating input buffers of {B * D * 4 / 1e6:.1f} MB = {r['n_inputs'] * B * D * 4 / 1e6:.0f} MB > 126 MB L2: "
                             f"x comes from HBM every step; the prepared weights (33.5 MB bf16 encoder + 8.4 MB int4 dictionary) stay "
                             f"L2-resident as in a steady-state serving loop",
                       "weights": "pre-packed once (bf16 encoder, sampled rows, int4 dictionary); not in the step",
                       "precision": "synthetic x and encoder weights are bf16-representable (SURVEY 8d config 1), so the bf16 "
                                    "tensor-core products are exact and the result equals the fp32 reference up to fp32 "
                                    "accumulation order; int4 decode accumulates exact integers. exact_mode = same step with "
                                    "fp32 re-scoring from the fp32 weights (valid for arbitrary fp32 operands)",
                       "parallelism": f"batch-sharded x{world}, replicated weights, no collective",
                       "parity_checked": r["parity_checked"], "numa": numa},
            "roofline": roofline_block(peaks, flops, r["kernel_ms"], flops, r["ms_per_step"], r["elapsed_ms"], r["clocks"],
                                       "encode_topk_kernel<8,0,3> (range schedule over cta_group::2 pairs, one CTA per SM)" if B < 16384 else "encode_topk_kernel<8,0,1>",
                                       "encode_topk_kernel_dram_bytes_per_launch_b4096" if B == 4096 else "encode_topk_kernel_dram_bytes_per_launch"),
            "e2e": r["e2e"], "gpu_launches": r["gpu_launches"], "clocks": r["clocks"],
            "exact_mode": r["exact_mode"],
        }
        for key in ("single_stream", "pipelined_results_identical"):
            if key in r:
                out[key] = r[key]
        if "direct_launch_ms" in r:
            out["direct_launches"] = {"value": world * B / (r["direct_launch_ms"] * 1e-3), "unit": UNIT, "ms_per_step": r["direct_launch_ms"],
                                      "note": "the same step without CUDA graphs (one qsae_bsae_forward call per step)"}
        if cfg == "all" and not args.quick:
            extra = {}
            # the round-1 headline shape (largest single-GPU batch of the configs) and the reference-default k = 65
            for name, (b2, k2) in {"1_b65536_k32": (65536, 32), "1_b4096_k65": (4096, 65), "1_b65536_k65": (65536, 65)}.items():
                r2 = bench_bsae(args, T, rank, world, device, b2, k2, max(5, steps // 2), 3, want_e2e=(b2 == 65536 and k2 == 32),
                                want_roofline=True, exact_too=(k2 == 32))
                f2 = 2.0 * b2 * H * D
                extra[name] = {"workload": workload_name(b2, k2), "value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"],
                               "launch": r2["launch"], "parity_checked": r2["parity_checked"],
                               "roofline": roofline_block(peaks, f2, r2["kernel_ms"], f2, r2["ms_per_step"], r2["elapsed_ms"], r2["clocks"],
                                                          "encode_topk_kernel", "encode_topk_kernel_dram_bytes_per_launch" if b2 == 65536 else None)}
                for key in ("exact_mode", "e2e", "single_stream", "pipelined_results_identical"):
                    if key in r2:
                        extra[name][key] = r2[key]
                torch.cuda.empty_cache()
            extra["2_baseline_sae"] = bench_baseline(args, T, rank, world, device, peaks, max(5, steps // 2), 3)
            torch.cuda.empty_cache()
            extra["3_t_sae"] = bench_tsae(args, T, rank, world, device, peaks, max(5, steps // 2), 3)
            torch.cuda.empty_cache()
            extra["4_q_sae"] = bench_qsae(args, T, rank, world, device, peaks, max(5, steps // 2), 3)
            torch.cuda.empty_cache()
            extra["soft_bit_decode"] = bench_soft_decode(args, T, device, peaks)
            extra["1_soft_bits_b4096_k65"] = bench_bsae_soft(args, T, rank, world, device, peaks, max(5, steps // 2), 3)
            torch.cuda.empty_cache()
            extra["f4_training_side"] = bench_training_side(args, T, device, peaks)
            torch.cuda.empty_cache()
            if world > 1:
                extra["5_dict_sharded"] = bench_dict_sharded(args, T, rank, world, device, peaks, max(5, steps // 2), 3)
            out["configs"] = extra
    elif cfg == "2":
        e = bench_baseline(args, T, rank, world, device, peaks, steps, warmup)
        out = headline_from(e, "baseline_sae 512->32768 top-32 fwd tokens/s", world, steps, warmup, "weak")
    elif cfg == "3":
        e = bench_tsae(args, T, rank, world, device, peaks, steps, warmup)
        out = headline_from(e, "t_sae 512->32768 fwd tokens/s", world, steps, warmup, "weak")
    elif cfg == "4":
        e = bench_qsae(args, T, rank, world, device, peaks, steps, warmup)
        h = dict(e["sparse_b4096"], workload=e["workload"], variants=e)
        out = headline_from(h, "q_sae 512->32768 4-bit fwd tokens/s", world, steps, warmup, "weak")
    elif cfg == "5":
        e = bench_dict_sharded(args, T, rank, world, device, peaks, steps, warmup, ks=(args.k,) if args.k != 32 else (32, 2097),
                               B=min(args.batch, 4096))
        key = f"{args.transport}_k{args.k if args.k != 32 else 32}"
        h = dict(e[key], workload=e["workload"], variants=e)
        out = headline_from(h, f"b_sae 512->{args.hidden} 4-bit dictionary-sharded fwd tokens/s", world, steps, warmup, "strong")

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and cfg in ("all", "1"):
            out["cpu_baseline"], _ = cpu_baseline_block(args.cpu_batch, args.k, 5, 1)
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.destroy_process_group()


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(directory, vals, idx, recon):
    """--dump-outputs: the last timed step's (values, indices, reconstruction) as DIR/<name>.npy, indices as float64
    (exact). When the whole batch would exceed DUMP_BYTES, a fixed-seed sample of rows is written; rows.npy lists the
    batch rows written, in order."""
    import numpy as np

    arrays = {"latent_values": vals.astype(np.float32), "latent_indices": idx.astype(np.float64),
              "reconstruction": recon.astype(np.float32)}
    B = recon.shape[0]
    row_bytes = 8 + sum(a[0].nbytes for a in arrays.values())
    n = min(B, (DUMP_BYTES - 4096) // row_bytes)          # 4096: the four .npy headers
    rows = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "rows.npy", rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a[rows])


def headline_from(e, metric, world, steps, warmup, scaling):
    out = {"metric": metric, "value": e["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": e["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "bf16",
           "data": "synthetic", "config": {"workload": e.get("workload")}}
    for k, v in e.items():
        if k not in ("value", "unit", "ms_per_step", "workload"):
            out[k] = v
    return out


def main():
    global HEAVY_TAIL
    args = parse()
    HEAVY_TAIL = bool(args.heavy_tail)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: spawn it ourselves so `python bench.py --gpus N` also works
        port = os.environ.get("MASTER_PORT", "29531")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", port, __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
