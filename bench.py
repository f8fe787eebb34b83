#!/usr/bin/env python
"""Headline benchmark: all-reduce bus bandwidth (BASELINE.json: "allreduce bus GB/s vs msg size at 1/2/4/8 B200,
device-timed, max over ranks").

    python bench.py --gpus N --steps K --warmup W            # ours (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N ...            # the unmodified reference (CPU/MPI library) from oracle/_ref
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's output to DIR/*.npy

One "step" = one fp32 SUM all-reduce of the headline message (1 GiB per rank, out of place, with the 1/N averaging
scale fused into the kernel) through the public API (mlsl_b200.allreduce -> Distribution::AllReduceEx ->
Environment::Wait).  The metric has the SAME name at every N: `allreduce_busbw_GBps`, value = the whole job's aggregate
bus bandwidth = N x (S / t) x f(N) with the nccl-tests factor f(N) = 2(N-1)/N (N > 1; a single GPU has no link, f(1) = 1
and the value is the bandwidth of the on-device pass).  Per-GPU bus bandwidth, algorithm bandwidth and the fraction of
the roofline of the kernel that actually ran are separate keys.  Timed with CUDA events on the launching stream, max
over ranks; random input, the whole output is verified.  The JSON line also carries a message-size sweep, the same
sweep through NCCL (+ the separate scale kernel) on the same box, the end-to-end number (pinned host -> device ->
all-reduce -> host every step) and the clocks sampled through NVML during the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HEADLINE_BYTES = 1 << 30


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bytes", type=int, default=HEADLINE_BYTES, help="headline message size per rank")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--sweep-sizes", default="", help="comma separated byte sizes instead of the default 1 KiB..1 GiB x4 ladder")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--nccl", action="store_true", help="(default at N > 1) also time torch.distributed (NCCL) all_reduce")
    ap.add_argument("--no-nccl", action="store_true", help="skip the NCCL comparison")
    ap.add_argument("--compress", action="store_true", help="headline through the fp8-compressed transport")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed step as DIR/<name>.npy")
    return ap.parse_args()


class ClockSampler:
    """SM clock and throttle reasons of this rank's GPU, polled through NVML (~1 kHz) from a thread while the timed
    region runs (nvidia-smi's fastest loop is too coarse for a 7 ms region); falls back to `nvidia-smi -lms`."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread, self.proc = index, [], False, None, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    why = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:  # noqa: BLE001
                    why = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((time.perf_counter(), float(mhz), int(why)))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.0005)

    def _read_smi(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            try:
                why = 0
                for bit, v in zip((0x8, 0x40, 0x20, 0x4), p[2:6]):
                    if v.lower().startswith("active"):
                        why |= bit
                self.max_mhz = float(p[1])
                self.samples.append((time.perf_counter(), float(p[0]), why))
            except (ValueError, IndexError):
                continue

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.max_mhz = None
            threading.Thread(target=self._read_smi, daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self, t0=None, t1=None):
        """summary of the samples taken in [t0, t1] (host perf_counter; the timed region), all samples if too few"""
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples (NVML and nvidia-smi unavailable)"]}
        inside = [x for x in self.samples if t0 is not None and t0 <= x[0] <= t1]
        window = "timed region"
        if len(inside) < 3:
            inside, window = self.samples, "warm-up + timed region (the timed region alone held < 3 samples)"
        mhz = sorted(x[1] for x in inside)
        why = 0
        for x in inside:
            why |= x[2]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": float(self.max_mhz) if self.max_mhz else max(mhz),
                "reasons": sorted(n for b, n in self.REASONS.items() if why & b), "samples": len(inside), "window": window,
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def busbw_factor(n):
    return 2.0 * (n - 1) / n if n > 1 else 1.0


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except (OSError, ValueError):
        return {"hbm_gbs": 6650.0}, "fallback"


LINK_GBS = 770.0     # measured peer copy per direction per GPU on this pool (B200_PROFILING.md; nominal 900)


def roofline(world, S, ms, nvls):
    """achieved / ceiling for the kernel that ran: N = 1 - the measured HBM copy peak (read + write bytes); two-shot
    peer-to-peer - every byte crosses a link once per direction per phase, bus bandwidth <= the link bandwidth; NVLS -
    S(1 + 1/N) bytes per direction per GPU, i.e. algorithm bandwidth <= link / (1 + 1/N)."""
    pk, src = peaks()
    algbw = S / (ms * 1e-3) / 1e9
    if world == 1:
        return {"frac": round(2 * algbw / pk["hbm_gbs"], 4), "ceiling": "HBM copy %.0f GB/s (read+write), of %s" % (pk["hbm_gbs"], src)}
    if nvls:
        ceil_alg = LINK_GBS / (1.0 + 1.0 / world)
        return {"frac": round(algbw / ceil_alg, 4), "ceiling": "NVLS: algbw <= %.0f / (1 + 1/N) = %.0f GB/s (measured 770 GB/s link; nominal 900)" % (LINK_GBS, ceil_alg)}
    return {"frac": round(algbw * busbw_factor(world) / LINK_GBS, 4), "ceiling": "peer-to-peer two-shot: busbw <= %.0f GB/s (measured link; nominal 900)" % LINK_GBS}


DUMP_ELEMS = 1 << 22     # 16 MiB of float32 per array: larger outputs are dumped as a fixed, seeded sample


def dump_outputs(d, arrays):
    """--dump-outputs: every array as <d>/<name>.npy in float32.  An array of more than DUMP_ELEMS elements is sampled at
    the same sorted, seeded indices on every run, so that the dumps of two builds compare element for element."""
    import numpy as np
    import torch

    os.makedirs(d, exist_ok=True)
    for name, t in arrays.items():
        flat = t.reshape(-1)
        if flat.numel() > DUMP_ELEMS:
            idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), DUMP_ELEMS))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(d, name + ".npy"), flat.float().cpu().numpy())


def run_ours(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and rank == 0:
        print("warning: WORLD_SIZE=%d but --gpus %d (launch with torchrun for N>1)" % (world, args.gpus), file=sys.stderr)
    torch.cuda.set_device(local)
    os.environ.setdefault("MLSL_BACKEND", "cuda")
    S = args.bytes
    need_gb = 2 * S / 2 ** 30 + 1.0
    os.environ.setdefault("MLSL_HEAP_SIZE_GB", "%.2f" % max(need_gb, 3.5))
    os.environ.setdefault("MLSL_WATCHDOG_SEC", "60")
    # a pure collective loop: run the kernels directly on the caller's stream (no comm-stream hop, no events)
    os.environ.setdefault("MLSL_STREAM_MODE", "inline")
    use_graph = os.environ.get("MLSL_BENCH_GRAPH", "1") == "1"

    import mlsl_b200 as mlsl

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    env = mlsl.init()
    assert env.get_backend_name() == "cuda", "bench needs the CUDA backend"
    assert mlsl.world_size() == world
    n = S // 4
    x = mlsl.alloc_tensor(n, torch.float32, zero=False)
    y = mlsl.alloc_tensor(n, torch.float32, zero=False)
    scale = 1.0 / world
    # random input with a closed-form sum: x_r = base + r * delta, base / delta drawn from the SAME seed on every rank,
    # so every rank can verify the WHOLE output locally: sum_r x_r / N = base + delta (N - 1) / 2
    gen = torch.Generator(device="cuda").manual_seed(1234)
    base = torch.empty(n, device="cuda").uniform_(-1.0, 1.0, generator=gen)
    delta = torch.empty(n, device="cuda").uniform_(-1.0, 1.0, generator=gen)
    torch.add(base, delta, alpha=float(rank), out=x)

    def verify(out, count, rtol=2e-5, atol=2e-5):
        bad, CH = 0, 1 << 26
        for o in range(0, count, CH):
            e = min(count, o + CH)
            want = torch.add(base[o:e], delta[o:e], alpha=(world - 1) / 2.0)
            bad += int((~torch.isclose(out[o:e], want, rtol=rtol, atol=atol)).sum().item())
        return bad

    def step_device(src, dst, count):
        mlsl.allreduce(src[:count], out=dst[:count], scale=scale, compress=args.compress)

    def timed(fn, steps, warm, graph=False, want_window=False):
        for _ in range(warm):
            fn()
        mlsl.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0 = time.perf_counter()
        if graph:
            # launch-bound sizes: capture the K collectives in one CUDA graph (tickets live in device memory, so a
            # replay runs the full handshake again) and time the replay
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for _ in range(steps):
                    fn()
            g.replay()
            torch.cuda.synchronize()
            mlsl.barrier()
            torch.cuda.synchronize()
            h0 = time.perf_counter()
            e0.record()
            g.replay()
            e1.record()
        else:
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
        torch.cuda.synchronize()
        h1 = time.perf_counter()
        mlsl.barrier()
        ms = e0.elapsed_time(e1) / steps
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        mlsl.allreduce(t, op="max")          # max over ranks, through our own library
        torch.cuda.synchronize()
        return (float(t.item()), h0, h1) if want_window else float(t.item())

    # ---- headline ---------------------------------------------------------------------------------------------
    gpu_index = (int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local]) if os.environ.get("CUDA_VISIBLE_DEVICES")
                 else local)
    sampler = ClockSampler(gpu_index) if rank == 0 else None
    if sampler:
        sampler.start()
    warm = max(args.warmup, 3)
    # warm-up: at least `warm` steps AND ~0.4 s of load, so the clocks have settled when the timed region starts.  The
    # number of extra steps must be the SAME on every rank (it is a collective): agree on the slowest rank's step time
    est = timed(lambda: step_device(x, y, n), 3, 1)
    extra = max(0, min(2000, int(400.0 / max(est, 1e-3))))
    for k in range(extra):
        step_device(x, y, n)
        if k % 8 == 7:
            torch.cuda.synchronize()
    ms, h0, h1 = timed(lambda: step_device(x, y, n), args.steps, warm, want_window=True)
    clocks = sampler.stop(h0, h1) if sampler else None
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"allreduce_out": y[:n]})
    y_bad = verify(y, n, *( (0.08, 0.08) if args.compress else (2e-5, 2e-5)))
    ok = y_bad == 0
    describe = env.describe_backend()
    nvls = ("NVLS" in describe and world >= int(os.environ.get("MLSL_NVLS_MIN_RANKS", "4"))
            and os.environ.get("MLSL_NVLS", "1") != "0" and not args.compress)
    algbw = S / (ms * 1e-3) / 1e9
    busbw = algbw * busbw_factor(world)
    value = busbw * world

    # ---- sweep -------------------------------------------------------------------------------------------------
    def iters(b):
        return 200 if b <= (1 << 16) else (60 if b <= (1 << 22) else (20 if b <= (1 << 26) else 6))

    sizes = []
    if not args.no_sweep:
        sizes = [1 << k for k in range(10, 31, 2)]
        if S not in sizes:
            sizes.append(S)
        if args.sweep_sizes:
            sizes = [int(v) for v in args.sweep_sizes.split(",")]
        sizes = [b for b in sorted(sizes) if b <= S]
    sweep = []
    for b in sizes:
        cnt = b // 4
        gr = use_graph and b <= (1 << 26)
        y[:cnt].zero_()
        m = timed(lambda: step_device(x, y, cnt), iters(b), 5, graph=gr)
        sweep.append({"bytes": b, "us": round(m * 1e3, 3), "algbw_GBps": round(b / (m * 1e-3) / 1e9, 3),
                      "busbw_GBps": round(b / (m * 1e-3) / 1e9 * busbw_factor(world), 3), "cuda_graph": gr,
                      "correct": verify(y, cnt) == 0})

    # ---- NCCL on the same box: all_reduce + the separate scale kernel our epilogue fuses away (default at N > 1) ------
    nccl = None
    if world > 1 and not args.no_nccl:
        try:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            xt = torch.empty(n, device="cuda")
            nccl = {"sweep": []}
            for b in sorted(set(sizes + [S])):
                v = xt[:b // 4]

                def f():
                    dist.all_reduce(v)
                    v.mul_(scale)
                try:
                    m = timed(f, iters(b), 5, graph=use_graph and b <= (1 << 26))
                except Exception:  # noqa: BLE001 - capture not supported by this NCCL build: time eager launches
                    m = timed(f, iters(b), 5, graph=False)
                nccl["sweep"].append({"bytes": b, "us": round(m * 1e3, 3),
                                      "busbw_GBps": round(b / (m * 1e-3) / 1e9 * busbw_factor(world), 3)})
                xt.fill_(1.0)
            head = [r for r in nccl["sweep"] if r["bytes"] == S][0]
            nccl["headline_busbw_GBps"] = head["busbw_GBps"]
            nccl["ours_over_nccl"] = round(busbw / head["busbw_GBps"], 3)
            nccl["what"] = "torch.distributed all_reduce (NCCL %s) + tensor.mul_(1/N), same sizes, same timing" % ".".join(map(str, torch.cuda.nccl.version()))
            dist.destroy_process_group()
        except Exception as ex:  # noqa: BLE001 - the comparison must never cost the headline
            nccl = {"error": repr(ex)[:300]}

    # ---- end to end: pinned host -> device, all-reduce, device -> host, every step ------------------------------------
    e2e = None
    if not args.no_e2e:
        hin = torch.empty(n, dtype=torch.float32).pin_memory()
        hout = torch.empty(n, dtype=torch.float32).pin_memory()
        hin.copy_(x)
        torch.cuda.synchronize()

        def step_e2e():
            # the public call with host-resident buffers: the library pipelines H2D / all-reduce / D2H in chunks
            mlsl.allreduce(hin, out=hout, scale=scale)

        try:
            ms_e = timed(step_e2e, max(3, min(args.steps, 10)), 3)
            y.copy_(hout)
            e_alg = S / (ms_e * 1e-3) / 1e9
            e2e = {"value": round(e_alg * busbw_factor(world) * world, 3), "unit": "GB/s",
                   "h2d_bytes_per_step": S, "d2h_bytes_per_step": S, "ms_per_step": round(ms_e, 4),
                   "algbw_per_gpu_GBps": round(e_alg, 3),
                   "how": "mlsl.allreduce(pinned_host_in, out=pinned_host_out): chunked H2D -> NVLink all-reduce -> D2H pipeline, "
                          "same aggregate definition as `value`; per GPU the PCIe link carries S up and S down per step",
                   "correct": verify(y, n) == 0}
        except Exception as ex:  # noqa: BLE001 - the device-timed headline must still be reported
            e2e = {"error": repr(ex)[:300]}

    # kernels per timed step: giant messages on the multicast (NVLS) path may be issued as several launches
    launches_per_step = 1                     # one persistent kernel walks the whole message ...
    chunk = int(env.get_tuning("nvls_chunk_mb")) << 20
    if nvls and chunk and S >= chunk + chunk // 2:
        launches_per_step = -(-S // chunk)    # ... unless MLSL_NVLS_CHUNK_MB splits giant multicast messages
    out = {
        "metric": "allreduce_busbw_GBps",
        "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": round(ms, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "impl": "ours",
        "busbw_per_gpu_GBps": round(busbw, 3), "algbw_GBps": round(algbw, 3), "roofline": roofline(world, S, ms, nvls),
        "config": {"model": "allreduce fp32 SUM, %d MiB per rank, out of place, fused 1/N scale" % (S >> 20),
                   "global_batch": None, "seq_len": None, "parallelism": "dp%d" % world, "message_bytes": S,
                   "l2": ("inputs (%d MiB per buffer) larger than the 126 MB L2, no flush needed" % (S >> 20) if S > (126 << 20) else
                          "send + receive buffers of %d MiB each against a 126 MB L2, NO flush between iterations" % (S >> 20)),
                   # `warmup` = the W asked for; the clocks settle over ~0.4 s more of the same step before the timed region
                   "warmup_steps_run": warm + extra + 4, "transport": "fp8" if args.compress else "fp32",
                   "api": "mlsl_b200.allreduce -> Distribution::AllReduceEx -> Environment::Wait",
                   "backend": env.get_backend_name(), "backend_detail": describe, "stream_mode": os.environ.get("MLSL_STREAM_MODE"),
                   "kernel": ("k_scale_copy" if world == 1 else ("k_allreduce_quant" if args.compress else
                                                                 ("k_allreduce<NVLS multimem>" if nvls else "k_allreduce<peer-to-peer two-shot>"))),
                   "correct": ok, "verified": "whole output (%d elements) against the closed form of the random input; %d mismatches" % (n, y_bad),
                   "value_definition": "whole-job aggregate bus bandwidth: N x S / t x f(N), f = 2(N-1)/N as in nccl-tests (f(1) = 1: "
                                       "no link, the on-device pass).  Weak scaling: S per rank fixed, the aggregate grows with N; "
                                       "busbw_per_gpu_GBps is the per-link figure that stays constant under ideal scaling"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * launches_per_step,
        "sweep": sweep, "nccl": nccl,
    }
    mlsl.free_tensor(x)
    mlsl.free_tensor(y)
    mlsl.finalize()
    if rank == 0:
        print(json.dumps(out))


def run_reference(args):
    """The unmodified reference library (CPU, Intel MPI runtime) driven by baseline/ref_bench.py."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import ref_bench
        print(json.dumps(ref_bench.run(args.gpus, args.steps, max(args.warmup, 3), args.bytes)))
    except Exception as e:  # noqa: BLE001 - must never fail the driver
        print(json.dumps({"impl": "reference", "unavailable": ("%s: %s" % (type(e).__name__, e))[:300].replace("\n", " ")}))


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
