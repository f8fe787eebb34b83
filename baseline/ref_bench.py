"""Reference arm of bench.py: the UNMODIFIED intel/MLSL (oracle/_ref, built by oracle/install_ref.sh) running the
same metric - fp32 SUM all-reduce bus bandwidth of the headline message through its own public API
(Environment::Alloc + Distribution::AllReduce + Environment::Wait, stock "process" mode, N MPI ranks on this node
launched by its bundled mpiexec.hydra).  The reference is a CPU library: its buffers live in host memory, so the
end-to-end number equals the measured one (no device copies exist on that path).
"""
import json
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(HERE), "oracle", "_ref")


def _env(overrides=None):
    env = dict(os.environ)
    mp = os.path.join(REF, "mpirt")
    env["I_MPI_ROOT"] = mp
    env["MLSL_ROOT"] = REF
    env["PATH"] = os.path.join(mp, "bin") + os.pathsep + env.get("PATH", "")
    env["LD_LIBRARY_PATH"] = os.pathsep.join([os.path.join(REF, "intel64", "lib"), os.path.join(mp, "lib"),
                                              env.get("LD_LIBRARY_PATH", "")])
    # torchrun's variables must not leak into the MPI ranks
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "MLSL_BACKEND", "MLSL_JOB_ID"):
        env.pop(k, None)
    env.setdefault("I_MPI_FABRICS", "shm")
    # Intel MPI 2018's default large-message shm transfer is cross-memory attach (process_vm_readv), which containers
    # commonly forbid ("Cannot read from remote process"); the runtime's own error text names this switch.  An MPI
    # runtime setting: the library and its code path stay stock.
    env.setdefault("I_MPI_SHM_LMT", "shm")
    # the form bench.py times on the GPU: separate send and receive buffers (harness option, the library is untouched)
    env["MLSL_BENCH_OUT_OF_PLACE"] = "1"
    env.update(overrides or {})
    return env


def _run(nranks, minb, maxb, iters, warm, factor, timeout):
    exe = os.path.join(REF, "bin", "ref_allreduce_bench")
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref is not installed (run oracle/install_ref.sh <reference checkout>)")
    hydra = os.path.join(REF, "mpirt", "bin", "mpiexec.hydra")
    tail = [exe, str(minb), str(maxb), str(iters), str(warm), str(factor)]
    res = None
    # launcher options only (the library and its code path stay stock): the second form names the host by address for
    # boxes whose hostname does not resolve
    # MPI runtime ladder, fastest first: shared memory with copy-through-shm large messages, then the TCP fabric
    ladder = [{}, {"I_MPI_FABRICS": "shm:tcp"}, {"I_MPI_FABRICS": "tcp"}]
    for over in ladder:
        for extra in ([], ["-hosts", "127.0.0.1", "-localhost", "127.0.0.1"]):
            res = subprocess.run([hydra] + extra + ["-n", str(nranks)] + tail, env=_env(over), stdout=subprocess.PIPE,
                                 stderr=subprocess.PIPE, text=True, timeout=timeout)
            if res.returncode == 0 and "{" in res.stdout:
                break
        if res.returncode == 0 and "{" in res.stdout:
            break
    rows = []
    for line in res.stdout.splitlines():
        line = line.strip()
        if line.startswith("{"):
            rows.append(json.loads(line))
    if res.returncode != 0 or not rows:
        raise RuntimeError("reference run failed rc=%d: %s" % (res.returncode, (res.stderr or res.stdout)[-300:]))
    return rows


def run(n_gpus, steps, warmup, headline_bytes):
    n = max(int(n_gpus), 1)
    head = _run(n, headline_bytes, headline_bytes, steps, warmup, 4, timeout=3000)[-1]
    sweep = []
    try:
        for r in _run(n, 1024, min(headline_bytes, 1 << 24), 5, 2, 16, timeout=600):
            sweep.append({"bytes": r["bytes"], "us": r["us"], "busbw_GBps": r["busbw_GBps"]})
    except Exception:  # noqa: BLE001 - the sweep is informative only
        pass
    # same definition as the other arm: whole-job aggregate bus bandwidth N x S / t x f(N), f(1) = 1
    per_rank = head["busbw_GBps"] if n > 1 else head["algbw_GBps"]
    value = per_rank * n
    return {
        "metric": "allreduce_busbw_GBps",
        "value": round(value, 4), "busbw_per_gpu_GBps": round(per_rank, 4), "algbw_GBps": round(head["algbw_GBps"], 4), "unit": "GB/s", "n_gpus": n, "steps": steps, "warmup": warmup,
        "ms_per_step": round(head["us"] / 1e3, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "impl": "reference",
        "config": {"model": "allreduce fp32 SUM, %d MiB per rank, out of place" % (headline_bytes >> 20),
                   "parallelism": "dp%d" % n, "message_bytes": headline_bytes,
                   "api": "MLSL::Distribution::AllReduce + Environment::Wait (intel/MLSL process mode, Intel MPI shm)",
                   "device": "CPU (the reference has no GPU path); host-timed, max over ranks",
                   "launcher": "oracle/_ref/mpirt/bin/mpiexec.hydra -n %d" % n},
        "e2e": {"value": round(value, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "buffers are host resident: the measured value already is end to end"},
        "gpu_launches": 0, "sweep": sweep,
    }


if __name__ == "__main__":
    import sys
    print(json.dumps(run(int(sys.argv[1]) if len(sys.argv) > 1 else 2, 3, 1, 1 << 24)))
