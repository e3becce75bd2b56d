#!/usr/bin/env python
"""bench.py — EM iterations/s of the GMM-EM hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N=1)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N>1)

A "step" is one pass of the EM loop body of the reference (gaussian.cu:532-755):
M-step statistics -> all-reduce of the packed statistics -> normalisation +
DxD inversions + constants + E-step operand (one device kernel; option "finalize" = 0
/ GMM_FINALIZE=host: on the host with one D2H and one H2D) -> E-step (responsibilities
+ log-likelihood), on the synthetic workload of BASELINE.json config 3
(N=10M, D=24, K=64; config 4 shards the same 10M events over N GPUs = strong
scaling).  `value` is measured with the events resident in HBM: exactly K steps are
timed, split as evenly as possible into at most `--repeats` blocks (barrier +
synchronize on both sides, device clock, max over ranks); the MEDIAN block time per
step is reported (`blocks_ms_per_step` lists all of them).  `e2e` is measured through the C ABI from
HOST buffers (pinned events H2D, parameters H2D, initial E-step, the K steps,
parameters + log-likelihood D2H all inside the timed region: one upload per K steps).

Also on the line: `roofline` (E-step, HBM), `roofline_mstep` (tensor, against the measured
dense BF16/FP16 peak — the pipe the kernel's kind::f16 MMAs run on), `cpu_baseline` (the
sequential-EM CPU port on the host cores, median of 3), `reference_gpu` (the UNMODIFIED
reference program compiled for sm_100a, oracle/_ref/gaussianMPI_ref_perf, run on this GPU at
config 2 and config 3) and `config5` (the model-order-reduction loop K=128 -> 16, gmm_fit).

`--dump-outputs DIR` writes, right after the timed steps, what the last of them computed
(rank 0: parameters, log-likelihood, memberships of a fixed seeded sample of its events) as
DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be
compared array for array.

`--impl reference` times the reference's algorithm on the host cores (the
sequential-EM CPU port in oracle/, FP32, OpenMP over the physical cores) on a bounded
slice of the same workload.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG", os.environ.get("GMM_NCCL_DEBUG", "WARN"))   # the driver's own setting wins
import __graft_entry__ as entry  # noqa: E402

WORKLOADS = {
    "c3": dict(N=10_000_000, D=24, K=64),      # BASELINE.json configs[2] / [3]
    "c2": dict(N=1_000_000, D=16, K=32),       # configs[1]
    "c1": dict(N=10_000, D=4, K=8),            # configs[0]
}
C5 = dict(N=10_000_000, D=24, K0=128, target=16, K_true=16)      # configs[4]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region, in-process through NVML (two cheap
    queries every 25 ms from a thread; the GIL is free while the main thread sits in the C library).  Falls back to
    one `nvidia-smi -lms 100` child when pynvml is unavailable.  Round 1 ran `nvidia-smi -lms 20` with eight
    query fields next to rank 0 and rank 0 lagged its peers."""

    def __init__(self, device):
        self.device, self.samples, self.stop_flag, self.t, self.proc = device, [], False, None, None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else device
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.samples.append((mhz, r))
            except Exception:
                pass
            time.sleep(0.025)

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                bits = 0
                for b, v in zip((0x8, 0x40, 0x20, 0x4), f[3:7]):
                    if v.lower().startswith("active"):
                        bits |= b
                self.max_mhz = float(f[2])
                self.samples.append((float(f[1]), bits))
            except (ValueError, IndexError):
                continue

    def start(self):
        if self.h is not None:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
            return
        q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.max_mhz = None
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def wait_ready(self, timeout=5.0):
        t_end = time.time() + timeout
        while self.t and not self.samples and time.time() < t_end:
            time.sleep(0.01)

    def mark(self):
        return len(self.samples)

    def stop(self, begin=0, end=None):
        if not self.t:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["clock sampler unavailable"])
        time.sleep(0.06)
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        self.t.join(timeout=2)
        s = self.samples[begin:(end + 1 if end is not None else None)]
        if not s:                                        # region shorter than one sampling period: nearest samples
            s = self.samples[max(0, begin - 1):begin + 1] or self.samples[-1:]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = sorted({n for _, r in s for b, n in names.items() if r & b})
        sm = [m for m, _ in s]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=self.max_mhz, reasons=reasons, samples=len(sm),
                    source="nvml" if self.h is not None else "nvidia-smi")


# ---------------------------------------------------------------------------------------------
# CPU baseline: the sequential-EM CPU port (oracle/gmm_oracle.c, FP32), timed in a CHILD process with its own
# OpenMP environment (torchrun exports OMP_NUM_THREADS=1 to its ranks; round 1 inherited it at N >= 2).
# ---------------------------------------------------------------------------------------------
def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def cpu_worker(args):
    """Child: time `steps` EM iterations of the CPU port `repeats` times on the first `sample` events."""
    pkg = entry.load_package()
    orc = entry.load_oracle("f32")
    wl = WORKLOADS[args.workload]
    N, D, K = wl["N"], wl["D"], wl["K"]
    n = min(args.cpu_sample, N)
    ev = pkg.synth.make_blobs(n, D, K, seed=pkg.synth.SEED + 1)
    cl = pkg.Clusters(K, D, n)
    orc.seed(ev, K, cl)
    soa = orc.transpose(ev)
    orc.estep(soa, cl, K)
    for _ in range(args.warmup):
        orc.mstep(soa, cl, K); orc.constants(cl, K); orc.estep(soa, cl, K)
    times = []
    for _ in range(max(1, args.repeats)):
        t0 = time.perf_counter()
        for _ in range(max(1, args.steps)):
            orc.mstep(soa, cl, K); orc.constants(cl, K); orc.estep(soa, cl, K)
        times.append((time.perf_counter() - t0) / max(1, args.steps))
    print(json.dumps(dict(times=times, n=n, threads=int(os.environ.get("OMP_NUM_THREADS", "0")))))
    return 0


def run_cpu_baseline(workload, sample_events, steps, warmup, repeats):
    """(it/s at full N by linear extrapolation [median], cores, sample text, s/step median, all s/step)."""
    wl = WORKLOADS[workload]
    cores = physical_cores()
    env = {k: v for k, v in os.environ.items() if not k.startswith(("OMP_", "GOMP_", "KMP_"))}
    env.update(OMP_NUM_THREADS=str(cores), OMP_PROC_BIND="spread", OMP_PLACES="cores", OMP_WAIT_POLICY="active")
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "cpu-worker", "--workload", workload, "--cpu-sample", str(sample_events),
           "--steps", str(steps), "--warmup", str(warmup), "--repeats", str(repeats)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1500)
    out = json.loads(r.stdout.strip().splitlines()[-1])
    n, times = out["n"], out["times"]
    dt = float(np.median(times))
    scale = wl["N"] / n
    its = 1.0 / (dt * scale)
    sample = (f"{steps} EM iteration(s) x {len(times)} repeats (median; all: {[round(1.0 / (t * scale), 5) for t in times]} it/s) of the "
              f"sequential-EM CPU port (oracle/gmm_oracle.c, FP32, OpenMP {cores} threads = physical cores, bound, own process) "
              f"on {n} of {wl['N']} events, D={wl['D']}, K={wl['K']}; it/s extrapolated linearly to N={wl['N']}")
    return its, cores, sample, dt, times


# ---------------------------------------------------------------------------------------------
# reference_gpu: the unmodified reference program (shim-built, oracle/_ref/gaussianMPI_ref_perf) on this GPU
# ---------------------------------------------------------------------------------------------
def run_reference_gpu(pkg, workload, device, iters=3):
    exe = os.path.join(ROOT, "oracle", "_ref", "gaussianMPI_ref_perf")
    if not os.path.exists(exe):
        return dict(unavailable="oracle/_ref/gaussianMPI_ref_perf not built (needs /root/reference at build time)")
    wl = WORKLOADS[workload]
    N, D, K = wl["N"], wl["D"], wl["K"]
    with tempfile.TemporaryDirectory(prefix="gmmref_") as td:
        data = os.path.join(td, "d.bin")
        pkg.synth.write_bin(data, pkg.synth.make_blobs(N, D, K))
        env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES=str(device), GMM_REF_ITERS=str(iters))
        try:
            r = subprocess.run([exe, str(K), data, os.path.join(td, "out"), str(K)], capture_output=True, text=True, env=env, timeout=420)
        except subprocess.TimeoutExpired:
            return dict(unavailable=f"reference binary exceeded 420 s at {workload}")
    if r.returncode != 0:
        return dict(unavailable=f"reference binary rc={r.returncode}: {(r.stdout + r.stderr)[-300:]}")
    prof = {}
    for name in ("E-step Kernel", "M-step Kernel", "Consts Kernel"):
        m = re.search(name + r":\s+([\d.]+)\s+(\d+)\s+([\d.]+)", r.stdout)
        if m:
            prof[name] = (float(m.group(1)), int(m.group(2)), float(m.group(3)))
    extra = {}
    for name in ("GPU Memcpy", "CPU", "MPI"):
        m = re.search(name + r":\s+([\d.]+)", r.stdout)
        if m:
            extra[name] = float(m.group(1))
    if len(prof) < 3:
        return dict(unavailable="could not parse the reference's profile output")
    kern = sum(v[2] for v in prof.values())                       # mean seconds per launch group, summed = one iteration
    allin = kern + sum(extra.values()) / max(1, iters)            # + its synchronous copies / host reductions per iteration
    return dict(value=1.0 / allin, unit="it/s", kernels_only_its=1.0 / kern, iterations=iters,
                seconds_per_iteration=dict(estep=prof["E-step Kernel"][2], mstep=prof["M-step Kernel"][2], constants=prof["Consts Kernel"][2],
                                           memcpy_cpu_mpi=sum(extra.values()) / max(1, iters)),
                how=f"unmodified gaussian.cu/gaussian_kernel.cu compiled -arch=sm_100a with cutil.h/mpi.h shims (oracle/Makefile ref), shipped "
                    f"ENABLE_OUTPUT 0, MIN=MAX_ITERS={iters}, 1 GPU, {workload}: N={N} D={D} K={K}; its own profile_t timers (gaussian.cu:967)")


def block_sizes(steps, repeats):
    """`steps` timed steps split as evenly as possible into at most `repeats` blocks (at least one step each)."""
    n = max(1, min(repeats, steps))
    return [steps // n + (1 if i < steps % n else 0) for i in range(n)]


DUMP_MEMB_BYTES = 32 << 20         # memberships written by --dump-outputs: 131072 events at K = 64


def dump_outputs(pkg, eng, K, D, n, ll, out_dir):
    """Write what a caller of gmm_em_iterations receives after the last timed step (gmm_get_clusters with memberships,
    and the log-likelihood) as <out_dir>/<name>.npy.  Memberships [K][n] larger than DUMP_MEMB_BYTES are sampled: a
    fixed, seeded, sorted choice of events, whose indices are written next to them (35 MB in all at config 3)."""
    os.makedirs(out_dir, exist_ok=True)
    cl = eng.get_clusters(K, out=pkg.Clusters(K, D, n), with_memberships=True)
    arrays = {f: getattr(cl, f)[:K] for f in pkg.Clusters.FIELDS}
    arrays["loglik"] = np.array([ll], np.float64)
    m = DUMP_MEMB_BYTES // (4 * K)
    if n > m:
        idx = np.sort(np.random.default_rng(pkg.synth.SEED).choice(n, m, replace=False))
        arrays["memberships"] = cl.memberships[:K, idx]
        arrays["memberships_events"] = idx.astype(np.float64)
    else:
        arrays["memberships"] = cl.memberships[:K]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    return dict(dir=out_dir, arrays=sorted(arrays), bytes=int(sum(a.nbytes for a in arrays.values())),
                memberships_events=int(arrays["memberships"].shape[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5,
                    help="timed blocks the --steps iterations are split into; the median time per step of a block is reported")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "cpu-worker"])
    ap.add_argument("--workload", default=os.environ.get("GMM_BENCH_WORKLOAD", "c3"), choices=list(WORKLOADS))
    ap.add_argument("--path", default=os.environ.get("GMM_BENCH_PATH", "auto"), choices=["auto", "simt", "tensor"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--cpu-sample", type=int, default=1_000_000, help="events in the cpu_baseline slice (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference-on-B200 runs (config 2 and 3)")
    ap.add_argument("--c5-iters", type=int, default=int(os.environ.get("GMM_BENCH_C5_ITERS", "2")),
                    help="EM iterations per model order of the config-5 measurement (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the parameters, log-likelihood and (sampled) memberships they computed "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "cpu-worker":
        return cpu_worker(args)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = dict(WORKLOADS[args.workload])
    metric = "EM iterations/sec at N=10M D=24 K=64; E-step HBM GB/s vs roofline" if args.workload == "c3" else \
        f"EM iterations/sec at N={wl['N']} D={wl['D']} K={wl['K']}"
    pkg = entry.load_package()

    # ---------------- reference arm: CPU port on the host cores ----------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        sample = args.cpu_sample or 1_000_000
        # bounded: `steps` iterations per repeat would be minutes at K = 20; one repeat of `steps` iterations, W warm-up
        its, cores, text, dt, _ = run_cpu_baseline(args.workload, sample, steps=max(1, args.steps), warmup=args.warmup, repeats=1)
        line = dict(metric=metric, value=its, unit="it/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                    ms_per_step=dt * 1e3 * (wl["N"] / min(sample, wl["N"])), higher_is_better=True, scaling=args.scaling,
                    vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                    config=dict(workload=f"{args.workload}: N={wl['N']} D={wl['D']} K={wl['K']} Gaussian blobs (seed {pkg.synth.SEED})"),
                    cpu_baseline=dict(value=its, unit="it/s", cores=cores, kind="port", sample=text),
                    e2e=dict(value=its, unit="it/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return 0

    # ---------------- B200 arm --------------------------------------------------
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local_rank))
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    torch.cuda.set_device(local_rank)
    pkg.load_library()                                   # raises if the CUDA library is missing: no fallback

    N, D, K = wl["N"], wl["D"], wl["K"]
    if args.scaling == "weak":
        N = N * world
    begin, count = pkg.shard_range(N, world, rank)
    # synthetic data: every rank draws the same seeded data set and keeps its shard (pinned host memory)
    ev_all = pkg.synth.make_blobs(N, D, K)
    ev_pinned = torch.empty((count, D), dtype=torch.float32, pin_memory=True)
    ev_pinned.numpy()[...] = ev_all[begin:begin + count]
    del ev_all
    path = {"auto": pkg.PATH_AUTO, "simt": pkg.PATH_SIMT, "tensor": pkg.PATH_TENSOR}[args.path]
    want_c5 = args.c5_iters > 0 and args.workload == "c3" and args.scaling == "strong"
    Kmax = C5["K0"] if want_c5 else K

    def fresh_nccl_id():
        """A ncclUniqueId can bootstrap ONE communicator: every engine gets its own (rank 0 draws it,
        torch.distributed broadcasts the 128 bytes)."""
        buf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = torch.frombuffer(bytearray(pkg.nccl_unique_id()), dtype=torch.uint8).clone()
        dist.broadcast(buf, src=0)
        return bytes(buf.numpy().tobytes())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    eng = pkg.Engine(None, Kmax, device=local_rank, n_global=N, offset=begin, events_ptr=ev_pinned.data_ptr(), n_local=count, D=D)
    eng.set_option("path", path)
    if "GMM_BENCH_ALLREDUCE" in os.environ:              # A/B: 1 = the library's peer-memory kernel (default), 0 = ncclAllReduce
        eng.set_option("allreduce", int(os.environ["GMM_BENCH_ALLREDUCE"]))
    if world > 1:
        eng.comm_init(world, rank, fresh_nccl_id())
    r_, n_ = eng.comm_rank()
    print(f"[gmm] rank {r_} of nranks {n_} (NCCL communicator of the engine) on cuda:{local_rank}", file=sys.stderr, flush=True)

    # ---- device-resident measurement: value ----
    seeded = eng.seed(K)
    eng.estep(K)                                         # initial E-step (gaussian.cu:487-523)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                  # before the warm-up: start-up cost stays outside the timed region
    eng.em_iterations(K, args.warmup)
    if rank == 0:
        sampler.wait_ready()
    eng.profile(reset=True)
    blocks, walls = [], []                               # seconds per step of each timed block
    m0 = None
    ll = 0.0
    for n_block in block_sizes(args.steps, args.repeats):
        barrier()
        if m0 is None:
            m0 = sampler.mark()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        t0 = time.perf_counter()
        ll = eng.em_iterations(K, n_block)               # exactly `n_block` iterations; returns after a stream sync
        ev1.record()
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) / n_block)
        blocks.append(max_over_ranks(ev0.elapsed_time(ev1) * 1e-3) / n_block)   # device clock around the block, max over ranks
    m1 = sampler.mark()
    barrier()
    clocks = sampler.stop(m0, m1) if rank == 0 else None
    dt = float(np.median(blocks))
    dt_wall = float(np.median(walls))
    prof = eng.profile()
    value = 1.0 / dt
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(pkg, eng, K, D, count, ll, args.dump_outputs)

    # ---- end to end from host buffers: e2e ----
    e2e = None
    if not args.no_e2e:
        e2e_times = []
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            eng.upload_events(events_ptr=ev_pinned.data_ptr())   # H2D of the pinned shard + device transpose
            eng.set_clusters(K, seeded)                      # parameters H2D
            eng.estep(K)
            ll_e2e = eng.em_iterations(K, args.steps)
            res = eng.get_clusters(K)                        # parameters D2H (log-likelihood already read back)
            torch.cuda.synchronize()
            e2e_times.append(max_over_ranks(time.perf_counter() - t0))
            assert np.isfinite(ll_e2e) and np.all(np.isfinite(res.means[:K]))
        dt_e2e = float(np.median(e2e_times))
        F = 1 + D + D * (D + 1) // 2
        params_bytes = 4 * K * (4 + D + 2 * D * D)
        # host finalisation: the reduced statistics come to the host and the packed E-step operand goes back every iteration;
        # device finalisation (option "finalize", the default): neither — parameters and log-likelihood once per batch
        dev_fin_e2e = eng.fit_profile().get("device_finalize_launches", 0) > 0
        upload_bytes = 0 if dev_fin_e2e else 4 * K * (D + D * (D + 1) // 2 + 8)
        stats_bytes = 0 if dev_fin_e2e else 8 * (K * F + 1)
        e2e = dict(value=args.steps / dt_e2e, unit="it/s",
                   h2d_bytes_per_step=int((count * D * 4 + params_bytes) / args.steps + upload_bytes),
                   d2h_bytes_per_step=int(stats_bytes + (params_bytes + 8) / args.steps),
                   iterations_per_upload=args.steps, all_its=[args.steps / t for t in e2e_times],
                   note=f"median of 3; each measurement = ONE gmm_upload_events (pinned H2D of the {count}x{D} shard) + gmm_set_clusters + "
                        f"gmm_estep + {args.steps} iterations + gmm_get_clusters (D2H): {args.steps} iterations per upload, per-step bytes "
                        f"amortise the one-time copies; context / NCCL communicator creation is setup and outside the region")

    # ---- roofline of the dominant kernels (per-launch CUDA-event times from the engine, on the engine's stream) ----
    peaks = measured_peaks()
    n_it = max(1, int(prof["iterations"]))
    estep_ms = prof["estep_ms"] / n_it
    mstep_ms = prof["mstep_ms"] / n_it
    e_bytes = 4.0 * count * (D + K)                       # read X once + write memberships once (SURVEY §8d)
    m_flops = 2.0 * count * K * D * D                     # covariance contraction (SURVEY §8d)
    e_gbs = e_bytes / (estep_ms * 1e-3) / 1e9 if estep_ms > 0 else 0.0
    m_tfs = m_flops / (mstep_ms * 1e-3) / 1e12 if mstep_ms > 0 else 0.0
    tensor_m = args.path != "simt" and D in (4, 8, 12, 16, 20, 24)
    dev_fin = eng.fit_profile().get("device_finalize_launches", 0) > 0
    launches_per_step = (3 if tensor_m else 2) + (1 if dev_fin else 0)     # E-step, M-step (+ its reduction), finalize_params_kernel
    n_tensor, n_simt = int(prof.get("mstep_tensor_launches", 0)), int(prof.get("mstep_simt_launches", 0))
    F = 1 + D + D * (D + 1) // 2
    mt_rows = (F + 127) // 128 * 128
    # executed MMA flops per launch of mstep_tc_kernel: per 16 events and feature tile one M=128,N=128 (ph x [gh;gl]) and one
    # M=128,N=64 (pl x gh) MMA = 3 products of the padded (mt_rows x 64-cluster) tile
    exec_flops = 2.0 * count * mt_rows * ((K + 63) // 64 * 64) * 3 if n_tensor else 0.0
    traffic = traffic_m = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath))
        kind = "tensor" if args.path != "simt" else "simt"
        traffic = tj.get(f"{args.workload}:{kind}:estep")
        traffic_m = tj.get(f"{args.workload}:{kind}:mstep")
    roofline = dict(kernel="estep", bound="hbm", achieved=e_gbs, peak=peaks["hbm_gbs"], unit="GB/s",
                    frac=e_gbs / peaks["hbm_gbs"], traffic=traffic, peak_source=peaks["source"],
                    ms_per_launch=estep_ms, algorithmic_bytes_per_launch=e_bytes)
    roofline_mstep = dict(kernel="mstep_covariance", bound="tensor", achieved=m_tfs, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                          frac=m_tfs / peaks["bf16_tflops_sustained"], traffic=traffic_m,
                          peak_source=peaks["source"] + " dense bf16/fp16 sustained (the kernel issues kind::f16 MMAs)",
                          ms_per_launch=mstep_ms, algorithmic_flops_per_launch=m_flops,
                          executed_mma_flops_per_launch=exec_flops, executed_tflops=exec_flops / (mstep_ms * 1e-3) / 1e12 if mstep_ms > 0 else 0.0,
                          kernels=dict(mstep_tc_kernel_launches=n_tensor, mstep_simt_kernel_launches=n_simt,
                                      note="launch counts in the timed region; mstep_tc_kernel = fixed-point leading parts (exact TMEM "
                                           "accumulation) + FP16 remainders, three products per element"))

    # ---- config 5: model-order reduction K0=128 -> 16 (gmm_fit) on the same GPUs ----
    config5 = None
    if want_c5:
        ev5 = pkg.synth.make_blobs(C5["N"], D, C5["K_true"], seed=pkg.synth.SEED + 5)
        ev_pinned.numpy()[...] = ev5[begin:begin + count]
        del ev5
        eng.upload_events(events_ptr=ev_pinned.data_ptr())
        eng.profile(reset=True)
        barrier()
        t0 = time.perf_counter()
        ideal, mr, _saved = eng.fit(C5["K0"], C5["target"], args.c5_iters, args.c5_iters)
        torch.cuda.synchronize()
        dt5 = max_over_ranks(time.perf_counter() - t0)
        p5 = eng.profile()
        fp = eng.fit_profile()
        config5 = dict(seconds=dt5, final_K=int(ideal), min_rissanen=float(mr), iters_per_K=args.c5_iters, n_gpus=world,
                       em_iterations=int(p5["iterations"]),
                       phases_s=dict(estep=p5["estep_ms"] / 1e3, mstep=p5["mstep_ms"] / 1e3, allreduce=p5["allreduce_ms"] / 1e3,
                                     finalize_upload_host=p5["upload_ms"] / 1e3, reduce_order_host=fp["reduce_order_ms"] / 1e3,
                                     seed=fp["seed_ms"] / 1e3, save_best=fp["save_ms"] / 1e3),
                       workload=f"c5: N={C5['N']} D={D} K0={C5['K0']} -> target {C5['target']} ({C5['K_true']} true blobs, seed {pkg.synth.SEED + 5}), "
                                f"gaussian.cu:479-960 with MIN=MAX_ITERS={args.c5_iters}")

    if rank != 0:
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return 0
    eng.close()

    cpu_baseline = None
    if world == 1 and args.cpu_sample > 0:
        its, cores, text, _, _ = run_cpu_baseline(args.workload, args.cpu_sample, steps=1, warmup=1, repeats=3)
        cpu_baseline = dict(value=its, unit="it/s", cores=cores, kind="port", sample=text)
    reference_gpu = None
    if world == 1 and not args.no_ref_gpu:
        torch.cuda.empty_cache()
        reference_gpu = {w: run_reference_gpu(pkg, w, local_rank) for w in (("c2", "c3") if args.workload == "c3" else (args.workload,))}

    line = dict(metric=metric, value=value, unit="it/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                dtype="f32", data="synthetic",
                config=dict(workload=f"{args.workload}: N={N} D={D} K={K} Gaussian blobs (seed {pkg.synth.SEED}), "
                                     f"{count} events on rank 0", path=args.path, l2="inputs (X 0.96 GB + memberships 2.56 GB at c3) exceed the 126 MB L2",
                            parallelism=f"dp{world} (events sharded, one all-reduce of {8 * (K * (1 + D + D * (D + 1) // 2) + 1)} B per step)",
                            finalisation=("device (finalize_params_kernel, timed under 'upload')" if dev_fin else "host"),
                            arithmetic=("fp32 data and results; tensor path: fp16 hi/lo split operands, fp32 TMEM accumulation, fp64 "
                                        "statistics reduction and finalisation" if args.path != "simt" else
                                        "fp32 E-step, fp64 M-step statistics and host finalisation"),
                            timing=f"{args.steps} timed steps in {len(blocks)} blocks; median over the blocks of the time per step"),
                clocks=clocks, e2e=e2e, gpu_launches=launches_per_step * args.steps, roofline=roofline, roofline_mstep=roofline_mstep,
                phases_ms_per_step=dict(estep=estep_ms, mstep=mstep_ms, constants_host=prof["constants_host_ms"] / n_it,
                                        allreduce=prof["allreduce_ms"] / n_it, upload=prof["upload_ms"] / n_it),
                blocks_ms_per_step=[b * 1e3 for b in blocks],
                loglik=ll, wall_ms_per_step=dt_wall * 1e3, cpu_baseline=cpu_baseline, reference_gpu=reference_gpu,
                config5=config5, comm=dict(rank=r_, nranks=n_), dump_outputs=dumped)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
