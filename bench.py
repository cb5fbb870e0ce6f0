#!/usr/bin/env python
"""bench.py -- ensemble adjoint trajectories/sec on BASELINE.json's headline workload (config C2):
Lorenz d=3 P=3, N=65536 members per GPU, GaussAdjoint, Tsit5 fixed dt=0.01, T=10 (S=1000 steps), saveat 0.1 (K=101),
cotangent dgdu = u - 2, fp64, shared p, synthetic u0 = [1,0,0] + 0.1 z.

One "step" = one full gradient evaluation of the ensemble: forward solve + fused reverse adjoint pass + dG/dp
reduction (+ the one all-reduce of dp over ranks for N>1, issued by b200adj_reverse itself through the handle's NCCL
communicator; members are sharded, weak scaling: 65536 per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--members M] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

--dump-outputs DIR writes what the timed C2 loop hands its caller after its last step, DIR/dp.npy [3] and DIR/du0.npy [3, N]
(rank 0's members), both float64.  The inputs are seeded, so two builds run with the same arguments can be compared array
for array.  Above 60 MB du0 is thinned to every k-th member (the smallest k that fits).

Keys of the one JSON line (rank 0):
`value`     members/s with inputs resident in HBM (device pointers through the C ABI), CUDA-event timed, max over ranks.
`e2e`       same metric through the public API (solve + adjoint_sensitivities(AffineCost)) with HOST buffers: pinned u0 H2D and
            du0/dp D2H inside the timed region every step.
`e2e_rrule` same metric through the plugin seam `_concrete_solve_adjoint` (src/concrete_solve.jl:523-543, 776-1040):
            host primal sol.u[K,d,N] OUT (D2H) and host cotangent Delta[K,d,N] IN (H2D) every step.
`roofline`  the reverse kernel (dominant): SURVEY 8d's per-step algorithmic bytes against the measured HBM peak, the
            compulsory (really moved) bytes, and the fp64-pipe figure that actually bounds the kernel.
`parity`    device gradient vs the CPU oracle on a bounded sub-ensemble, sharded exactly like the timed run (every rank
            owns a slice, dp all-reduced behind the C ABI); the run exits non-zero above 1e-8.
`strong`    (N>1) the metric's fixed total N=65536 split over the ranks.
`secondary` BASELINE configs C4 (bf16 tensor-core neural ODE), C5 (SDE), C1 as a 65536-member adaptive-Tsit5 ensemble and C3
            (Robertson / Rosenbrock23 / QuadratureAdjoint) sharded over the same ranks, each timed, roofline'd and oracle-checked.
`cpu_baseline` the C oracle (a PORT of the reference algorithm; Julia cannot run here) on the host cores.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(family="lorenz", sensealg="gauss", stepper="tsit5_fixed", T=10.0, dt=0.01, nsave=101,
                members_per_gpu=65536, cost=(1.0, -2.0), seed=20260923)
ALG_BYTES_PER_MEMBER_STEP = 8 * (3 + 2 * 6 + 101.0 / 1000.0 * 3)   # 122.4 B (SURVEY.md 8d, C2 fp64)
# fp64 work of one reverse member-step (cuobjdump -sass of tsit5_reverse_kernel<Lorenz,GAUSS>, DESIGN.md 4.2)
DP_INSTR_PER_MEMBER_STEP = dict(dfma=366, dmul=33, dadd=27)
PARITY_TOL = 1e-8
DUMP_BYTES = 60_000_000


def make_inputs(N, offset=0):
    rng = np.random.Generator(np.random.Philox(key=WORKLOAD["seed"] + offset))
    u0 = np.array([1.0, 0.0, 0.0])[:, None] + 0.1 * rng.standard_normal((3, N))
    p = np.array([10.0, 28.0, 8.0 / 3.0])
    return np.ascontiguousarray(u0), p


def c2_config(world, members_per_gpu, block):
    """identical for `--impl ours` and `--impl reference` (the driver compares the two arms' config)"""
    W = WORKLOAD
    return {"workload": "C2 Lorenz d=3 P=3 N=65536/GPU GaussAdjoint Tsit5 fixed dt=0.01 T=10 saveat=0.1 dgdu=u-2 shared p",
            "members_per_gpu": members_per_gpu, "S": int(round(W["T"] / W["dt"])), "K": W["nsave"],
            "parallelism": f"ensemble-shard x{world}",
            "l2": "per-step working set = 1.57 GB of checkpoints per GPU (>> 126 MB L2), no explicit flush",
            "block_threads": block or "auto: ceil32(N / (n_SM * waves)) = 448, one block per SM"}


def host_cores():
    """cores this process may actually run on (the box reports 128 CPUs but the cgroup/affinity mask is smaller)"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:                                                     # cgroup v2 CPU quota (the GPU boxes show 128 CPUs but grant fewer)
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(np.ceil(int(quota) / int(period)))))
    except Exception:
        try:                                                 # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, int(np.ceil(q / per))))
        except Exception:
            pass
    return n


_BEST_THREADS = None


def best_threads():
    """OpenMP thread count that actually maximises the oracle's throughput on this host (affinity masks and CPU quotas
    differ between boxes: probe 8 .. host_cores() on a small sample, keep the best)."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        cap = host_cores()
        cands = sorted({c for c in (4, 8, 16, 32, 64, 128, cap) if c <= cap}) or [1]
        cpu_oracle_rate(256, cands[0])                        # load the library
        rates = {c: cpu_oracle_rate(max(1024, 16 * c), c, repeats=2)[0] for c in cands}
        _BEST_THREADS = max(rates, key=rates.get)
        sys.stderr.write(f"[bench] oracle threads probe: {rates} -> {_BEST_THREADS}\n")
    return _BEST_THREADS


def profile_metric(fname, *names):
    """metrics of a committed ncu summary (profiles/*.json, written by profiles/summarize.py); None when absent"""
    try:
        with open(os.path.join(ROOT, "profiles", fname)) as f:
            m = json.load(f)
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "%": 1.0}
        out = []
        for n in names:
            v = m[n]
            out.append(v["value"] * scale.get(v.get("unit", ""), 1.0))
        return out
    except Exception:
        return None


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the reverse kernel per launch, from the committed ncu capture"""
    for f in ("r2_reverse_ncu_summary.json", "r1_reverse_ncu_summary.json"):
        v = profile_metric(f, "dram__bytes_read.sum", "dram__bytes_write.sum")
        if v is not None:
            return v[0] + v[1], f"profiles/{f} (ncu --set full of this command; not re-measured in this run)"
    return None, None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            m = json.load(f)
        return m.get("hbm_gbs", 6650.0), m.get("bf16_tflops_sustained", 1426.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1426.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, f"/tmp/b200adj_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.device)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)          # a run that dies before stop() must not leave the sampler behind
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        """t_begin/t_end: wall-clock (time.time()) bounds of the timed region; samples outside are dropped."""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        rows = []
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(c[1]), float(c[2]), [name for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[5:9])
                                                            if v.lower().startswith("active")]))
            except ValueError:
                continue
        window = "timed region"
        sel = rows if t_begin is None else [r for r in rows if t_begin - 0.02 <= r[0] <= t_end + 0.02]
        if not sel and rows and t_begin is not None:
            # a timed region shorter than the sampling period (nvidia-smi -lms 20 delivers ~50-100 ms on a busy box): the
            # nearest samples, taken under the load of the warm-up steps just before / the legs just after
            mid = 0.5 * (t_begin + t_end)
            sel = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            window = "nearest samples (%.0f ms from the timed region)" % (1e3 * max(abs(r[0] - mid) for r in sel))
        if sel:
            out.update(sm_mhz=float(np.median([r[1] for r in sel])), sm_max_mhz=float(np.max([r[2] for r in sel])),
                       reasons=sorted({x for r in sel for x in r[3]}), samples=len(sel), window=window)
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


def cpu_oracle_rate(sample_members, threads, repeats=1):
    """members/s of the C oracle (port of the reference algorithm) on `threads` host cores, same workload."""
    from oracle import oracle as O
    W = WORKLOAD
    saveat = np.linspace(0.0, W["T"], W["nsave"])
    u0, p = make_inputs(sample_members)
    cfg = O.make_cfg(W["family"], W["sensealg"], W["stepper"], sample_members, saveat, 0.0, W["T"], dt=W["dt"],
                     cost=("affine",) + W["cost"])
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.gradient(cfg, saveat, u0, p, want_saved=False, nthreads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return sample_members / best, best


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; Julia is not installed, so the
    reference itself cannot run) on all host cores.  Every step is ONE gradient of the same 65536-member ensemble the
    GPU arm evaluates per GPU (same config dict); under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = best_threads()
    sample = args.members or WORKLOAD["members_per_gpu"]
    times = []
    for i in range(args.warmup + args.steps):
        rate, dt = cpu_oracle_rate(sample, threads)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms * 1e-3)
    line = {
        "impl": "reference", "metric": "ensemble adjoint trajectories/sec", "value": value, "unit": "trajectories/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": c2_config(args.gpus, sample, args.block),
        "cpu_baseline": {"value": value, "unit": "trajectories/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} members of the C2 workload per step (one GPU's share), OpenMP over members"},
        "e2e": {"value": value, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------------------
# secondary BASELINE configs (C4, C5) and the generic sharded timing / parity machinery
# ------------------------------------------------------------------------------------------------------------------
def _mlp_params(rng, H=64):
    return np.concatenate([(rng.standard_normal((H, 2)) / np.sqrt(2)).ravel(order="F"), 0.1 * rng.standard_normal(H),
                           (rng.standard_normal((H, H)) / np.sqrt(H)).ravel(order="F"), 0.1 * rng.standard_normal(H),
                           (rng.standard_normal((2, H)) / np.sqrt(H)).ravel(order="F"), 0.1 * rng.standard_normal(2)])


def spec_c4(dtype="bf16_f32acc"):
    T, dt = 1.5, 0.05
    p = _mlp_params(np.random.default_rng(WORKLOAD["seed"]))
    return dict(name="C4 MLP 2->64->64->2 shared weights P=4482, InterpolatingAdjoint, Tsit5 fixed dt=0.05, T=1.5, 30 saves, bf16 tensor-core VJP",
                family="mlp", sensealg="interpolating", stepper="tsit5_fixed", T=T, dt=dt, saveat=np.linspace(0.05, T, 30),
                cost=(1.0, -0.5), dtype=dtype, shared_p=True, okw=dict(mlp_hidden=64), ekw={}, tol=2e-2 if dtype == "bf16_f32acc" else 1e-4,
                inputs=lambda n, off: (np.random.default_rng(1000 + off).uniform(-2, 2, (2, n)), p), parity_members=128, cpu_sample=512,
                # SURVEY 8d: 156 672 flop per member-step of the reverse pass (6 stages x (fwd + 2 VJP GEMM passes))
                roofline=lambda n, S, rev_s, hbm, tf: {"bound": "tensor", "kernel": "mlp_tc_reverse_kernel", "achieved": 156672.0 * n * S / rev_s / 1e12,
                                                       "peak": tf, "unit": "TFLOP/s", "frac": 156672.0 * n * S / rev_s / 1e12 / tf,
                                                       "algorithmic_flops_per_launch": 156672.0 * n * S})


def spec_c5():
    T, dt = 1.0, 0.01
    p = np.array([1.5, 1.0, 3.0, 1.0, 0.1, 0.1])
    return dict(name="C5 SDE-LV diag noise d=2 P=6, BacksolveAdjoint (Ito transformed drift), EM dt=0.01, T=1, saveat 0.01, Philox noise regenerated in reverse",
                family="sde_lv", sensealg="backsolve", stepper="em", T=T, dt=dt, saveat=np.linspace(0.0, T, 101), cost=(0.0, 1.0),
                dtype="f64", shared_p=True, okw={}, ekw=dict(seed=20260923), tol=1e-8,
                inputs=lambda n, off: (np.ones((2, n)), p), parity_members=1024, cpu_sample=131072,
                # SURVEY 8d: 176 B per member-step (z = [lam; mu; y] read+write, checkpoint reset read); compulsory: 16 B
                roofline=lambda n, S, rev_s, hbm, tf: {"bound": "hbm", "kernel": "sde_backsolve_kernel", "achieved": 176.0 * n * S / rev_s / 1e9,
                                                       "peak": hbm, "unit": "GB/s", "frac": 176.0 * n * S / rev_s / 1e9 / hbm,
                                                       "algorithmic_bytes_per_launch": 176.0 * n * S,
                                                       "compulsory_bytes_per_launch": 8.0 * (2 * (S + 1) + 2) * n,
                                                       "note": "per-step accounting (state as if it lived in HBM between steps) is not a bound for an "
                                                               "in-kernel time loop: frac may exceed 1; the compulsory stream is 16 B per member-step"})


def spec_c1():
    """BASELINE configs[0] (LV, InterpolatingAdjoint, ADAPTIVE Tsit5) as an ensemble: every member its own PI-controlled steps."""
    T = 10.0
    p = np.array([1.5, 1.0, 3.0, 1.0])
    tol = dict(abstol=1e-8, reltol=1e-8)
    REC = 8 * 2 + 4       # doubles per member-major record (u_n, k1..k7, t_n, h, 1/h, t_{n+1}): written once, read once
    return dict(name="C1-ensemble Lotka-Volterra d=2 P=4 shared p, InterpolatingAdjoint, adaptive Tsit5 (PI controller) tol 1e-8, T=10, saveat=0.1, loss=sum(sol)",
                family="lv", sensealg="interpolating", stepper="tsit5_adaptive", T=T, dt=0.0, saveat=np.linspace(0.0, T, 101), cost=(0.0, 1.0),
                dtype="f64", shared_p=True, okw=dict(tol), ekw=dict(max_steps=512, **tol), tol=1e-7,
                inputs=lambda n, off: (np.exp(0.2 * np.random.default_rng(3000 + off).standard_normal((2, n))), p), parity_members=256, cpu_sample=16384,
                # compulsory stream: one record per accepted forward step, read once by the reverse solve (TMA bulk copies)
                roofline=lambda n, S, rev_s, hbm, tf: {"bound": "hbm", "kernel": "t5a_reverse_kernel<LotkaVolterra,INTERP>", "achieved": REC * 8.0 * n * S / rev_s / 1e9,
                                                       "peak": hbm, "unit": "GB/s", "frac": REC * 8.0 * n * S / rev_s / 1e9 / hbm,
                                                       "algorithmic_bytes_per_launch": REC * 8.0 * n * S, "mean_forward_steps_per_member": S,
                                                       "note": "latency bound, not bandwidth bound: every member is a serial chain of dependent fp64 work with its own "
                                                               "step sequence (DESIGN.md 4.4); the bytes are the compulsory record stream"})


def spec_c3():
    """BASELINE configs[2]: Robertson, per-member rate constants, QuadratureAdjoint, adaptive Rosenbrock23."""
    T = 100.0
    saveat = np.logspace(-2, 2, 10); saveat[-1] = T
    tol = dict(abstol=1e-8, reltol=1e-8, quad_abstol=1e-10, quad_reltol=1e-10)

    def inputs(n, off):
        k = np.array([0.04, 3e7, 1e4])[:, None] * np.exp(0.05 * np.random.default_rng(4000 + off).standard_normal((3, n)))
        return np.repeat(np.array([[1.0], [0.0], [0.0]]), n, 1), k
    FWD, REV = 10, 12     # doubles per interval of the dense forward (t, u, k1, k2) / reverse (t, h, z, k1, k2, 1/h) solutions
    return dict(name="C3 Robertson d=3 P=3 per-member k, QuadratureAdjoint(1e-10), Rosenbrock23 adaptive tol 1e-8, T=100, 10 log-spaced saves",
                family="robertson", sensealg="quadrature", stepper="rosenbrock23", T=T, dt=0.0, saveat=saveat, cost=(1.0, 0.0),
                dtype="f64", shared_p=False, okw=dict(tol), ekw=dict(max_steps=8192, **tol), tol=1e-5,
                inputs=inputs, parity_members=256, cpu_sample=2048,
                roofline=lambda n, S, rev_s, hbm, tf: {"bound": "hbm", "kernel": "ros23_quadrature_kernel<Robertson> + ros23_reverse_kernel<Robertson,QUAD>",
                                                       "achieved": (FWD + REV) * 8.0 * n * S / rev_s / 1e9, "peak": hbm, "unit": "GB/s",
                                                       "frac": (FWD + REV) * 8.0 * n * S / rev_s / 1e9 / hbm,
                                                       "algorithmic_bytes_per_launch": (FWD + REV) * 8.0 * n * S, "mean_forward_steps_per_member": S,
                                                       "note": "latency bound (adaptive per-member step sequences, warp-per-member quadgk with data-dependent "
                                                               "bisection): the bytes are the dense forward + reverse solutions written and read once, taking "
                                                               "the forward step count for both (DESIGN.md 4.4); BASELINE bound on dp: 1e-5 per member"})


def spec_c2(T=None):
    W = WORKLOAD
    T = T or W["T"]
    nsave = int(round(T / 0.1)) + 1
    return dict(name="C2", family=W["family"], sensealg=W["sensealg"], stepper=W["stepper"], T=T, dt=W["dt"], saveat=np.linspace(0.0, T, nsave),
                cost=W["cost"], dtype="f64", shared_p=True, okw={}, ekw={}, tol=PARITY_TOL,
                inputs=lambda n, off: make_inputs(n, off), parity_members=256)


class Shard:
    """one rank's device-resident engine for a workload spec (+ NCCL communicator behind the C ABI when world > 1)"""

    nccl_allreduce = False        # --nccl-allreduce: A/B against the all-reduce fused into the reverse kernel

    def __init__(self, spec, n_local, rank, world, local, block=0):
        import torch
        import scimlsensitivity_jl_b200 as b
        from scimlsensitivity_jl_b200 import distributed as D
        self.spec, self.n, self.torch = spec, n_local, torch
        self.eng = b.DeviceEnsemble(spec["family"], spec["sensealg"], spec["stepper"], n_local, spec["saveat"], (0.0, spec["T"]), spec["dt"],
                                    on_device=True, device=local, dtype=spec["dtype"], cost=b.AffineCost(*spec["cost"]),
                                    traj_offset=rank * n_local, block_threads=block, nccl_allreduce=Shard.nccl_allreduce,
                                    shared_p=spec.get("shared_p", True), **spec["ekw"])
        self.eng.use_current_torch_stream()
        if world > 1:
            D.attach_comm(self.eng)
        u0, p = spec["inputs"](n_local, rank)
        self.u0_h, self.p_h = u0, p
        td = torch.float64 if spec["dtype"] == "f64" else torch.float32
        dev = f"cuda:{local}"
        self.u0 = torch.tensor(u0, device=dev, dtype=td); self.p = torch.tensor(p, device=dev, dtype=td)
        self.du0 = torch.empty(u0.shape, dtype=td, device=dev); self.dp = torch.empty(p.shape, dtype=td, device=dev)

    def step(self):
        self.eng.handle.forward(self.u0, self.p, None, None, None)
        self.eng.handle.reverse(None, self.du0, self.dp)

    def close(self):
        self.eng.close()


def timed(shard, steps, warmup, barrier, world, dev):
    """W warm-up + K timed gradients; CUDA events on the launching stream; max over ranks -> (ms/step, fwd ms, rev ms)"""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        shard.step()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps + 1)]
    ev[0].record()
    for i in range(steps):
        shard.eng.handle.forward(shard.u0, shard.p, None, None, None); ev[2 * i + 1].record()
        shard.eng.handle.reverse(None, shard.du0, shard.dp); ev[2 * i + 2].record()
    barrier()
    t = torch.tensor([ev[0].elapsed_time(ev[-1]) / steps,
                      float(np.mean([ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(steps)])),
                      float(np.mean([ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(steps)]))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return tuple(float(x) for x in t.cpu())


def parity_pass(spec, rank, world, local, threads):
    """Sub-ensemble of spec['parity_members'] members per rank, sharded exactly like the timed run: every rank computes its
    slice's gradient, dp is all-reduced behind the C ABI; rank 0 recomputes ALL slices with the CPU oracle and compares the
    reduced dp and its own du0.  Returns {dp_rel, du0_rel, members} on rank 0."""
    import torch
    import torch.distributed as dist
    from oracle import oracle as O
    n = spec["parity_members"]
    sh = Shard(spec, n, rank, world, local)
    sh.step()
    torch.cuda.synchronize()
    dp = sh.dp.double().cpu().numpy(); du0 = sh.du0.double().cpu().numpy()
    dW_all = None
    if spec["stepper"] in ("em", "euler_heun"):
        dW = sh.eng.noise()                                    # the Philox increments this shard used (global member index keyed)
        if world > 1:
            parts = [torch.empty_like(dW) for _ in range(world)]
            dist.all_gather(parts, dW.contiguous())
            dW_all = torch.cat(parts, dim=2).cpu().numpy()
        else:
            dW_all = dW.cpu().numpy()
    sh.close()
    if rank != 0:
        return None
    u0s, p = zip(*[spec["inputs"](n, r) for r in range(world)])
    u0 = np.concatenate(u0s, axis=1)
    shared = spec.get("shared_p", True)
    cfg = O.make_cfg(spec["family"], spec["sensealg"], spec["stepper"], n * world, spec["saveat"], 0.0, spec["T"], dt=spec["dt"],
                     cost=("affine",) + tuple(spec["cost"]), shared_p=shared, **spec["okw"])
    ref = O.gradient(cfg, spec["saveat"], u0, p[0] if shared else np.concatenate(p, axis=1), dW=dW_all, want_saved=False, nthreads=threads)
    du0_rel = float(np.abs(du0 - ref["du0"][:, :n]).max() / np.abs(ref["du0"]).max())
    if shared:
        dp_rel = float(np.abs(dp - ref["dp"]).max() / np.abs(ref["dp"]).max())
        against = "CPU oracle (oracle/adjoint_oracle.c) on the same members; dp all-reduced over the ranks by b200adj_reverse"
    else:       # per-member parameters: rank 0's rows, worst member, every row of dp scaled by its own magnitude over the sample
        rdp = ref["dp"][:, :n]
        dp_rel = float((np.abs(dp - rdp) / np.abs(rdp).max(axis=1, keepdims=True)).max())
        against = "CPU oracle (oracle/adjoint_oracle.c) on the same members; per-member dp (no reduction), worst member of rank 0's slice"
    return {"dp_rel": dp_rel, "du0_rel": du0_rel, "members": n * world, "tol": spec["tol"], "ok": bool(dp_rel <= spec["tol"] and du0_rel <= spec["tol"]),
            "against": against}


def cpu_leg_baseline(spec, threads):
    """The C oracle (port of the reference algorithm) on the host cores, on spec['cpu_sample'] members of the same workload."""
    from oracle import oracle as O
    n = spec["cpu_sample"]
    shared = spec.get("shared_p", True)
    u0, p = spec["inputs"](n, 0)
    cfg = O.make_cfg(spec["family"], spec["sensealg"], spec["stepper"], n, spec["saveat"], 0.0, spec["T"], dt=spec["dt"],
                     cost=("affine",) + tuple(spec["cost"]), shared_p=shared, **spec["okw"])
    dW = None
    if spec["stepper"] in ("em", "euler_heun"):        # timing only: any increments of the right law
        S = int(round(spec["T"] / spec["dt"]))
        dW = np.sqrt(spec["dt"]) * np.random.default_rng(1).standard_normal((S, 2, n))
    t0 = time.perf_counter()
    O.gradient(cfg, spec["saveat"], u0, p, dW=dW, want_saved=False, nthreads=threads)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "trajectories/s", "cores": threads, "kind": "port",
            "sample": f"{n} members of the same workload, one gradient, {dt:.2f} s wall"}


def secondary_leg(spec, n_total, rank, world, local, steps, warmup, barrier, threads, with_parity=True):
    import torch
    hbm, tf, _ = peaks()
    dev = f"cuda:{local}"
    n_local = n_total // world
    sh = Shard(spec, n_local, rank, world, local)
    l0 = sh.eng.handle.launch_count
    ms, fwd, rev = timed(sh, steps, warmup, barrier, world, dev)
    launches = sh.eng.handle.launch_count - l0
    S_adaptive = float(sh.eng.step_counts()[0].double().mean().cpu()) if spec["dt"] <= 0 else None      # accepted forward steps per member
    sh.close()
    par = parity_pass(spec, rank, world, local, threads) if with_parity else None
    if rank != 0:
        return None
    S = int(round(spec["T"] / spec["dt"])) if spec["dt"] > 0 else S_adaptive
    out = {"workload": spec["name"], "members_total": n_local * world, "members_per_gpu": n_local, "dtype": spec["dtype"],
           "value": n_local * world / (ms * 1e-3), "unit": "trajectories/s", "ms_per_step": ms,
           "phases_ms": {"forward": fwd, "reverse_incl_allreduce": rev}, "gpu_launches_per_step": launches / max(1, steps + warmup),
           "roofline": spec["roofline"](n_local, S, rev * 1e-3, hbm, tf)}
    if par is not None:
        out["parity"] = par
        out["cpu_baseline"] = cpu_leg_baseline(spec, threads)
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import scimlsensitivity_jl_b200 as b

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    W = WORKLOAD
    N = args.members or W["members_per_gpu"]       # per GPU (weak scaling)
    S = int(round(W["T"] / W["dt"]))
    saveat = np.linspace(0.0, W["T"], W["nsave"])
    cost = b.AffineCost(*W["cost"])
    dev = f"cuda:{local}"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm (`value`) ----------------
    main = Shard(spec_c2(), N, rank, world, local, block=args.block)
    comm_fused = world > 1 and main.eng.handle.comm_is_fused and not args.nccl_allreduce
    eng, u0_h, p_h = main.eng, main.u0_h, main.p_h
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        main.step()
    barrier()
    launches0 = eng.handle.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    barrier()
    wall0 = time.time()
    ev[0].record()
    for i in range(args.steps):
        eng.handle.forward(main.u0, main.p, None, None, None)
        ev[2 * i + 1].record()
        eng.handle.reverse(None, main.du0, main.dp)            # N>1: ends with the NCCL all-reduce of dp on the same stream
        ev[2 * i + 2].record()
    barrier()
    wall1 = time.time()
    total_ms = ev[0].elapsed_time(ev[-1])
    fwd_ms = float(np.mean([ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)]))
    rev_ms = float(np.mean([ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)]))
    launches = eng.handle.launch_count - launches0
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    t = torch.tensor([total_ms, fwd_ms, rev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, fwd_ms, rev_ms = (float(x) for x in t.cpu())
    ms_per_step = total_ms / args.steps
    value = N * world / (ms_per_step * 1e-3)
    dp_check = main.dp.cpu().numpy().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main.du0.cpu().numpy(), main.dp.cpu().numpy())
    main.close()

    # ---------------- end-to-end arms: public API, host buffers ----------------
    u0_pin = torch.tensor(u0_h).pin_memory(); p_pin = torch.tensor(p_h).pin_memory()
    prob = b.EnsembleProblem(b.ODEProblem(W["family"], u0_h[:, 0], (0.0, W["T"]), p_pin.numpy()), u0s=u0_pin.numpy())
    ealg = b.EnsembleB200(device=local, buffers_on_device=False, reuse_handle=True, presharded=True, pin_outputs=True)   # each rank owns its members
    alg = b.Tsit5(dt=W["dt"])
    sens = b.B200Adjoint(b.GaussAdjoint(), block_threads=args.block)

    def step_e2e():
        sol = b.solve(prob, alg, ealg, saveat=saveat, sensealg=sens, save_on=False)
        return b.adjoint_sensitivities(sol, alg, t=saveat, dgdu_discrete=cost, sensealg=b.GaussAdjoint())

    def time_host(fn, nsteps, nwarm):
        for _ in range(nwarm):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(nsteps):
            out = fn()
        barrier()
        s = (time.perf_counter() - t0) / nsteps
        te = torch.tensor([s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.cpu()[0]), out

    e2e_steps = max(1, min(args.steps, 10))
    e2e_s, (du0_e, dp_e) = time_host(step_e2e, e2e_steps, max(1, min(args.warmup, 3)))
    e2e_value = N * world / e2e_s
    h2d = u0_h.nbytes + p_h.nbytes
    d2h = 3 * N * 8 + 3 * 8
    e2e_ok = bool(np.allclose(np.asarray(dp_e).ravel(), np.asarray(dp_check), rtol=1e-12))

    # the plugin seam: _concrete_solve_adjoint -> (primal on the host, pullback(Delta on the host))
    delta_pin = torch.empty((W["nsave"], 3, N), dtype=torch.float64).pin_memory()

    def step_rrule(fill=False):
        out, pullback = b._concrete_solve_adjoint(prob, alg, sens, u0_pin.numpy(), p_pin.numpy(), b.ChainRulesOriginator(),
                                                  saveat=saveat, ensemblealg=ealg)
        if fill:                                                    # the user's loss gradient dL/du(t_k) = u - 2, computed once
            np.subtract(out.u, 2.0, out=delta_pin.numpy())
        return pullback(delta_pin.numpy())

    step_rrule(fill=True)
    rr_steps = max(1, min(args.steps, 5))
    rr_s, tang = time_host(step_rrule, rr_steps, 1)
    rr_ok = bool(np.allclose(np.asarray(tang[4]).ravel(), np.asarray(dp_check), rtol=1e-10))
    kd = W["nsave"] * 3 * N * 8
    b.clear_handle_cache()                                          # frees the host-mode handle (1.6 GB of checkpoints + staging)

    # ---------------- parity of the sharded run against the oracle ----------------
    threads = best_threads() if rank == 0 else 1
    parity = parity_pass(spec_c2(T=2.0), rank, world, local, threads)

    # ---------------- strong scaling of the metric's fixed N = 65536 (N > 1) ----------------
    strong = None
    if world > 1 and not args.members:
        ntot = W["members_per_gpu"]
        sh = Shard(spec_c2(), ntot // world, rank, world, local)
        s_ms, s_f, s_r = timed(sh, args.steps, args.warmup, barrier, world, dev)
        sh.close()
        strong = {"members_total": ntot, "members_per_gpu": ntot // world, "ms_per_step": s_ms, "value": ntot / (s_ms * 1e-3),
                  "unit": "trajectories/s", "phases_ms": {"forward": s_f, "reverse_incl_allreduce": s_r}}

    # ---------------- secondary BASELINE configs, sharded over the same ranks ----------------
    secondary = {}
    if not args.no_secondary and not args.members:
        sec_steps, sec_warm = max(5, min(args.steps, 20)), 3
        few = max(3, min(sec_steps, 5))
        legs = [("c4", spec_c4, 4096, sec_steps, sec_warm, True), ("c4_full", spec_c4, 18944 * world, sec_steps, sec_warm, False),
                ("c5", spec_c5, 131072, sec_steps, sec_warm, True), ("c1_ensemble", spec_c1, 65536 * world, few, 2, True),
                ("c3", spec_c3, 16384, few, 2, True)]
        for key, mk, n_total, k_steps, k_warm, with_par in legs:
            try:
                secondary[key] = secondary_leg(mk(), n_total, rank, world, local, k_steps, k_warm, barrier, threads, with_parity=with_par)
            except Exception as exc:        # a secondary leg must not take the headline down; with several ranks a one-sided
                if world > 1:               # failure would leave the others in a barrier, so there it stays fatal
                    raise
                sys.stderr.write(f"[bench] secondary leg {key} failed: {exc!r}\n")
                secondary[key] = {"error": repr(exc)}

    if rank == 0:
        hbm, tf, peak_src = peaks()
        alg_bytes = ALG_BYTES_PER_MEMBER_STEP * N * S
        achieved = alg_bytes / (rev_ms * 1e-3) / 1e9
        compulsory = 8.0 * (S * 3 + 3) * N                       # checkpoint read + du0 write (affine cost: no cotangent read)
        I = DP_INSTR_PER_MEMBER_STEP
        flops = (2 * I["dfma"] + I["dmul"] + I["dadd"]) * float(N) * S
        dp_issue = (I["dfma"] + I["dmul"] + I["dadd"]) * float(N) * S            # thread-level fp64 instructions per launch
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        nsm = torch.cuda.get_device_properties(local).multi_processor_count
        fp64_peak_tf = nsm * 64 * 2 * sm_mhz * 1e6 / 1e12                         # 64 DFMA/clk/SM
        pipe = profile_metric("r2_reverse_ncu_summary.json", "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active") or \
            profile_metric("r1_reverse_ncu_summary.json", "sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active")
        traffic, traffic_src = ncu_traffic() if N == W["members_per_gpu"] else (None, None)
        cpu_sample = W["members_per_gpu"]
        cpu_oracle_rate(256, threads)                      # warm the library / thread pool
        cpu_rate, cpu_s = cpu_oracle_rate(cpu_sample, threads)
        line = {
            "metric": "ensemble adjoint trajectories/sec", "value": value, "unit": "trajectories/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": c2_config(world, N, args.block),
            "phases_ms": {"forward": fwd_ms, "reverse_incl_allreduce": rev_ms},
            "allreduce": None if world == 1 else ("ncclAllReduce after the reverse kernel (--nccl-allreduce)" if args.nccl_allreduce else
                                                  "fused into the reverse kernel (peer-memory mailboxes)" if comm_fused else
                                                  "ncclAllReduce after the reverse kernel (the GPUs do not map each other)"),
            "roofline": {"bound": "hbm", "kernel": "tsit5_reverse_kernel<Lorenz,GAUSS>", "achieved": achieved, "peak": hbm,
                         "unit": "GB/s", "frac": achieved / hbm,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_member_step": ALG_BYTES_PER_MEMBER_STEP,
                         "compulsory_bytes_per_launch": compulsory,
                         "compulsory_frac": compulsory / (rev_ms * 1e-3) / 1e9 / hbm,
                         "fp64": {"tflops": flops / (rev_ms * 1e-3) / 1e12, "peak_tflops": fp64_peak_tf,
                                  "frac": dp_issue / (rev_ms * 1e-3) / (nsm * 64 * sm_mhz * 1e6),
                                  "pipe_active_pct_ncu": None if pipe is None else pipe[0],
                                  "note": "fp64 pipe: 64 DFMA/clk/SM at the SM clock sampled in this run; frac = issued DFMA+DMUL+DADD / pipe slots "
                                          "(426 per member-step, counted in SASS); pipe_active from the committed ncu capture"},
                         "note": "per-step accounting of SURVEY 8d (state counted as if it lived in HBM between steps); the time "
                                 "loop is in-kernel so real DRAM traffic is the compulsory stream (compulsory_frac of the HBM peak); "
                                 "the binding resource is the fp64 FMA pipe (fp64.frac)"},
            "cpu_baseline": {"value": cpu_rate, "unit": "trajectories/s", "cores": threads, "kind": "port",
                             "sample": f"{cpu_sample} members of the same C2 workload (one GPU's share), one gradient, {cpu_s:.2f} s wall"},
            "e2e": {"value": e2e_value, "unit": "trajectories/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_s * 1e3, "steps": e2e_steps, "api": "solve(EnsembleProblem, Tsit5, EnsembleB200) + adjoint_sensitivities(AffineCost)",
                    "matches_device_arm": e2e_ok},
            "e2e_rrule": {"value": N * world / rr_s, "unit": "trajectories/s", "h2d_bytes_per_step": h2d + kd, "d2h_bytes_per_step": d2h + kd,
                          "ms_per_step": rr_s * 1e3, "steps": rr_steps,
                          "api": "_concrete_solve_adjoint(prob, Tsit5, B200Adjoint(GaussAdjoint)) -> host primal sol.u[K,d,N]; pullback(host Delta[K,d,N])",
                          "matches_device_arm": rr_ok},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "dp": dp_check,
            "parity": parity,
        }
        if strong is not None:
            line["strong"] = strong
        if secondary:
            line["secondary"] = secondary
        emit(line)
        bad = [k for k, v in [("c2", parity)] + [(k, (v or {}).get("parity")) for k, v in secondary.items()] if v is not None and not v["ok"]]
        bad += [k for k, v in secondary.items() if v is not None and "error" in v]
        if bad or not e2e_ok or not rr_ok:
            sys.stderr.write(f"[bench] PARITY FAILURE: {bad} e2e_ok={e2e_ok} rrule_ok={rr_ok}\n")
            if world > 1:
                dist.destroy_process_group()
            sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


def run_secondary(args):
    """--workload c1|c2f32|c3|c4|c5: one BASELINE config alone on one GPU (profiling / tuning; same JSON shape)."""
    import torch
    import scimlsensitivity_jl_b200 as b
    from oracle import oracle as O
    torch.cuda.set_device(0)
    w = args.workload
    rng = np.random.default_rng(WORKLOAD["seed"])
    threads = best_threads()
    if w == "c3":
        N = args.members or 16384
        T = 100.0
        saveat = np.logspace(-2, 2, 10); saveat[-1] = T
        u0 = np.repeat(np.array([[1.0], [0.0], [0.0]]), N, 1)
        p = np.array([0.04, 3e7, 1e4])[:, None] * np.exp(0.05 * rng.standard_normal((3, N)))
        kw = dict(abstol=1e-8, reltol=1e-8, quad_abstol=1e-10, quad_reltol=1e-10)
        eng = b.DeviceEnsemble("robertson", "quadrature", "rosenbrock23", N, saveat, (0.0, T), 0.0, shared_p=False, on_device=True,
                               cost=b.AffineCost(1.0, 0.0), max_steps=8192, **kw)
        ocfg = lambda n: O.make_cfg("robertson", "quadrature", "rosenbrock23", n, saveat, 0.0, T, cost=("affine", 1.0, 0.0), shared_p=False, **kw)
        name, dtype, sample = "C3 Robertson d=3 P=3 per-member k, QuadratureAdjoint(1e-10), Rosenbrock23 adaptive tol 1e-8, T=100, 10 log-spaced saves", "f64", 2048
    elif w == "c1":
        # BASELINE configs[0] (Lotka-Volterra, InterpolatingAdjoint, ADAPTIVE Tsit5 -- the reference's own CPU-runnable case,
        # test/Core1/concrete_solve_derivatives.jl:106-157) as an ensemble: every member runs its own PI-controlled step sequence
        N = args.members or 65536
        T = 10.0
        saveat = np.linspace(0.0, T, 101)
        u0 = np.exp(0.2 * rng.standard_normal((2, N)))
        p = np.array([1.5, 1.0, 3.0, 1.0])
        kw = dict(abstol=1e-8, reltol=1e-8)
        eng = b.DeviceEnsemble("lv", "interpolating", "tsit5_adaptive", N, saveat, (0.0, T), 0.0, on_device=True, cost=b.AffineCost(0.0, 1.0),
                               max_steps=512, block_threads=args.block, **kw)
        ocfg = lambda n: O.make_cfg("lv", "interpolating", "tsit5_adaptive", n, saveat, 0.0, T, cost=("affine", 0.0, 1.0), **kw)
        name, dtype, sample = "C1-ensemble Lotka-Volterra d=2 P=4 shared p, InterpolatingAdjoint, adaptive Tsit5 (PI controller) tol 1e-8, T=10, saveat=0.1, loss=sum(sol)", "f64", 4096
    elif w == "c2f32":
        # the fp32 throughput variant of C2 (SURVEY.md 8d): same ensemble, T = 1 (S = 100, K = 11), fp32 state and tables
        N = args.members or 65536
        T, dt = 1.0, 0.01
        saveat = np.linspace(0.0, T, 11)
        u0, p = make_inputs(N)
        dtype = "f32"
        eng = b.DeviceEnsemble("lorenz", "gauss", "tsit5_fixed", N, saveat, (0.0, T), dt, on_device=True, dtype=dtype, cost=b.AffineCost(1.0, -2.0))
        ocfg = lambda n: O.make_cfg("lorenz", "gauss", "tsit5_fixed", n, saveat, 0.0, T, dt=dt, cost=("affine", 1.0, -2.0))
        name, sample = "C2-fp32 Lorenz d=3 P=3 GaussAdjoint Tsit5 fixed dt=0.01 T=1 saveat=0.1 dgdu=u-2 shared p, fp32 state (fp64 oracle on the CPU side)", 16384
    elif w == "c4":
        N = args.members or 4096
        T, dt = 1.5, 0.05
        saveat = np.linspace(0.05, T, 30)
        u0 = rng.uniform(-2, 2, (2, N))
        H = 64
        p = _mlp_params(rng, H)
        dtype = args.dtype or "bf16_f32acc"       # bf16_f32acc (the named config: tensor-core VJP) | f32 | f64
        eng = b.DeviceEnsemble("mlp", "interpolating", "tsit5_fixed", N, saveat, (0.0, T), dt, on_device=True, dtype=dtype, cost=b.AffineCost(1.0, -0.5))
        ocfg = lambda n: O.make_cfg("mlp", "interpolating", "tsit5_fixed", n, saveat, 0.0, T, dt=dt, cost=("affine", 1.0, -0.5), mlp_hidden=H)
        name, sample = "C4 MLP 2->64->64->2 shared weights P=4482, InterpolatingAdjoint, Tsit5 fixed dt=0.05, T=1.5, 30 saves", 512
    else:
        N = args.members or 131072
        T, dt = 1.0, 0.01
        saveat = np.linspace(0.0, T, 101)
        u0 = np.ones((2, N)); p = np.array([1.5, 1.0, 3.0, 1.0, 0.1, 0.1])
        eng = b.DeviceEnsemble("sde_lv", "backsolve", "em", N, saveat, (0.0, T), dt, on_device=True, cost=b.AffineCost(0.0, 1.0), seed=20260923)
        ocfg = lambda n: O.make_cfg("sde_lv", "backsolve", "em", n, saveat, 0.0, T, dt=dt, cost=("affine", 0.0, 1.0))
        name, dtype, sample = "C5 SDE-LV diag noise d=2 P=6, BacksolveAdjoint (Ito transformed drift), EM dt=0.01, T=1, saveat 0.01, Philox noise regenerated", "f64", 131072
    td = torch.float64 if dtype == "f64" else torch.float32
    u0_d = torch.tensor(u0, device="cuda", dtype=td); p_d = torch.tensor(p, device="cuda", dtype=td)
    du0_d = torch.empty(u0.shape, dtype=td, device="cuda"); dp_d = torch.empty(p.shape, dtype=td, device="cuda")

    def step():
        eng.handle.forward(u0_d, p_d, None, None, None)
        eng.handle.reverse(None, du0_d, dp_d)
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    l0 = eng.handle.launch_count
    ev[0].record()
    for i in range(args.steps):
        eng.handle.forward(u0_d, p_d, None, None, None); ev[2 * i + 1].record()
        eng.handle.reverse(None, du0_d, dp_d); ev[2 * i + 2].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[-1]) / args.steps
    fwd = float(np.mean([ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)]))
    rev = float(np.mean([ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)]))
    # CPU oracle on a bounded sample of the same workload
    cfgs = ocfg(sample)
    dW = None
    if w == "c5":
        dW = np.sqrt(dt) * rng.standard_normal((100, 2, sample))
    pc = p if p.ndim == 1 else p[:, :sample]
    O.gradient(ocfg(min(sample, 16)), saveat, u0[:, :min(sample, 16)], p if p.ndim == 1 else p[:, :min(sample, 16)], dW=None if dW is None else dW[:, :, :min(sample, 16)], want_saved=False, nthreads=threads)
    t0 = time.perf_counter()
    O.gradient(cfgs, saveat, u0[:, :sample], pc, dW=dW, want_saved=False, nthreads=threads)
    cpu_s = time.perf_counter() - t0
    parity = None
    if w in ("c1", "c3"):           # deterministic inputs: the oracle's gradient of the sample vs the device's rows of the same members
        refg = O.gradient(cfgs, saveat, u0[:, :sample], pc, want_saved=False, nthreads=threads)
        du0_h = du0_d.double().cpu().numpy()[:, :sample]
        parity = {"du0_rel": float(np.abs(du0_h - refg["du0"]).max() / np.abs(refg["du0"]).max()), "members": sample}
        if p.ndim == 2:
            parity["dp_rel_worst_member"] = float((np.abs(dp_d.double().cpu().numpy()[:, :sample] - refg["dp"]) / np.abs(refg["dp"]).max(axis=1, keepdims=True)).max())
    line = {"metric": "ensemble adjoint trajectories/sec", "value": N / (ms * 1e-3), "unit": "trajectories/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": {"workload": name, "members_per_gpu": N},
            "phases_ms": {"forward": fwd, "reverse": rev},
            "cpu_baseline": {"value": sample / cpu_s, "unit": "trajectories/s", "cores": threads, "kind": "port",
                             "sample": f"{sample} members of the same workload, one gradient, {cpu_s:.2f} s wall"},
            "gpu_launches": int(eng.handle.launch_count - l0)}
    if parity is not None:
        line["parity"] = parity
    if w == "c1":
        fwd_n, rev_n = [x.cpu().numpy() for x in eng.step_counts()]
        line["steps_per_member"] = {"forward_mean": float(fwd_n.mean()), "forward_max": int(fwd_n.max()), "forward_min": int(fwd_n.min())}
    emit(line)
    eng.close()


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything libraries print (NCCL's version banner, torchrun notices) goes to stderr; stdout carries exactly the
    one JSON line, written through the saved descriptor by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def dump_outputs(out_dir, du0, dp):
    """dp whole; du0 [d, N] at the smallest member stride that keeps it within DUMP_BYTES"""
    os.makedirs(out_dir, exist_ok=True)
    stride = -(-du0.nbytes // DUMP_BYTES)
    np.save(os.path.join(out_dir, "dp.npy"), dp)
    np.save(os.path.join(out_dir, "du0.npy"), np.ascontiguousarray(du0[:, ::stride]))


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members", type=int, default=0, help="override members per GPU (default 65536) / reference sample")
    ap.add_argument("--block", type=int, default=0, help="CUDA block size override (multiple of 32, <= 512)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c1", "c2f32", "c3", "c4", "c5"], help="c2 = BASELINE headline (default)")
    ap.add_argument("--dtype", default="", help="c4 only: bf16_f32acc (default), f32 or f64")
    ap.add_argument("--no-secondary", action="store_true", help="skip the sharded C4 / C5 legs (profiling runs)")
    ap.add_argument("--nccl-allreduce", action="store_true", help="N > 1: ncclAllReduce instead of the fused peer-memory all-reduce (A/B)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write du0 and dp of the last timed C2 step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs applies to the C2 device run (--impl ours --workload c2)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    Shard.nccl_allreduce = args.nccl_allreduce
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload != "c2":
        run_secondary(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
