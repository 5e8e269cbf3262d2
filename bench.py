#!/usr/bin/env python
"""bench.py -- headline benchmark of the HMC hot path (BASELINE.json metric
"leapfrog-steps*chains/sec").

Workload (configs[1]): 1024-dim dense-covariance Gaussian HMC, 65 536 chains
PER GPU, 50 leapfrog steps, step-size + mass adaptation ON during the timed
steps.  A "step" is one HMC iteration = one ``sample_op()`` call: mass
statistics + update, momentum draw (in-kernel Philox), L+1 fused
GEMM+leapfrog passes, MH test + select, dual-averaging update.

    python bench.py --gpus N --steps K --warmup W            (N=1)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...     CPU arm (torch-CPU restatement)

    python bench.py --scaling strong ...     65 536 chains TOTAL (8 192/GPU at N=8),
                                             the north_star's 8-GPU point
    python bench.py --workload iwae ...      the other half of BASELINE.json's metric:
                                             particle-ELBOs/s, VAE IWAE K=64, batch 4096/GPU
    python bench.py --dump-outputs DIR ...   also write the last timed step's outputs as
                                             DIR/<name>.npy, to compare two builds

Chains shard across ranks with no data-path collective; the only exchange is
ONE packed all-reduce per iteration: [sum acc, n] + the EWMV statistics
[S1(D), S2(D)] of the post-select state (8 B + 8*D B), zhusuan_b200/dist.py.
"""
import argparse
import datetime
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "leapfrog-steps*chains/sec"
UNIT = "chain-steps/s"
DEFAULT_DENSE_IMPL = 5


def make_dense_gaussian_problem(D_, seed=2):
    """Config 2 synthetic target (SURVEY.md 8d): Sigma = A A^T / D + 0.1 I rescaled to unit
    diagonal; returns (precision P float64, const = -1/2 log|2 pi Sigma|)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    A = rng.standard_normal((D_, D_))
    S = A @ A.T / D_ + 0.1 * np.eye(D_)
    d = 1.0 / np.sqrt(np.diag(S))
    S = S * d[:, None] * d[None, :]
    P = np.linalg.inv(S)
    P = 0.5 * (P + P.T)
    _, logdet = np.linalg.slogdet(S)
    return P, -0.5 * (D_ * np.log(2 * np.pi) + logdet)


def host_threads():
    """Threads for the CPU arms: the physical cores (torchrun exports OMP_NUM_THREADS=1, which
    would otherwise leave the reference arm single-threaded at N > 1)."""
    import torch
    n = max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n)
    return torch.get_num_threads()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="hmc", choices=["hmc", "iwae"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --chains-per-gpu on every GPU; strong: "
                         "--total-chains split over the GPUs")
    ap.add_argument("--total-chains", type=int, default=65536)
    ap.add_argument("--chains-per-gpu", type=int, default=65536)
    ap.add_argument("--cuda-graph", action="store_true", default=None,
                    help="replay the step (incl. its all-reduce) from a CUDA graph; default: on "
                         "for --workload iwae (the eager step is host-bound: ~80 launches + "
                         "autograd bookkeeping), off for hmc")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false")
    ap.add_argument("--iwae-batch", type=int, default=4096)
    ap.add_argument("--iwae-particles", type=int, default=64)
    ap.add_argument("--cpu-batch", type=int, default=128)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--leapfrogs", type=int, default=50)
    ap.add_argument("--burnin", type=int, default=20,
                    help="untimed adaptive iterations run as setup, before "
                         "the W warm-up steps (covers both step-size searches)")
    ap.add_argument("--dense-impl", type=int, default=None,
                    help="0 SIMT fp32, 1 tcgen05 3xTF32, 2 tcgen05 fp16-split per "
                         "pass, 4 cluster-of-8 trajectory, 5 L2-resident trajectory "
                         "(default: see DEFAULT_DENSE_IMPL)")
    ap.add_argument("--cpu-chains", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-adapt", action="store_true",
                    help="kernel-timing experiments only: fixed step size, no "
                         "adaptation (not the benchmark configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as "
                         "DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    return args


DUMP_ROWS = 4096


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy in float32 (float64 stays float64).  Arrays with
    more than DUMP_ROWS rows keep the same seeded sample of DUMP_ROWS rows (one per chain or
    datum, aligned across the arrays), so the files stay below 64 MB and two builds run with
    the same arguments can be compared file by file."""
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.dim() > 0 and t.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.Generator(np.random.PCG64(0)).choice(
                t.shape[0], DUMP_ROWS, replace=False))
            t = t[torch.as_tensor(rows, device=t.device)]
        if t.dtype != torch.float64:
            t = t.float()
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf": d.get("bf16_tflops_sustained",
                                                     d["bf16_tflops"]),
                "tf_burst": d["bf16_tflops"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf": 1400.0, "tf_burst": 1590.0,
            "src": "fallback"}


class ClockSampler(object):
    """nvidia-smi clock / throttle-reason sampling DURING the timed region.

    nvidia-smi takes a few hundred ms to produce its first row, so the sampler
    is started ahead of the warm-up and the rows are filtered afterwards by
    their own timestamps against the [mark_begin, mark_end] host-clock window
    of the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,"
         "clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
             "sw_power_cap"]

    def __init__(self, gpu_index, period_ms=50):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.idx = gpu_index
        self.period = period_ms
        self.p = None
        self.windows = {}

    def start(self):
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", str(self.period)],
                stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def wait_first(self, timeout=2.0):
        """Block until nvidia-smi has written its first row (call BEFORE the
        warm-up so the GPU does not idle right ahead of the timed region)."""
        t0 = time.time()
        while self.p is not None and time.time() - t0 < timeout:
            if os.path.getsize(self.f.name) > 0:
                return True
            time.sleep(0.02)
        return False

    def mark_begin(self, name):
        self.windows[name] = [time.time(), None]

    def mark_end(self, name):
        self.windows[name][1] = time.time()

    def stop(self):
        """-> {window name: clocks dict}"""
        if self.p is not None:
            time.sleep(2.5 * self.period * 1e-3)
            self.p.terminate()          # exact PID we started
            try:
                self.p.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
        self.f.flush()
        rows = []
        for line in open(self.f.name):
            r = [x.strip() for x in line.strip().split(",")]
            try:
                ts = datetime.datetime.strptime(
                    r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(r[1]), float(r[2]), float(r[3]),
                             [v.lower() == "active" for v in r[4:8]]))
            except (ValueError, IndexError):
                continue
        os.unlink(self.f.name)
        out = {}
        for name, (t0, t1) in self.windows.items():
            sel = [r for r in rows if t0 <= r[0] <= (t1 or t0)]
            how = "in-window"
            if not sel and rows:       # window shorter than the sampling period
                mid = 0.5 * (t0 + (t1 or t0))
                sel = sorted(rows, key=lambda r: abs(r[0] - mid))[:2]
                how = "nearest"
            if not sel:
                out[name] = {"sm_mhz": None, "sm_max_mhz": None,
                             "reasons": [], "samples": 0}
                continue
            reasons = sorted({n for r in sel
                              for n, v in zip(self.NAMES, r[4]) if v})
            out[name] = {"sm_mhz": float(np.median([r[1] for r in sel])),
                         "sm_max_mhz": float(max(r[2] for r in sel)),
                         "power_w": float(np.median([r[3] for r in sel])),
                         "reasons": reasons, "samples": len(sel),
                         "sampling": how}
        return out


def time_cpu_hmc(args, P=None, n_iters=5, warmup=1):
    """CPU arm of the HMC workload: oracle/cpu_baseline.py (torch-CPU restatement of
    hmc.py:382-522, kind "port": TensorFlow is not installable here) on a bounded chain
    sub-sample; per-iteration times, the MEDIAN is reported (the host also runs the driver)."""
    from oracle.cpu_baseline import time_dense_hmc
    cores = host_threads()
    chains = min(args.cpu_chains, args.chains_per_gpu)
    if P is None:
        P = make_dense_gaussian_problem(args.dim, seed=2)
    rates, ms = [], []
    time_dense_hmc(args.dim, chains, args.leapfrogs, n_iters=warmup, warmup=0, P=P)
    for _ in range(max(1, n_iters)):
        r = time_dense_hmc(args.dim, chains, args.leapfrogs, n_iters=1, warmup=0, P=P)
        rates.append(r["value"]); ms.append(r["ms_per_iter"])
    med = float(np.median(rates))
    return {"value": med, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d chains x %d-d, L=%d, %d timed iteration(s) (median; min %.3g max "
                      "%.3g chain-steps/s), torch-CPU restatement of hmc.py:382-522 (unfused, "
                      "autograd gradient per leapfrog pass)"
                      % (chains, args.dim, args.leapfrogs, len(rates), min(rates), max(rates)),
            "host_cpu_count": os.cpu_count()}, float(np.median(ms))


def time_cpu_iwae(args, n_iters=3):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from bench_iwae import make_cpu_step
    cores = host_threads()
    K, Nc = args.iwae_particles, args.cpu_batch
    rng = np.random.Generator(np.random.PCG64(4))
    xc = torch.tensor(rng.random((Nc, 784)) < 0.13, dtype=torch.float32)
    step = make_cpu_step(xc, K)
    step()
    ts = []
    for _ in range(max(1, n_iters)):
        t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    return {"value": K * Nc / dt, "unit": "particle-ELBOs/s", "cores": cores, "kind": "port",
            "sample": "batch %d of %d, K=%d, %d timed step(s) (median), torch-CPU restatement "
                      "of examples/variational_autoencoders/iwae.py:23-78 (forward + SGVB "
                      "backward)" % (Nc, args.iwae_batch, K, len(ts)),
            "host_cpu_count": os.cpu_count()}, 1e3 * dt


def run_reference(args):
    """--impl reference: the reference's own CPU path.  TensorFlow (and so zhusuan) cannot be
    installed here, so this arm times the torch-CPU restatement (kind "port") with all physical
    host cores on a bounded sub-sample of the same workload (chains / data are independent, so
    the rate is per unit).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "iwae":
        cpu, ms = time_cpu_iwae(args, n_iters=max(1, args.steps))
        metric, unit = "particle-ELBOs/sec", "particle-ELBOs/s"
        wl = ("IWAE, VAE 784-(500,500)-40, K=%d, forward + SGVB backward; CPU sample of %d "
              "data per step" % (args.iwae_particles, args.cpu_batch))
    else:
        cpu, ms = time_cpu_hmc(args, n_iters=max(1, args.steps), warmup=max(1, args.warmup))
        metric, unit = METRIC, UNIT
        wl = ("HMC, %d-dim dense-covariance Gaussian, L=%d; CPU sample of %d chains per step"
              % (args.dim, args.leapfrogs, min(args.cpu_chains, args.chains_per_gpu)))
    out = {
        "impl": "reference", "metric": metric, "value": cpu["value"],
        "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": unit, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "host_cpu_count": os.cpu_count(),
    }
    print(json.dumps(out))


def main():
    args = parse()
    if args.scaling == "strong":
        w = int(os.environ.get("WORLD_SIZE", "1")) if args.impl != "reference" else args.gpus
        args.chains_per_gpu = args.total_chains // max(1, w)
    if args.cuda_graph is None:
        args.cuda_graph = args.workload == "iwae"
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "iwae":
        return run_iwae(args)
    return run_hmc(args)


def run_iwae(args):
    """--workload iwae: the second half of BASELINE.json's metric, particle-ELBOs/s on config 3
    (VAE 784-(500,500)-40, IWAE K=64, batch 4096 per GPU, forward + SGVB reparameterised
    backward; examples/variational_autoencoders/iwae.py:23-78).  Every dense layer runs on the
    tcgen05 fp16-split kernel (fp32 accuracy), the decoder output fused with the Bernoulli
    log-likelihood; the batch axis shards over ranks, particles stay local, ONE packed gradient
    all-reduce per step."""
    import torch
    import torch.distributed as td
    import zhusuan_b200 as zs
    from zhusuan_b200._lib import lib
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from bench_iwae import build, step_fn

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        td.init_process_group("nccl", device_id=dev)
    K, N = args.iwae_particles, args.iwae_batch
    if args.scaling == "strong":
        N = N // world
    rng = np.random.Generator(np.random.PCG64(4 + rank))
    x_host = torch.tensor(rng.random((N, 784)) < 0.13, dtype=torch.int32).pin_memory()
    x = x_host.to(dev)
    W = build(dev)
    zs.set_random_seed(1234 + rank)
    local_step = step_fn(W, x, K, dev, fused=True)
    unit = "particle-ELBOs/s"

    def eager_step():
        cost, g = local_step()
        if world > 1:
            g, (cost,) = zs.dist.all_reduce_mean_gradients(g, [cost.detach()], n_local=N)
        return cost, g

    step = eager_step
    launches_per_replay = None
    if args.cuda_graph:
        # The step (forward, SGVB backward, gradient all-reduce) captured ONCE and replayed: the
        # eager step is bound by the host (~170 launches + autograd bookkeeping per step).  The
        # samplers' Philox counters are frozen by the capture, so the device draw epoch
        # (zs.random.enable_device_epoch) is bumped at the end of the captured step: every
        # replay draws fresh eps.
        zs.random.enable_device_epoch(dev)
        for _ in range(3):
            eager_step()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        c0, l0 = zs.random.counter(), lib.launches
        with torch.cuda.graph(graph):
            g_cost, g_grads = eager_step()
            zs.random.bump_device_epoch(max(1, zs.random.counter() - c0))
        launches_per_replay = lib.launches - l0

        def step():
            graph.replay()
            return g_cost, g_grads

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first()
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    if sampler:
        sampler.mark_begin("timed")
    launches0 = lib.launches
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(args.steps):
        cost, g = step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    if sampler:
        sampler.mark_end("timed")
    if args.dump_outputs and rank == 0:     # before the e2e steps overwrite them
        dump_outputs(args.dump_outputs,
                     dict(cost=cost, **{"grad_" + k: v for k, v in zip(W, g)}))
    launches = lib.launches - launches0
    if launches_per_replay is not None:
        launches = launches_per_replay * args.steps
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        td.all_reduce(ms, op=td.ReduceOp.MAX)
    ms_per_step = float(ms.item()) / args.steps
    value = world * K * N / (ms_per_step * 1e-3)
    bound = float(-cost.detach())

    # e2e: per step, H2D of the step's batch from pinned memory, the step, D2H of the bound
    e2e = None
    if not args.no_e2e:
        cost_host = torch.zeros((), dtype=torch.float32).pin_memory()
        for _ in range(2):
            x.copy_(x_host, non_blocking=True); c, _ = step(); cost_host.copy_(c.detach())
        torch.cuda.synchronize()
        if world > 1:
            td.barrier()
        if sampler:
            sampler.mark_begin("e2e")
        a, b = torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        for _ in range(args.steps):
            x.copy_(x_host, non_blocking=True)
            c, _ = step()
            cost_host.copy_(c.detach(), non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        if sampler:
            sampler.mark_end("e2e")
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        e2e = {"value": world * K * N * args.steps / (float(t.item()) * 1e-3), "unit": unit,
               "h2d_bytes_per_step": N * 784 * 4, "d2h_bytes_per_step": 4,
               "steps": args.steps, "sm_mhz": None}

    def teardown():
        nonlocal step
        if world > 1:
            if args.cuda_graph:        # captured NCCL work must go before the communicator
                step = None
                graph.reset()
            torch.cuda.synchronize()
            td.destroy_process_group()
    if rank != 0:
        teardown()
        return
    win = sampler.stop() if sampler else {}
    if e2e is not None and "e2e" in win:
        e2e["sm_mhz"] = win["e2e"]["sm_mhz"]
    peaks = load_peaks()
    flop_per_unit = 3.97e6          # SURVEY 8d: dense layers, forward + backward, per particle-ELBO
    tfl = flop_per_unit * K * N / (ms_per_step * 1e-3) / 1e12
    roof = {"bound": "tensor", "achieved": tfl, "peak": peaks["tf"], "unit": "TFLOP/s",
            "frac": tfl / peaks["tf"], "traffic": None, "peak_source": peaks["src"],
            "kernel": "linear_tc2_kernel (all dense layers of the step; fp32-equivalent "
                      "FLOPs over the WHOLE step time, per GPU)",
            "algorithmic_flops_per_unit": flop_per_unit,
            "mma_issued_tflops": 3.0 * tfl,
            "mma_issued_frac_of_peak": 3.0 * tfl / peaks["tf"]}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu, _ = time_cpu_iwae(args, n_iters=3)
    out = {
        "metric": "particle-ELBOs/sec", "value": value, "unit": unit, "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": "IWAE, VAE 784-(500,500)-40 (random-init, Glorot), K=%d particles, "
                        "batch %d/GPU (%d total), forward + SGVB backward"
                        % (K, N, N * world),
            "l2": "activations larger than L2 ([K*N, 500] fp32 = %.0f MB per layer)"
                  % (K * N * 500 * 4 / 1e6),
            "cuda_graph": bool(args.cuda_graph),
            "parallelism": "batch sharded x%d, particles local, 1 packed gradient "
                           "all-reduce/step" % world},
        "clocks": win.get("timed"), "e2e": e2e, "gpu_launches": launches,
        "roofline": roof, "cpu_baseline": cpu, "bound_value": bound,
    }
    print(json.dumps(out), flush=True)
    teardown()


def run_hmc(args):
    import torch
    import torch.distributed as td
    import zhusuan_b200 as zs
    from zhusuan_b200._lib import lib

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        td.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1

    D, C, L = args.dim, args.chains_per_gpu, args.leapfrogs
    P, const = make_dense_gaussian_problem(D, seed=2)
    impl = args.dense_impl
    if impl is None:
        impl = DEFAULT_DENSE_IMPL if D % 64 == 0 else (1 if D % 32 == 0 else 0)
    lj = zs.fused.GaussianLogJoint(P, device=dev, impl=impl)
    g = torch.Generator(device=dev)
    g.manual_seed(3 + rank)
    q = torch.randn(C, D, device=dev, generator=g)          # q0 ~ N(0, I)
    if args.no_adapt:
        hmc = zs.HMC(step_size=0.2, n_leapfrogs=L, seed=1234, dense_impl=impl,
                     use_cuda_graph=args.cuda_graph)
    else:
        hmc = zs.HMC(step_size=0.05, n_leapfrogs=L, adapt_step_size=True,
                     adapt_mass=True, mass_collect_iters=10, seed=1234,
                     dense_impl=impl, use_cuda_graph=args.cuda_graph)
    sample_op, info = hmc.sample(lj, {}, {"x": q})

    def step():
        if args.no_adapt:
            sample_op()
        else:
            sample_op(adapt_step_size=True, adapt_mass=True)

    for _ in range(args.burnin):        # setup: adaptive burn-in (untimed)
        step()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()

    # ---------------- timed region: device-resident inputs -------------------
    if sampler:
        sampler.mark_begin("timed")
    hmc._profile_events = []
    launches0 = lib.launches
    coll0 = hmc._pk.n_collectives
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    launches = lib.launches - launches0
    collectives = hmc._pk.n_collectives - coll0
    kern_ms = [a.elapsed_time(b) for a, b in hmc._profile_events]
    hmc._profile_events = None
    if sampler:
        sampler.mark_end("timed")
    if world > 1:
        td.all_reduce(ms, op=td.ReduceOp.MAX)
    total_ms = float(ms.item())
    ms_per_step = total_ms / args.steps
    value = C * world * L * args.steps / (total_ms * 1e-3)
    acc_mean = float(info.acceptance_rate.mean())
    step_size = float(info.updated_step_size)
    if args.dump_outputs and rank == 0:     # before the e2e steps overwrite them
        dump_outputs(args.dump_outputs, {
            "samples_x": info.samples["x"], "init_momentum_x": info.init_momentum["x"],
            "acceptance_rate": info.acceptance_rate,
            "updated_step_size": info.updated_step_size,
            "orig_hamiltonian": info.orig_hamiltonian, "hamiltonian": info.hamiltonian,
            "orig_log_prob": info.orig_log_prob, "log_prob": info.log_prob})

    # ---------------- e2e: host buffers through the public API ---------------
    # Every step: H2D of the step's chain state from pinned host memory, one
    # sample_op() call, D2H of the step's samples + acceptance.  Copies run on
    # two side streams (PCIe is full duplex) one step ahead / behind the compute
    # stream, double-buffered on the device; all of them are inside the timed
    # region and every step's input and output crosses the bus.
    e2e = None
    if not args.no_e2e:
        q_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
        q_host.copy_(q)
        out_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
        acc_host = torch.empty(C, dtype=torch.float32).pin_memory()
        n_e2e = args.steps
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        main = torch.cuda.current_stream()
        stage_in = [torch.empty_like(q), torch.empty_like(q)]
        stage_out, acc_out = torch.empty_like(q), torch.empty(C, device=dev)
        ev_in = [None, None]
        ev_used = [None, None]       # main stream has consumed stage_in[k]
        ev_out_done = None

        def h2d(i):
            with torch.cuda.stream(s_in):
                if ev_used[i % 2] is not None:
                    s_in.wait_event(ev_used[i % 2])
                stage_in[i % 2].copy_(q_host, non_blocking=True)
                ev = torch.cuda.Event(); ev.record(s_in)
            ev_in[i % 2] = ev

        def e2e_loop(n):
            nonlocal ev_out_done
            h2d(0)
            for i in range(n):
                if i + 1 < n:
                    h2d(i + 1)                     # prefetch next step's input
                main.wait_event(ev_in[i % 2])
                q.copy_(stage_in[i % 2])           # D2D into the latent "variable"
                ev_used[i % 2] = torch.cuda.Event(); ev_used[i % 2].record(main)
                step()
                if ev_out_done is not None:
                    main.wait_event(ev_out_done)   # previous D2H has drained stage_out
                stage_out.copy_(info.samples["x"])
                acc_out.copy_(info.acceptance_rate)
                ev_step = torch.cuda.Event(); ev_step.record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_step)
                    out_host.copy_(stage_out, non_blocking=True)
                    acc_host.copy_(acc_out, non_blocking=True)
                    ev_out_done = torch.cuda.Event(); ev_out_done.record(s_out)
            main.wait_event(ev_out_done)
        e2e_loop(2)
        torch.cuda.synchronize()
        if world > 1:
            td.barrier()
        if sampler:
            sampler.mark_begin("e2e")
        a, b = torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        e2e_loop(n_e2e)
        b.record()
        torch.cuda.synchronize()
        if sampler:
            sampler.mark_end("e2e")
        if world > 1:
            td.barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        e2e = {"value": C * world * L * n_e2e / (float(t.item()) * 1e-3),
               "unit": UNIT, "h2d_bytes_per_step": C * D * 4,
               "d2h_bytes_per_step": C * D * 4 + C * 4, "steps": n_e2e,
               "overlap": "H2D/D2H on side streams, double-buffered",
               # the board is power-capped: the SM clock of THIS region (vs
               # clocks.sm_mhz of the device-resident region) explains e2e
               # landing a few % above or below `value`
               "sm_mhz": None}

    if rank != 0:
        if world > 1:
            hmc._graphs.clear()
            torch.cuda.synchronize()
            td.destroy_process_group()
        return
    win = sampler.stop() if sampler else {}
    clocks = win.get("timed")
    if e2e is not None and "e2e" in win:
        e2e["sm_mhz"] = win["e2e"]["sm_mhz"]

    # ---------------- roofline of the dominant kernel ------------------------
    peaks = load_peaks()
    kms = float(np.mean(kern_ms)) / (L + 1) if kern_ms else None
    roof = None
    if kms:
        bytes_per_launch = 16.0 * D * C              # SURVEY 8d: 16*D B/chain-step
        flops_per_launch = 2.0 * D * D * C           # one P.x product
        hbm = bytes_per_launch / (kms * 1e-3) / 1e9
        tfl = flops_per_launch / (kms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            ent = tj.get("impl%d" % impl) or {}
            traffic = ent.get("dram_bytes_per_pass", ent.get("dram_bytes_per_launch"))
            traffic_src = ("STATIC: dram__bytes_read+write of one `ncu --set full` capture "
                           "(%s), per leapfrog pass of 65 536 chains; not measured in this run"
                           % ent.get("source", "profiles/roofline_traffic.json"))
        f_h, f_t = hbm / peaks["hbm_gbs"], tfl / peaks["tf"]
        roof = {"bound": "hbm", "achieved": hbm, "peak": peaks["hbm_gbs"],
                "unit": "GB/s", "frac": f_h, "traffic": traffic,
                "traffic_source": traffic_src,
                "per": "leapfrog pass (one launch of the per-pass kernels; 1/(L+1) of the "
                       "trajectory launch for dense_impl 4/5)",
                "peak_source": peaks["src"],
                "kernel": "dense_leapfrog (impl %d)" % impl,
                "kernel_ms_per_launch": kms,
                "kernel_share_of_step": kms * (L + 1) / ms_per_step,
                "algorithmic_bytes_per_launch": bytes_per_launch,
                "tensor": {"achieved": tfl, "peak": peaks["tf"],
                           "unit": "TFLOP/s (fp32-equivalent 2*D^2 per "
                                   "chain-step vs measured bf16 dense peak)",
                           "frac": f_t}}
        if impl >= 1:
            # what the tensor pipe actually executes: 3 split products per algorithmic
            # product (fp16 for impl 2/3; TF32, half the bf16 rate, for impl 1)
            issued = 3.0 * tfl
            pk = peaks["tf"] if impl >= 2 else peaks["tf"] / 2.0
            roof["tensor"]["mma_issued_tflops"] = issued
            roof["tensor"]["mma_issued_frac_of_peak"] = issued / pk

    # ---------------- CPU baseline on this box's host cores ------------------
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu, _ = time_cpu_hmc(args, P=(P, const), n_iters=5, warmup=1)

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "HMC, %d-dim dense-covariance Gaussian, %d chains/GPU "
                        "(%d total), L=%d, %s"
                        % (D, C, C * world, L,
                           "fixed step size (--no-adapt: NOT the benchmark configuration)"
                           if args.no_adapt else "step-size + mass adaptation on"),
            "chains_per_gpu": C, "dim": D, "n_leapfrogs": L,
            "burnin_iters": args.burnin, "dense_impl": impl,
            "l2": "inputs larger than L2 (q,p = %.0f MB each per GPU vs 126 "
                  "MB L2)" % (C * D * 4 / 1e6),
            "rng": "in-kernel Philox4x32-10",
            "cuda_graph": bool(args.cuda_graph),
            "parallelism": "chains sharded x%d (%s scaling), no data-path collective; "
                           "%d all-reduce(s) of the packed statistics [sum acc, n, S1(D), "
                           "S2(D)] (%d B) in the %d timed iterations"
                           % (world, args.scaling, collectives, 8 + 8 * D, args.steps)},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "collectives_in_timed_region": collectives,
        "roofline": roof, "cpu_baseline": cpu,
        "acceptance_mean": acc_mean, "step_size": step_size,
    }
    print(json.dumps(out), flush=True)
    if world > 1:
        hmc._graphs.clear()             # captured NCCL work must go before the communicator
        torch.cuda.synchronize()
        td.destroy_process_group()


if __name__ == "__main__":
    main()
