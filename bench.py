#!/usr/bin/env python
"""Benchmark of the x500 rotor-fault env-step path (BASELINE.json metric: env-steps/s, whole box).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference [...]                         the reference-structured CPU path (oracle port)
  python bench.py [...] --dump-outputs DIR                       also write the last timed step's outputs (see dump_outputs)

One "step" = one pass of the fused step kernel over every env of every rank, actions read from HBM,
obs / reward / reset / progress written to HBM (SURVEY 8d "mode A").  Workload = BASELINE configs[1]:
x500 tracking with a single-rotor loss-of-effectiveness fault, 16384 envs per GPU (weak scaling).

Timing: W warm-up steps, then EXACTLY K timed steps.  The per-GPU working set at this workload (4.9 MB)
is far below the 126 MB L2, so the K timed steps rotate over 64 independent 16384-env shards (314 MB of state and
buffers > L2: "inputs larger than L2"): every step starts with cold caches and the K steps are block-timed with one
CUDA-event pair, max over ranks.  The same K steps on ONE shard with an explicit L2 flush before each step and per-step
events (`value_flush_per_step_events`), and back to back with a warm L2 (`value_warm_l2`), are reported beside it.  The roofline object is measured live on the same kernel at 1 Mi envs (311 MB
per launch > L2, so no flush is needed there) -- both are labelled.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALG_BYTES_PER_ENV_STEP = 284          # SURVEY.md 8(d): reads 144 + writes 140
WORKLOAD = "x500 trajectory tracking + single-rotor loss-of-effectiveness fault, 16384 envs per GPU (BASELINE configs[1])"
METRIC, UNIT = "env_steps_per_sec", "env-steps/s"
SHARDS = 64                           # independent 16384-env shards the timed steps rotate over (64 x 4.9 MB = 314 MB > 126 MB L2)
METRICS_EVERY = 16                    # BASELINE config 4: metrics vector read (+ NCCL all-reduce when N > 1) every 16 steps
METRICS_PHASE = 4                     # ... after steps 4, 20, 36, ...: the asynchronous all-reduce has the following steps to hide behind (at the driver's K = 20: one read, 15 steps of cover)


def config_of(envs_per_gpu, world):
    """The `config` object, IDENTICAL in both arms (the reference arm runs on the GPU arm's config)."""
    return {"workload": WORKLOAD, "envs_per_gpu": envs_per_gpu, "envs_total": world * envs_per_gpu,
            "mode": "A: actions read from HBM, obs/rew/reset/progress written to HBM",
            "l2": f"inputs larger than L2: the K timed steps rotate over {SHARDS} independent {envs_per_gpu}-env shards "
                  f"({SHARDS} x 4.9 MB = 314 MB > 126 MB L2) and the L2 is overwritten (256 MiB) between the warm-up replay and the "
                  "timed replay, so every timed step starts cold at any K; K steps block-timed with one CUDA-event pair (CUDA graph replay) "
                  "behind a GPU pre-roll that lets the host finish enqueueing before the first event fires",
            "parallelism": f"env-sharded x{world}, no data-path collective; the 16-double metrics vector is read every {METRICS_EVERY} steps "
                           "INSIDE the timed graph and, for N > 1, summed over the ranks inside the same graph (NVLink peer-memory "
                           "exchange issued by the metrics kernel itself, on a side stream forked inside the graph; "
                           "`--metrics-collective nccl`: NCCL all-reduce on a side stream)"}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1000)
    p.add_argument("--warmup", type=int, default=100)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--envs", type=int, default=16384, help="envs per GPU")
    p.add_argument("--roofline-envs", type=int, default=1 << 20)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-side-configs", action="store_true")
    p.add_argument("--metrics-collective", default="peer", choices=["peer", "peer-inline", "nccl", "none"],
                   help="N > 1: how the metrics vector is summed over the ranks inside the timed graph ('none': diagnostic -- "
                        "every rank only reads its own vector, as a one-GPU run does)")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--roofline-only", action="store_true", help="profiling aid: run only the 1 Mi-env roofline region")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return a


DUMP_MAX_BYTES = 64 << 20          # every file of one `--dump-outputs` run together (all ranks), .npy headers included


def _npy_bytes(a):
    """Size of the file `np.save` writes for `a`: the .npy header, then the raw data."""
    import io
    import numpy as np
    f = io.BytesIO()
    np.lib.format.write_array_header_1_0(f, np.lib.format.header_data_from_array_1_0(a))
    return f.tell() + a.nbytes


def dump_outputs(out_dir, per_env, whole=None, suffix="", max_bytes=DUMP_MAX_BYTES):
    """Writes the arrays of `per_env` (name -> tensor with one row per env) and of `whole` (name -> small tensor, written whole)
    as <out_dir>/<name><suffix>.npy, so that two builds can be compared output for output: float64 stays float64, other
    floating outputs become float32 and integer / flag outputs float64.  When the files would exceed `max_bytes` together,
    every per-env array keeps the same fixed, seeded sample of env rows (numpy default_rng(0), sorted)."""
    import numpy as np

    def host(t):
        a = t.detach().cpu().numpy()
        return a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind != "f" else np.float32)
    rows_out = {name: host(t) for name, t in per_env.items()}
    whole = {name: host(t) for name, t in (whole or {}).items()}
    n = len(next(iter(rows_out.values())))
    total = sum(_npy_bytes(a) for a in (*rows_out.values(), *whole.values()))
    if total > max_bytes:
        row_bytes = sum(a.nbytes // n for a in rows_out.values())
        fixed = total - n * row_bytes                  # headers (not longer for fewer rows) and the whole arrays
        rows = np.sort(np.random.default_rng(0).choice(n, (max_bytes - fixed) // row_bytes, replace=False))
        rows_out = {name: a[rows] for name, a in rows_out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in {**rows_out, **whole}.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def task_cfg_kwargs():
    """configs[1]: Ouzelum + rotor fault (rotor = Philox & 3, onset ~ U{0..1999}, effectiveness ~ U(0, 0.5))."""
    return dict(fault_mode=1, fault_eff_lo=0.0, fault_eff_range=0.5, collect_metrics=1)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while a timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.ok = [], set(), False
        self._stop = threading.Event()
        self._active = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:  # noqa: BLE001
                    pass
            time.sleep(0.001)

    def start(self):
        if self.ok:
            self.th.start()

    def region(self, on):
        (self._active.set if on else self._active.clear)()

    def result(self):
        self._stop.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": getattr(self, "max_mhz", None), "reasons": sorted(self.reasons),
                    "note": "no NVML samples inside the timed region"}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------ CPU arm
def _cpu_oracle(n_envs, seed, flavour):
    """flavour "c": the multi-threaded C restatement (oracle/quad_step_c.c, OpenMP over envs) -- the strongest CPU arm;
    flavour "torch": the torch-CPU eager restatement (same op sequence as the reference's Python, oracle/quad_step.py)."""
    import torch
    from oracle.quad_step import QuadStepOracle, default_cfg
    cfg = default_cfg(n_envs, seed=seed, **{k: v for k, v in task_cfg_kwargs().items() if k != "collect_metrics"})
    if flavour == "c":
        try:
            from oracle.c_oracle import COracle, make_cfg
            ora = COracle(make_cfg(QuadStepOracle(cfg).cfg))      # QuadStepOracle rounds the float fields exactly like the struct
            return ora, (lambda a: ora.step(a.numpy()))
        except Exception as e:                                    # no C compiler on the box: fall back to the torch-eager port
            sys.stderr.write(f"[bench] C oracle unavailable ({e!r}); using the torch-eager port\n")
    torch.set_num_threads(os.cpu_count() or 1)
    ora = QuadStepOracle(cfg)
    return ora, ora.step


def cpu_port_rate(n_envs, budget_s, seed, max_steps=None, flavour="c"):
    """Times an oracle port of the reference step on all host threads, on a bounded sample.
    Returns (env-steps/s, steps run, envs per step, threads)."""
    import torch
    threads = os.cpu_count() or 1
    _, step = _cpu_oracle(n_envs, seed, flavour)
    g = torch.Generator().manual_seed(seed)
    acts = [torch.rand(n_envs, 4, generator=g) * 2 - 1 for _ in range(4)]

    class _O:
        pass
    ora = _O()
    ora.step = step
    for k in range(2):
        ora.step(acts[k])                       # warm-up (allocator, thread pool)
    t0 = time.perf_counter()
    ora.step(acts[2])
    per = max(time.perf_counter() - t0, 1e-4)
    steps = max(3, int(budget_s / per))
    if max_steps:
        steps = min(steps, max_steps)
    t0 = time.perf_counter()
    for k in range(steps):
        ora.step(acts[k & 3])
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, steps, n_envs, threads


def run_reference(args):
    """`--impl reference`: the reference's own step cannot run here or on the GPU box (Isaac Gym / PhysX is a closed
    binary that is not in the reference tree; see DESIGN.md), so the arm times the oracle PORT of it -- the same
    torch-eager op sequence on the host cores -- on our arm's workload.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.envs * max(1, int(os.environ.get("WORLD_SIZE", "1")))     # whole-job workload of the GPU arm (weak scaling)
    # bound the run: K+W steps of the full workload if that fits ~2 minutes, else a smaller env sample per step
    import torch
    threads = os.cpu_count() or 1

    def mk(m):
        return _cpu_oracle(m, args.seed, "c")[1]
    probe = mk(n)
    a = torch.rand(n, 4) * 2 - 1
    probe(a)
    t0 = time.perf_counter()
    probe(a)
    per = time.perf_counter() - t0
    total = per * (args.steps + args.warmup)
    sample = n
    if total > 120.0:
        sample = max(256, int(n * 120.0 / total) // 256 * 256)
    step = mk(sample)
    g = torch.Generator().manual_seed(args.seed)
    acts = [torch.rand(sample, 4, generator=g) * 2 - 1 for _ in range(4)]
    for k in range(args.warmup):
        step(acts[k & 3])
    t0 = time.perf_counter()
    for k in range(args.steps):
        step(acts[k & 3])
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.envs, max(1, int(os.environ.get("WORLD_SIZE", "1")))),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps x {sample} envs of the workload (host cores only; the whole-job workload is {n} envs per step)",
                         "note": "CPU restatement of the reference step (PhysX unavailable): C port of the oracle, OpenMP over envs, all host threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import ouzelum_b200
    from ouzelum_b200 import _lib
    from ouzelum_b200.sim import QuadSim
    from ouzelum_b200.dist import allreduce_metrics, bind_to_gpu_numa_node, rank_info

    rank, world, local = rank_info()
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = bind_to_gpu_numa_node(local)      # before any pinned allocation: host buffers land on the GPU's own NUMA node
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.envs
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = _lib.default_cfg(n, seed=args.seed, env_id_base=rank * n, **task_cfg_kwargs())
    sim = QuadSim(cfg, dev)
    obs = torch.zeros(n, 13, device=dev)
    rew = torch.zeros(n, device=dev)
    reset = torch.ones(n, dtype=torch.int64, device=dev)
    prog = torch.zeros(n, dtype=torch.int64, device=dev)
    tout = torch.zeros(n, dtype=torch.uint8, device=dev)
    epr = torch.zeros(n, device=dev)
    g = torch.Generator(device=dev).manual_seed(args.seed + rank)
    pool = [torch.rand(n, 4, device=dev, generator=g) * 2 - 1 for _ in range(8)]   # synthetic actions, resident in HBM
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)                  # > 126 MB L2
    metrics_dev = torch.zeros(16, dtype=torch.float64, device=dev)
    side = torch.cuda.Stream(device=dev)

    def step(k):
        sim.step(pool[k & 7], obs, rew, reset, prog, tout, epr)

    def metrics_allreduce():
        # config 4: the ONLY collective on the path -- a 16-double metrics vector, every 16 steps, off the step stream
        sim.metrics(clear=False, out=metrics_dev)
        if world > 1:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                allreduce_metrics(metrics_dev)

    clocks = ClockSampler(local)
    clocks.start()
    if args.roofline_only:
        K, W = 1, 1
        args.no_e2e = args.no_cpu_baseline = args.no_side_configs = True

    # ---- headline: EXACTLY K steps, block-timed; every step's inputs are cold because (a) the steps rotate over S independent
    #      16384-env shards whose combined footprint (S x 4.9 MB) exceeds the 126 MB L2 and (b) the L2 is overwritten between the
    #      warm-up replay and the timed replay (K < S would otherwise re-touch warm shards).  The metrics vector is read every 16
    #      steps inside the graph and, for N > 1, summed over the ranks inside the same graph (config 4's only collective: NVLink
    #      peer-memory exchange issued by the metrics kernel, or an NCCL all-reduce on a side stream).  A ~0.4 ms GPU pre-roll sits in front of the first event so the host has enqueued every graph launch
    #      before the timed region begins: the event pair sees device time only, no host launch gaps.
    S = SHARDS
    shards = [(sim, obs, rew, reset, prog, tout, epr)]
    # one allocation per buffer kind, sliced per shard (keeps the ncu launch list free of hundreds of fill kernels)
    b_obs, b_rew, b_epr = torch.zeros(S, n, 13, device=dev), torch.zeros(S, n, device=dev), torch.zeros(S, n, device=dev)
    b_rst, b_prog = torch.ones(S, n, dtype=torch.int64, device=dev), torch.zeros(S, n, dtype=torch.int64, device=dev)
    b_tout = torch.zeros(S, n, dtype=torch.uint8, device=dev)
    for j in range(1, S):
        shards.append((QuadSim(_lib.default_cfg(n, seed=args.seed + j, env_id_base=(rank * S + j) * n, **task_cfg_kwargs()), dev),
                       b_obs[j], b_rew[j], b_rst[j], b_prog[j], b_tout[j], b_epr[j]))
    rendezvous = torch.zeros(1, device=dev)
    n_reads = (K + METRICS_EVERY - 1) // METRICS_EVERY + 1
    metrics_ring = torch.zeros(n_reads, 16, dtype=torch.float64, device=dev)
    # config 4's only collective, the sum of the 16-double metrics vector over the ranks: NVLink peer-memory exchange issued by the
    # metrics-read kernel itself (ouzelum_b200/csrc/peer_metrics.cu); `--metrics-collective nccl` keeps the NCCL all-reduce on a
    # side stream for comparison
    collective = "none"
    peer = None
    peer_on_side = False
    if world > 1:
        collective = args.metrics_collective
        # "peer": the exchange kernels run on a side stream forked inside the graph (SURVEY 8e: "issued on a side stream ... consumed
        # asynchronously"), off the chain of step launches -- K = 20, 2 GPUs: 90.2 us for the 20 steps vs 92.2-94.2 with the kernels in
        # the chain ("peer-inline") and 88.1 without any collective.  Every step of this bench runs on its own handle (rotating
        # shards), so the side-stream read of a handle's metrics never overlaps a step on that handle.
        peer_on_side = collective == "peer"
        if collective == "peer-inline":
            collective = "peer"
        if collective == "peer":
            from ouzelum_b200.dist import PeerMetrics
            try:
                peer = PeerMetrics(dev, connect=False)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] rank {rank}: metrics mailbox could not be created ({e!r})\n")
                peer = None
            flag = torch.tensor([1 if peer is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 1:
                try:
                    peer._connect_ipc()                      # collective; raises on EVERY rank if any rank failed
                except Exception as e:  # noqa: BLE001 -- no cudaIpc between the ranks on this box: fall back to NCCL, and say so
                    sys.stderr.write(f"[bench] rank {rank}: peer-memory metrics exchange unavailable ({e!r}); using NCCL\n")
                    peer = None
            else:
                peer = None
            if peer is None:
                collective = "nccl"
    nccl_in_graph = collective == "nccl"
    metrics_sum = torch.zeros(16, dtype=torch.float64, device=dev)

    def step_rot(k):
        sm, o_, r_, rs_, pg_, to_, er_ = shards[k % S]
        sm.step(pool[k & 7], o_, r_, rs_, pg_, to_, er_)

    forked = [False]

    def metrics_in_graph(k, with_nccl):
        # one metrics_read kernel on the step stream; the all-reduce forks to the side stream and joins at the end of the capture
        m = metrics_ring[(k // METRICS_EVERY) % n_reads]
        if peer is not None:
            # ONE launch: read + 16-byte stores into every rank's mailbox over NVLink; the sum of the previous exchange is folded in
            if peer_on_side:
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    peer.push(shards[k % S][0], local=m, prev_sum=metrics_sum)
                forked[0] = True
                return
            peer.push(shards[k % S][0], local=m, prev_sum=metrics_sum)
            return
        shards[k % S][0].metrics(clear=False, out=m)
        if with_nccl:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                dist.all_reduce(m, op=dist.ReduceOp.SUM)
            forked[0] = True

    for k in range(max(W, S)):
        step_rot(k)

    def graph_of(step_fn, count, k0=0, extra=None):
        g_ = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        forked[0] = False
        with torch.cuda.graph(g_, capture_error_mode="thread_local"):
            for k in range(k0, k0 + count):
                step_fn(k)
                if extra is not None and (k % METRICS_EVERY) == METRICS_PHASE:
                    extra(k)
            if peer is not None and extra is not None and peer_on_side and forked[0]:
                with torch.cuda.stream(side):
                    peer.sum(shards[0][0], out=metrics_sum)
            if forked[0]:
                torch.cuda.current_stream().wait_stream(side)     # join the side stream the all-reduces were forked to
                forked[0] = False
            if peer is not None and extra is not None and not peer_on_side:
                peer.sum(shards[0][0], out=metrics_sum)           # the last exchange of the capture is summed inside it
        return g_

    chunk_r = K if K <= 512 else 512
    reps_r, rem_r = K // chunk_r, K % chunk_r

    def build_headline(with_nccl):
        ex = (lambda k: metrics_in_graph(k, with_nccl))
        g1 = graph_of(step_rot, chunk_r, 0, ex)
        g2 = graph_of(step_rot, rem_r, reps_r * chunk_r, ex) if rem_r else None    # the remainder is graph-launched too: EXACTLY K steps
        return g1, g2
    try:
        gr_rot, gr_rot_rem = build_headline(nccl_in_graph)
    except Exception as e:  # noqa: BLE001  -- NCCL capture refused on this stack: keep the metrics read, drop the in-graph all-reduce
        sys.stderr.write(f"[bench] rank {rank}: NCCL all-reduce could not be captured ({e!r}); timing without it\n")
        nccl_in_graph = False
        torch.cuda.synchronize()
        gr_rot, gr_rot_rem = build_headline(False)
    if world > 1:      # every rank must agree on what was captured
        flag = torch.tensor([1 if nccl_in_graph else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and nccl_in_graph:
            nccl_in_graph = False
            gr_rot, gr_rot_rem = build_headline(False)
    n_metric_reads = sum(1 for k in range(K) if (k % METRICS_EVERY) == METRICS_PHASE)
    n_peer_sums = (reps_r + (1 if rem_r else 0)) if peer is not None else 0
    clocks.region(True)          # NVML sampling (1 ms period) runs from here to the end of the warm-L2 region: the timed replay alone
    gr_rot.replay()              # (K x ~4 us) is shorter than one NVML query, so the window also covers the warm-up replays around it
    if gr_rot_rem is not None:
        gr_rot_rem.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush.zero_()                                   # overwrite the L2: the warm-up replay touched the same shards the timed one will
    torch.cuda._sleep(800_000)                      # ~0.4 ms spin kernel: the host enqueues everything below while it runs
    if world > 1:
        # device-side rendezvous: the host barrier above releases the ranks' HOSTS ~0.2 ms apart, and the all-reduce inside the timed
        # graph would charge that start skew to every rank but the last (measured at 8 GPUs, K = 20: 15.9 instead of 4.4 us per step)
        dist.all_reduce(rendezvous)
    e0.record()
    for _ in range(reps_r):
        gr_rot.replay()
    if gr_rot_rem is not None:
        gr_rot_rem.replay()
    e1.record()
    barrier()
    tr = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    per_rank_ms = [float(tr.item())]
    if world > 1:
        gathered = [torch.zeros_like(tr) for _ in range(world)]
        dist.all_gather(gathered, tr)
        per_rank_ms = [float(t_.item()) for t_ in gathered]
        dist.all_reduce(tr, op=dist.ReduceOp.MAX)
    rot_ms = float(tr.item())
    value_rot = world * n * K / (rot_ms * 1e-3)
    if args.dump_outputs:
        # what the caller of the timed path holds after it: the per-env outputs of timed step K - 1 (its shard's buffers are not
        # touched again before this), the last metrics vector read inside the timed graph and, with the peer exchange, the sum
        # over the ranks it produced.  Graph 1 (steps 0 .. chunk_r - 1) is replayed reps_r times, then graph 2 runs the rest.
        _, o_, r_, rs_, pg_, to_, er_ = shards[(K - 1) % S]
        reads = [k for k in range(reps_r * chunk_r, K) if (k % METRICS_EVERY) == METRICS_PHASE] or \
                [k for k in range(chunk_r) if (k % METRICS_EVERY) == METRICS_PHASE]
        whole = {"metrics": metrics_ring[(reads[-1] // METRICS_EVERY) % n_reads]} if reads else {}
        if peer is not None:
            whole["metrics_sum"] = metrics_sum
        dump_outputs(args.dump_outputs, {"obs": o_, "reward": r_, "reset": rs_, "progress": pg_, "time_outs": to_,
                                         "episode_return": er_}, whole, f"_rank{rank}" if world > 1 else "",
                     DUMP_MAX_BYTES // world)
    peer_check = None
    if peer is not None:
        # outside the timed region: the sum the last in-graph exchange produced equals an NCCL all-reduce of the vectors it was fed
        last_k = max(k for k in range(K) if (k % METRICS_EVERY) == METRICS_PHASE) if n_metric_reads else None
        if last_k is not None:
            ref = metrics_ring[(last_k // METRICS_EVERY) % n_reads].clone()
            gathered = [torch.zeros_like(ref) for _ in range(world)]
            dist.all_gather(gathered, ref)
            want = torch.zeros_like(ref)
            for g_ in gathered:
                want += g_
            st_ = peer.status()
            okf = torch.tensor([1 if (torch.equal(metrics_sum, want) and st_["error"] == 0) else 0], device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            peer_check = {"sum_equals_rank_ordered_allgather_sum_on_every_rank": bool(okf.item()),
                          "env_steps_in_summed_vector": float(metrics_sum[8].item()), "exchanges": st_["pushed"]}
    del gr_rot, gr_rot_rem
    shards = shards[:1]
    del b_obs, b_rew, b_epr, b_rst, b_prog, b_tout

    # ---- same K steps on ONE shard, L2 flushed (256 MiB overwritten) before each step, per-step CUDA events -------------------
    for k in range(W):
        step(k)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    for k in range(K):
        flush.zero_()
        ev[k][0].record()
        step(k)
        ev[k][1].record()
        if (k & 15) == 15:
            metrics_allreduce()
    barrier()
    ms = sum(s.elapsed_time(e) for s, e in ev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.cuda.current_stream().wait_stream(side)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value_flush = world * n * K / (ms * 1e-3)
    value = value_rot

    # ---- warm-L2 variant (what a resident 16k-env rollout actually sees): CUDA graph of back-to-back steps ---------
    chunk = K if K <= 500 else 500
    reps, rem = K // chunk, K % chunk
    gr = graph_of(step, chunk)
    gr_rem = graph_of(step, rem) if rem else None
    gr.replay()
    if gr_rem is not None:
        gr_rem.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(800_000)
    e0.record()
    for _ in range(reps):
        gr.replay()
    if gr_rem is not None:
        gr_rem.replay()
    e1.record()
    barrier()
    clocks.region(False)
    tw = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
    warm_ms = float(tw.item())
    value_warm = world * n * K / (warm_ms * 1e-3)

    # ---- e2e through the public API (make -> VecTask.step) with HOST buffers ---------------------------------------
    e2e = None
    if not args.no_e2e:
        tc = ouzelum_b200.task_config("Ouzelum", n, rotorFault={"enable": True}, seed=args.seed, envIdBase=rank * n)
        env = ouzelum_b200.make(seed=args.seed, task="Ouzelum", num_envs=n, sim_device=str(dev), rl_device=str(dev),
                                headless=True, cfg=tc)
        env.reset()
        h_act = [(torch.rand(n, 4) * 2 - 1).pin_memory() for _ in range(4)]
        d_act = torch.empty(n, 4, device=dev)
        h_obs = torch.empty(n, 13).pin_memory()
        h_rew = torch.empty(n).pin_memory()
        h_rst = torch.empty(n, dtype=torch.int64).pin_memory()

        def e2e_step(k):
            d_act.copy_(h_act[k & 3], non_blocking=True)
            o, r, d, _ = env.step(d_act)
            h_obs.copy_(o["obs"], non_blocking=True)
            h_rew.copy_(r, non_blocking=True)
            h_rst.copy_(d, non_blocking=True)
            torch.cuda.current_stream().synchronize()      # the host consumes the result before the next action

        def e2e_step_host(k):
            # public host-consumer API: the kernel reads the pinned actions and writes pinned obs / reward / done in place
            # (zero-copy over PCIe); step_host() returns after a stream synchronise, results are valid on the host
            env.step_host(h_act[k & 3])

        e2e_ranks = {}

        # untimed host-path warm-up: like the headline's max(W, S) pre-roll.  The host <-> device round trip keeps getting faster for
        # the first ~200 steps (8 ms) of a run -- measured at K = 20: 40.6-41.2 us per step after 5 warm-up steps, 39.8-42.0 after 64,
        # 37.7 after 256 = the K = 1000 figure (profiles/r02an_*) -- so the steady state is what gets timed; the count is in the line
        W_e2e = max(W, int(os.environ.get("OZL_BENCH_E2E_WARMUP", "256")))

        def timed(fn, tag=None):
            for k in range(W_e2e):
                fn(k)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            lat = []
            e0.record()
            for k in range(K):
                t0 = time.perf_counter()
                fn(k)
                lat.append(time.perf_counter() - t0)
            e1.record()
            barrier()
            te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if tag is not None:
                lat.sort()
                mine = torch.tensor([float(te.item()) / K * 1e3, lat[len(lat) // 2] * 1e6, lat[min(len(lat) - 1, int(0.99 * len(lat)))] * 1e6],
                                    dtype=torch.float64, device=dev)
                allr = [mine.clone() for _ in range(world)]
                if world > 1:
                    dist.all_gather(allr, mine)
                e2e_ranks[tag] = [{"rank": r_, "us_per_step_device": float(v[0]), "host_p50_us": float(v[1]), "host_p99_us": float(v[2])}
                                  for r_, v in enumerate(allr)]
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return world * n * K / (float(te.item()) * 1e-3)

        v_copy = timed(e2e_step)
        v_host = timed(e2e_step_host, "step_host")
        env.close()
        # EnvPool-style pipelining for a consumer that can work on halves: two task objects of n/2 envs on two streams; while the
        # host consumes half A's results and writes its next actions, half B's step (action reads, compute, PCIe write-back) runs
        half = n // 2
        halves = []
        for hx in range(2):
            tch = ouzelum_b200.task_config("Ouzelum", half, rotorFault={"enable": True}, seed=args.seed, envIdBase=rank * n + hx * half)
            eh = ouzelum_b200.make(seed=args.seed, task="Ouzelum", num_envs=half, sim_device=str(dev), rl_device=str(dev),
                                   headless=True, cfg=tch)
            eh.reset()
            halves.append((eh, torch.cuda.Stream(device=dev), [(torch.rand(half, 4) * 2 - 1).pin_memory() for _ in range(4)]))
        for eh, st_, ah in halves:
            eh.step_host_async(ah[0], st_)
        for eh, _, _ in halves:
            eh.step_host_wait()

        def e2e_step_halves(k):
            # one "step" = both halves advanced once (n env-steps); each wait is followed at once by that half's next launch
            for eh, st_, ah in halves:
                eh.step_host_wait()
                eh.step_host_async(ah[k & 3], st_)
        v_halves = timed(e2e_step_halves)
        for eh, _, _ in halves:
            eh.step_host_wait()
            eh.close()
        e2e = {"value": v_host, "unit": UNIT, "warmup_steps": W_e2e,
               "h2d_bytes_per_step": world * h_act[0].numel() * 4,
               "d2h_bytes_per_step": world * (n * 13 * 4 + n * 4 + n * 8 + n),
               "api": "ouzelum_b200.make(...).step_host(pinned actions) -> pinned (obs f32 [N,13], reward f32 [N], reset int64 [N]; + the same flags as u8): one launch, zero-copy PCIe reads/writes inside the kernel, stream sync",
               "per_rank": e2e_ranks.get("step_host"), "numa_cpus_rank0": (f"{numa_cpus[0]}-{numa_cpus[-1]} ({len(numa_cpus)} cpus)" if numa_cpus else None),
               "value_pipelined_two_halves": v_halves,
               "pipelined_two_halves": "two task objects of n/2 envs on two streams, step_host_async / step_host_wait: one half's PCIe write-back overlaps the other half's step (for consumers that can work on halves; not the reference's synchronous step)",
               "value_with_explicit_copies": v_copy,
               "explicit_copies": {"api": "make(...).step(device actions) bracketed by cudaMemcpyAsync pinned->device / device->pinned + sync",
                                   "d2h_bytes_per_step": world * (h_obs.numel() * 4 + h_rew.numel() * 4 + h_rst.numel() * 8)}}

    # ---- roofline of the dominant (only) kernel, live, at an L2-exceeding size ------------------------------------
    roofline = roofline_wl = None
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            traffic = json.load(f)
    except Exception:  # noqa: BLE001
        pass
    if rank == 0:
        nb = args.roofline_envs
        del flush
        cfgb = _lib.default_cfg(nb, seed=args.seed, **task_cfg_kwargs())
        simb = QuadSim(cfgb, dev)
        ob, rb = torch.zeros(nb, 13, device=dev), torch.zeros(nb, device=dev)
        rsb, pb = torch.ones(nb, dtype=torch.int64, device=dev), torch.zeros(nb, dtype=torch.int64, device=dev)
        tb, eb = torch.zeros(nb, dtype=torch.uint8, device=dev), torch.zeros(nb, device=dev)
        ab = [torch.rand(nb, 4, device=dev) * 2 - 1 for _ in range(2)]
        for k in range(10):
            simb.step(ab[k & 1], ob, rb, rsb, pb, tb, eb)
        reps_b = 50
        gb = graph_of(lambda k: simb.step(ab[k & 1], ob, rb, rsb, pb, tb, eb), reps_b)     # launches back to back, no host gaps
        gb.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.region(True)
        e0.record()
        gb.replay()
        e1.record()
        torch.cuda.synchronize()
        clocks.region(False)
        per_launch_s = e0.elapsed_time(e1) * 1e-3 / reps_b
        del gb
        ach = ALG_BYTES_PER_ENV_STEP * nb / per_launch_s / 1e9
        roofline = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                    "kernel": "quad_step_tma_kernel (persistent, TMA-pipelined; the same step as quad_step_kernel<128> which serves one-wave sizes, N <= 132608)", "n_envs": nb, "launch_us": per_launch_s * 1e6,
                    "alg_bytes_per_env_step": ALG_BYTES_PER_ENV_STEP, "peak_source": peak_src,
                    "l2": "inputs (311 MB/launch) exceed the 126 MB L2; no flush; 50 launches replayed from a CUDA graph, one event pair",
                    "env_steps_per_sec_at_this_size": nb / per_launch_s}
        del simb, ob, rb, rsb, pb, tb, eb, ab
        # the same measurement over the shard sizes of BASELINE config 4 (1 Mi envs over 8 / 4 / 2 / 1 GPUs) and 4 Mi: how the
        # step approaches the HBM roofline as a launch grows (<= 262144 envs fit the 126 MB L2 when replayed on one buffer set)
        sweep = []
        if not args.roofline_only:
            for ns in (131072, 262144, 524288, 4194304):
                sm_ = QuadSim(_lib.default_cfg(ns, seed=args.seed, **task_cfg_kwargs()), dev)
                o_, r_ = torch.zeros(ns, 13, device=dev), torch.zeros(ns, device=dev)
                rs_, p_ = torch.ones(ns, dtype=torch.int64, device=dev), torch.zeros(ns, dtype=torch.int64, device=dev)
                t_, e_ = torch.zeros(ns, dtype=torch.uint8, device=dev), torch.zeros(ns, device=dev)
                a_ = torch.rand(ns, 4, device=dev) * 2 - 1
                for _ in range(10):
                    sm_.step(a_, o_, r_, rs_, p_, t_, e_)
                reps_s = 40
                gs_ = graph_of(lambda k: sm_.step(a_, o_, r_, rs_, p_, t_, e_), reps_s)
                gs_.replay()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                gs_.replay()
                e1.record()
                torch.cuda.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / reps_s
                del gs_
                sweep.append({"n_envs": ns, "launch_us": us, "frac": ALG_BYTES_PER_ENV_STEP * ns / (us * 1e-6) / 1e9 / peak,
                              "l2": "fits L2 (warm)" if ns * 297 < 120e6 else "exceeds L2"})
                del sm_, o_, r_, rs_, p_, t_, e_, a_
        roofline["sweep"] = sweep
        ach_wl = ALG_BYTES_PER_ENV_STEP * n / (rot_ms * 1e-3 / K) / 1e9
        roofline_wl = {"bound": "launch/latency (4.9 MB per launch, one partial wave)", "achieved": ach_wl, "peak": peak,
                       "unit": "GB/s", "frac": ach_wl / peak, "n_envs": n, "launch_us": rot_ms * 1e3 / K}

    # ---- CPU baseline beside it (rank 0, N=1 only) -------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)         # the CPU arm gets every host core again (the GPU arm was bound to one NUMA node)
        v, steps_c, envs_c, threads = cpu_port_rate(n, budget_s=8.0, seed=args.seed, flavour="c")
        vt, steps_t, envs_t, _ = cpu_port_rate(n, budget_s=6.0, seed=args.seed, flavour="torch")
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{steps_c} steps x {envs_c} envs (C restatement of the reference step, OpenMP over envs; PhysX unavailable)",
               "torch_eager_port": {"value": vt, "sample": f"{steps_t} steps x {envs_t} envs (torch-CPU eager restatement, the reference's own op-by-op style)"}}

    # ---- the other BASELINE configs, driver-visible (configs 1 and 3 on one GPU; config 5 on every rank, max over ranks) -------
    side_configs = None
    if not args.no_side_configs:
        try:
            from benchmarks import configs as side
            side_configs = {}
            torch.cuda.set_device(local)
            c5 = side.config5(str(dev), iters=8)
            if rank == 0:
                side_configs["config5_rpo_lstm_rollout_collection"] = c5
            if world == 1:
                side_configs["config1_quadcopter_hover_256"] = side.config1(str(dev))
                side_configs["config3_ekf_pv_lee_65536"] = side.config3(str(dev), steps=100)
        except Exception as e:  # noqa: BLE001 -- a side line must never take the headline down
            side_configs = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": rot_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_of(n, world),
            "ms_per_rank": per_rank_ms,
            "metrics_reads_in_timed_graph": n_metric_reads, "nccl_allreduce_in_timed_graph": bool(nccl_in_graph),
            "metrics_collective_in_timed_graph": collective, "peer_exchange": peer_check,
            "value_flush_per_step_events": value_flush, "ms_per_step_flush_per_step_events": ms / K,
            "value_warm_l2": value_warm, "ms_per_step_warm_l2": warm_ms / K,
            "clocks": clocks.result(),
            "e2e": e2e, "gpu_launches": K + n_metric_reads + n_peer_sums,
            "gpu_launches_note": f"{K} quad_step_kernel<128> + {n_metric_reads} "
                                 + ("metrics_push_kernel (read + NVLink peer stores" + (", side stream)" if peer_on_side else ")") if collective == "peer" else "metrics_read_kernel")
                                 + (f" + {n_peer_sums} metrics_sum_kernel" if n_peer_sums else "")
                                 + " per rank inside the timed region"
                                 + (f" (+ {n_metric_reads} NCCL all-reduce kernels, library)" if nccl_in_graph else ""),
            "side_configs": side_configs,
            "roofline": roofline, "roofline_at_workload": roofline_wl,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
