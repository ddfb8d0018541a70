"""Cost of the privileged critic-state output (ozl_set_states_output) on the x500 step: one JSON line per (N, states off / on).

Per line: us per step, warm (one buffer set, L2-resident where it fits) and cold (rotating buffer sets whose combined footprint
exceeds the 126 MB L2, as profiles/time_sizes.py does), each from CUDA events over >= 200 graph-replayed steps; env-steps/s; the
fraction of a device-to-device copy bandwidth measured in the same run, on 284 B per env-step without the states output and 412 B
with it (+128 B: one 32-float row per env); the GPU name and power limit.  The sizes cover both step kernels (generic up to one
wave of CTAs, the persistent TMA kernel above).  usage: python benchmarks/states_cost.py [sizes...] [--steps K]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from ouzelum_b200 import _lib  # noqa: E402
from ouzelum_b200.sim import QuadSim  # noqa: E402

BYTES = {False: 284, True: 412}
DEV = torch.device("cuda:0")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def copy_gbs():
    """Device-to-device copy bandwidth (read + write bytes / time) of a 2 GiB buffer, best of 5 x 20 copies."""
    src = torch.empty(1 << 29, dtype=torch.float32, device=DEV)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 20 * 1e-3)
    del src, dst
    return 2 * (1 << 31) / best / 1e9


class Shard:
    def __init__(self, n, seed, states):
        self.sim = QuadSim(_lib.default_cfg(n, fault_mode=1, seed=seed), DEV)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=DEV)
        self.bufs = (z(n, 13), z(n), torch.ones(n, dtype=torch.int64, device=DEV), z(n, dtype=torch.int64), z(n, dtype=torch.uint8), z(n))
        self.states = z(n, 32) if states else None
        if states:
            self.sim.set_states_output(self.states)

    def step(self, a):
        self.sim.step(a, *self.bufs)


def graph_time(fn, count, reps=3):
    """us per call of fn(k), k = 0..count-1 captured in one CUDA graph; best of `reps` replays."""
    for k in range(count):
        fn(k)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for k in range(count):
            fn(k)
    g.replay()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(400_000)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e3 / count)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sizes", nargs="*", type=int, default=[16384, 131072, 262144, 1048576])
    ap.add_argument("--steps", type=int, default=200, help="graph-replayed steps per timing (>= 200)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("states_cost.py measures on a CUDA device; none is visible")
    name, power = card()
    bw = copy_gbs()
    for n in args.sizes:
        a = [torch.rand(n, 4, device=DEV) * 2 - 1 for _ in range(2)]
        for states in (False, True):
            per = n * BYTES[states]
            sets = [Shard(n, j, states) for j in range(max(2, int(400e6 // per) + 1))]    # rotating sets: > 400 MB in total
            warm = graph_time(lambda k: sets[0].step(a[k & 1]), args.steps)
            cold = graph_time(lambda k: sets[k % len(sets)].step(a[k & 1]), max(args.steps, 2 * len(sets)))
            gbs = lambda us: per / (us * 1e-6) / 1e9
            print(json.dumps(dict(
                n=n, states=states, kernel="tma" if n // 128 >= 7 * torch.cuda.get_device_properties(0).multi_processor_count + 1
                else "generic", us_per_step_warm=round(warm, 3), us_per_step_cold=round(cold, 3),
                env_steps_per_s_warm=n / (warm * 1e-6), env_steps_per_s_cold=n / (cold * 1e-6),
                bytes_per_env_step=BYTES[states], copy_gbs=round(bw, 1), frac_of_copy_warm=round(gbs(warm) / bw, 3),
                frac_of_copy_cold=round(gbs(cold) / bw, 3), steps=args.steps, gpu=name, power_limit=power)), flush=True)
            for s in sets:
                s.sim.close()
            del sets
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
