"""Cost of rotorFault mode "multi" (cfg.fault_mode 2) on the x500 step: one JSON line per (N, fault model).

Fault models: mode 1 (one rotor, the default kernels); mode 2 with rotors [1, 2] and ramp 0; mode 2 with rotors [1, 2] and ramp 200
(the fault_mode 2 kernel twins, which read the env's 16-byte lane of per-rotor effectiveness every step and write it on resets).
maxEpisodeLength is 32, so about 1 env in 32 resets per step and the extra Philox draw of a mode-2 reset is in the numbers.  Per
line: us per step from CUDA events over graph-replayed steps, best of 5 replays, the three models alternated within each size.  The
replays repeat one buffer set, so L2 is warm where the working set fits the 126 MB L2 and overwritten by the step itself where it
does not; each line states its working set.  GPU name and power limit are read in the same run.
usage: python benchmarks/multi_fault_cost.py [sizes...] [--steps K] [--out F]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from benchmarks.states_cost import card, graph_time  # noqa: E402
from ouzelum_b200 import _lib  # noqa: E402
from ouzelum_b200.sim import QuadSim  # noqa: E402

DEV = torch.device("cuda:0")
EPISODE = 32
L2_BYTES = 126e6
# per env-step: state tile 120 B read + 72 B dynamic written (+ static planes on resets), actions 16, obs 52, reward 4, reset 2 x 8,
# progress 2 x 8, time-out 1, episode return 4 (DESIGN.md section 4); mode 2 adds its 16-byte lane read (and written on resets)
BYTES = {"mode1": 297, "mode2_ramp0": 297 + 16, "mode2_ramp200": 297 + 16}
MODELS = {"mode1": dict(fault_mode=1), "mode2_ramp0": dict(fault_mode=2, fault_rotors_lo=1, fault_rotors_hi=2),
          "mode2_ramp200": dict(fault_mode=2, fault_rotors_lo=1, fault_rotors_hi=2, fault_ramp_steps=200)}


class Shard:
    def __init__(self, n, model):
        self.sim = QuadSim(_lib.default_cfg(n, dr_enable=1, max_episode_length=EPISODE, seed=1, **MODELS[model]), DEV)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=DEV)
        self.bufs = (z(n, 13), z(n), torch.ones(n, dtype=torch.int64, device=DEV), z(n, dtype=torch.int64), z(n, dtype=torch.uint8), z(n))

    def step(self, a):
        self.sim.step(a, *self.bufs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sizes", nargs="*", type=int, default=[16384, 131072, 262144, 1048576])
    ap.add_argument("--steps", type=int, default=200, help="graph-replayed steps per timing (>= 200)")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the three fault models per size")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_fault_cost.py measures on a CUDA device; none is visible")
    name, power = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    out = open(args.out, "a") if args.out else None
    for n in args.sizes:
        a = [torch.rand(n, 4, device=DEV) * 2 - 1 for _ in range(2)]
        shards = {m: Shard(n, m) for m in MODELS}
        best = {m: 1e9 for m in MODELS}
        for _ in range(args.rounds):
            for m in MODELS:
                best[m] = min(best[m], graph_time(lambda k: shards[m].step(a[k & 1]), args.steps, reps=5))
        for m in MODELS:
            per_sm = 6 if MODELS[m]["fault_mode"] == 2 else 7          # the mode-2 generic twin is resident 6 CTAs per SM
            kernel = "tma" if n // 128 >= per_sm * sms + 1 else ("subwave" if n <= 4 * 128 * sms else "generic")
            mv = shards[m].sim.metrics().cpu()
            ws = BYTES[m] * n
            line = json.dumps(dict(
                n=n, model=m, kernel=kernel, us_per_step=round(best[m], 3), delta_vs_mode1_pct=round(100 * (best[m] / best["mode1"] - 1), 2),
                resets_per_step=round(float(mv[15]) / max(float(mv[8]) / n, 1.0), 1),
                fault_active_share=round(float(mv[14]) / max(float(mv[8]), 1.0), 3), max_episode_length=EPISODE, steps=args.steps,
                rounds=args.rounds, working_set_mb=round(ws / 1e6, 1),
                l2="warm (working set fits L2, repeated replays)" if ws < L2_BYTES else "overwritten (working set exceeds the 126 MB L2)",
                gpu=name, power_limit=power))
            print(line, flush=True)
            if out:
                out.write(line + "\n")
        for s in shards.values():
            s.sim.close()
        del shards
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
