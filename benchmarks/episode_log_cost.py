"""Cost of the episode log (ozl_set_episode_log) on the x500 step: one JSON line per (N, fault model, maxEpisodeLength, arm).

Fault models: mode 1 (one rotor) and mode 2 (rotors [1, 2], ramp 200); maxEpisodeLength 32 and the default 2000 (with the random
actions used here most episodes end in a crash long before 2000 steps, so both lengths end episodes in most warps every step).  Arms:
  off      the kernels without a log
  on       the log twins with a buffer of one row per env per timed step (an env ends at most one episode per step), so no record is
           ever dropped and every record is written; each line reports `dropped`, which must be 0
  nostore  the log twins with a one-row buffer: every warp still takes its ballot, shuffle and head atomic, but records past row 0
           are dropped, so nearly no record is stored -- on - nostore is the cost of the stores, nostore - off that of the rest
The head is zeroed by each timed graph's first node.  Per line: us per step from CUDA events over graph-replayed steps, best of 5
replays, the three arms alternated within each configuration.  The replays repeat one buffer set, so L2 is warm where the working set fits the 126 MB L2
and overwritten by the step itself where it does not.  GPU name and power limit are read in the same run.
usage: python benchmarks/episode_log_cost.py [sizes...] [--steps K] [--out F]"""
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
MODELS = {"mode1": dict(fault_mode=1), "mode2": dict(fault_mode=2, fault_rotors_lo=1, fault_rotors_hi=2, fault_ramp_steps=200)}
LENGTHS = (32, 2000)
ARMS = ("off", "on", "nostore")
# generic kernels resident per SM, by (fault_mode 2, log): 7 without either, 6 for the mode-2 and log twins
PER_SM = {(False, False): 7, (True, False): 6, (True, True): 6, (False, True): 6}


class Shard:
    def __init__(self, n, model, length, arm, steps):
        self.sim = QuadSim(_lib.default_cfg(n, dr_enable=1, max_episode_length=length, seed=1, **MODELS[model]), DEV)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=DEV)
        self.bufs = (z(n, 13), z(n), torch.ones(n, dtype=torch.int64, device=DEV), z(n, dtype=torch.int64), z(n, dtype=torch.uint8), z(n))
        self.head = None
        if arm != "off":       # "on": an env ends at most one episode per step, so n * steps rows never drop a record
            self.records = z(n * steps if arm == "on" else 1, _lib.EPLOG_WIDTH)
            self.head = z(1, dtype=torch.int64)
            self.sim.set_episode_log(self.records, self.head)

    def step(self, a, k):
        if self.head is not None and k == 0:
            self.head.zero_()
        self.sim.step(a, *self.bufs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sizes", nargs="*", type=int, default=[16384, 131072, 262144, 1048576])
    ap.add_argument("--steps", type=int, default=200, help="graph-replayed steps per timing (>= 200)")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the arms per configuration")
    ap.add_argument("--lengths", type=int, nargs="*", default=list(LENGTHS))
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("episode_log_cost.py measures on a CUDA device; none is visible")
    name, power = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    out = open(args.out, "a") if args.out else None
    for n in args.sizes:
        a = [torch.rand(n, 4, device=DEV) * 2 - 1 for _ in range(2)]
        for model in MODELS:
            for length in args.lengths:
                shards = {arm: Shard(n, model, length, arm, args.steps) for arm in ARMS}
                best = {arm: 1e9 for arm in shards}
                for _ in range(args.rounds):
                    for arm, s in shards.items():
                        best[arm] = min(best[arm], graph_time(lambda k, s=s: s.step(a[k & 1], k), args.steps, reps=5))
                for arm, s in shards.items():
                    log = arm != "off"
                    per_sm = PER_SM[(MODELS[model]["fault_mode"] == 2, log)]
                    kernel = "tma" if n // 128 >= per_sm * sms + 1 else ("subwave" if n <= 4 * 128 * sms else "generic")
                    mv = s.sim.metrics().cpu()
                    rec = {}
                    if log:       # the head counts the records of the last timed replay
                        made = int(s.head.item())
                        rec = dict(records_per_step=round(made / args.steps, 1), dropped=max(made - s.records.shape[0], 0))
                        if arm == "on" and rec["dropped"]:
                            raise SystemExit(f"n={n} {model} length {length}: {rec['dropped']} records dropped by the 'on' arm")
                    line = json.dumps(dict(
                        n=n, model=model, max_episode_length=length, arm=arm, kernel=kernel, us_per_step=round(best[arm], 3),
                        delta_vs_log_off_pct=round(100 * (best[arm] / best["off"] - 1), 2),
                        episodes_per_step=round(float(mv[9]) / max(float(mv[8]) / n, 1.0), 1), **rec, steps=args.steps,
                        rounds=args.rounds, gpu=name, power_limit=power))
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
