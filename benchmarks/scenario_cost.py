"""Cost of a scenario table (ozl_set_scenarios) on the x500 step: one JSON line per (N, table).

Tables: none; all NaN (every group keeps its draw: the scenario kernel runs and loads the row of every resetting env); fully pinned
(every group set: the row replaces every draw).  maxEpisodeLength is 32, so about 1 env in 32 resets per step -- the table is read
only on the reset path (and for a pinned target at the periodic re-samples), so this makes its cost visible.  Per line: us per
step from CUDA events over graph-replayed steps on one L2-warm buffer set, best of 5 replays, the three tables alternated within
each size; resets per step; the GPU name and power limit.  usage: python benchmarks/scenario_cost.py [sizes...] [--steps K] [--out F]"""
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
L = _lib.SCENARIO_LAYOUT


def pinned_rows(n, cfg):
    g = torch.Generator().manual_seed(0)
    u = lambda *s: torch.rand(*s, generator=g)
    r = torch.full((n, _lib.SCENARIO_WIDTH), float("nan"))
    r[:, L["OZL_SCN_POS"]:L["OZL_SCN_POS"] + 3] = torch.stack([u(n) * 2 - 1, u(n) * 2 - 1, u(n) + 1], 1)
    r[:, L["OZL_SCN_QUAT"]:L["OZL_SCN_QUAT"] + 4] = torch.tensor([0.0, 0.0, 0.0, 1.0])
    r[:, L["OZL_SCN_LINVEL"]:L["OZL_SCN_ANGVEL"] + 3] = (u(n, 6) - 0.5) * 0.2
    r[:, L["OZL_SCN_TARGET"]:L["OZL_SCN_TARGET"] + 3] = torch.stack([u(n) * 4 - 2, u(n) * 4 - 2, u(n) + 1], 1)
    r[:, L["OZL_SCN_FAULT_ROTOR"]] = (torch.arange(n) % 4).float()
    r[:, L["OZL_SCN_FAULT_ONSET"]] = (torch.arange(n) % EPISODE).float()
    r[:, L["OZL_SCN_FAULT_EFF"]] = u(n) * 0.5
    nominal = torch.tensor([cfg.mass, cfg.ixx, cfg.iyy, cfg.izz, cfg.arm, 1.0, 0.01])
    r[:, L["OZL_SCN_MASS"]:L["OZL_SCN_YAW_KM"] + 1] = nominal * (0.8 + 0.4 * u(n, 7))
    return r


class Shard:
    def __init__(self, n, table):
        cfg = _lib.default_cfg(n, fault_mode=1, dr_enable=1, max_episode_length=EPISODE, seed=1)
        self.sim = QuadSim(cfg, DEV)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=DEV)
        self.bufs = (z(n, 13), z(n), torch.ones(n, dtype=torch.int64, device=DEV), z(n, dtype=torch.int64), z(n, dtype=torch.uint8), z(n))
        if table == "nan":
            self.sim.set_scenarios(torch.full((n, _lib.SCENARIO_WIDTH), float("nan")))
        elif table == "pinned":
            self.sim.set_scenarios(pinned_rows(n, cfg))

    def step(self, a):
        self.sim.step(a, *self.bufs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("sizes", nargs="*", type=int, default=[16384, 131072, 262144, 1048576])
    ap.add_argument("--steps", type=int, default=200, help="graph-replayed steps per timing (>= 200)")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the three tables per size")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scenario_cost.py measures on a CUDA device; none is visible")
    name, power = card()
    out = open(args.out, "a") if args.out else None
    tables = ("none", "nan", "pinned")
    for n in args.sizes:
        a = [torch.rand(n, 4, device=DEV) * 2 - 1 for _ in range(2)]
        shards = {t: Shard(n, t) for t in tables}
        best = {t: 1e9 for t in tables}
        for _ in range(args.rounds):
            for t in tables:
                best[t] = min(best[t], graph_time(lambda k: shards[t].step(a[k & 1]), args.steps, reps=5))
        for t in tables:
            m = shards[t].sim.metrics().cpu()
            line = json.dumps(dict(
                n=n, table=t, kernel="tma" if n // 128 >= 7 * torch.cuda.get_device_properties(0).multi_processor_count + 1 else "generic",
                us_per_step_warm=round(best[t], 3), delta_vs_none_us=round(best[t] - best["none"], 3),
                resets_per_step=round(float(m[15]) / max(float(m[8]) / n, 1.0), 1), max_episode_length=EPISODE, steps=args.steps,
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
