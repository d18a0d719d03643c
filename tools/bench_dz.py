"""Cost of the vertical gradient (unc_eval_points_dz) against the drawdown at the same points
(unc_eval_points).  2^15 scattered points of the Cape Cod Neuman 1974 deck (model 5; rD 0.05-3,
tD 1e-1-1e6, zD uniform in [0, 1], so every layer occurs) through the device entries, the two
calls alternated in the same run, CUDA events around each call after a warm-up, median of the
repetitions.  Prints one JSON line with the card's name and power limit, read in the same run;
with --out DIR also writes it to DIR/dz_bench.json (nothing is written into the source tree).
  python tools/bench_dz.py [--log2 N] [--reps R] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import unconfined_b200 as ub  # noqa: E402
from oracle import deck  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return q


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", type=int, default=15)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n = 1 << a.log2
    d = deck.read_deck(os.path.join(ROOT, "configs", "cape-cod-neuman74.in"))
    pd = deck.params_dict(d)
    prm = ub.Params(pd)
    rng = np.random.default_rng(20261021)
    rD = rng.uniform(0.05, 3.0, n)
    tD = 10.0 ** rng.uniform(-1, 6, n)
    zD = rng.uniform(0.0, 1.0, n)
    sv = ub.split_index(tD, (2, 2))
    lay = ub.zlay(zD, pd["lD"], pd["dD"])
    dev = torch.device("cuda", 0)
    ub.set_device(0)
    g = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x)).to(dev, dtype=dt)  # noqa: E731
    t_, s_, r_, z_, l_ = (g(tD, torch.float64), g(sv, torch.int32), g(rD, torch.float64), g(zD, torch.float64),
                          g(lay, torch.int32))
    gz = torch.empty(n, dtype=torch.float64, device=dev); dgz = torch.empty_like(gz)
    s = torch.empty_like(gz); ds = torch.empty_like(gz)
    run_dz = lambda: ub.eval_points_dz_device(prm, t_, s_, r_, z_, gz, dgz)  # noqa: E731
    run_pt = lambda: ub.eval_points_device(prm, t_, s_, r_, z_, l_, s, ds)  # noqa: E731
    res = {"workload": f"2^{a.log2} scattered points, cape-cod-neuman74 (model 5)", "card": card(),
           "layers_1_2_3": [int((lay == k).sum()) for k in (1, 2, 3)]}
    run_dz(); run_pt()
    torch.cuda.synchronize()
    ms_dz, ms_pt = [], []
    for _ in range(a.reps):
        ms_dz.append(event_ms(run_dz))
        ms_pt.append(event_ms(run_pt))
    mdz, mpt = float(np.median(ms_dz)), float(np.median(ms_pt))
    res["dz"] = {"ms": mdz, "us_per_point": 1e3 * mdz / n, "all_ms": [round(x, 3) for x in ms_dz],
                 "finite": float(torch.isfinite(gz).float().mean())}
    res["points"] = {"ms": mpt, "us_per_point": 1e3 * mpt / n, "all_ms": [round(x, 3) for x in ms_pt],
                     "finite": float(torch.isfinite(s).float().mean())}
    res["dz_over_point"] = mdz / mpt
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "dz_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
