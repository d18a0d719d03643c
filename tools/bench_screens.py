"""Cost of one exact screen (unc_eval_screens) against the zOrd-point average it replaces.
2^15 scattered screens of the Cape Cod Moench deck (rD 0.05-3, tD 1e-1-1e6, widths 0.01-0.5,
placed anywhere in [0, 1] so that many cross one or both layer boundaries) through the device
entry, then the same screens as 2 and as 8 points each (linspace over the screen, the
reference's zOrd points) through unc_eval_points_device.  CUDA events around each call after a
warm-up; prints one JSON line with the card's name and power limit.
  python tools/bench_screens.py [log2_screens] [reps] [--out FILE]"""
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


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), [round(x, 3) for x in ms]


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out in args:
        args.remove(out)
    lg = int(args[0]) if args else 15
    reps = int(args[1]) if len(args) > 1 else 5
    n = 1 << lg
    d = deck.read_deck(os.path.join(ROOT, "configs", "cape-cod-moench.in"))
    pd = deck.params_dict(d)
    prm = ub.Params(pd)
    rng = np.random.default_rng(20261020)
    rD = rng.uniform(0.05, 3.0, n)
    tD = 10.0 ** rng.uniform(-1, 6, n)
    wdt = 10.0 ** rng.uniform(-2, np.log10(0.5), n)
    zb = rng.uniform(0.0, 1.0 - wdt)
    zt = zb + wdt
    sv = ub.split_index(tD, (2, 2))
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    nseg = 1 + ((zb < b1) & (zt > b1)).astype(int) + ((zb < b2) & (zt > b2)).astype(int)
    dev = torch.device("cuda", 0)
    g = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=dt)  # noqa: E731
    res = {"workload": f"2^{lg} scattered screens, cape-cod-moench (model 3)", "card": card(),
           "segments_1_2_3": [int((nseg == k).sum()) for k in (1, 2, 3)]}
    s = torch.empty(n, dtype=torch.float64, device=dev); ds = torch.empty_like(s)
    a = [g(tD, torch.float64), g(sv, torch.int32), g(rD, torch.float64), g(zb, torch.float64), g(zt, torch.float64)]
    ms, all_ms = timed(lambda: ub.eval_screens_device(prm, *a, s, ds), reps)
    res["screens"] = {"ms": ms, "us_per_screen": 1e3 * ms / n, "all_ms": all_ms,
                      "finite": float(torch.isfinite(s).float().mean())}
    for k in (2, 8):
        z = (zb[:, None] + wdt[:, None] * np.linspace(0.0, 1.0, k)[None, :]).ravel()
        lay = ub.zlay(z, pd["lD"], pd["dD"])
        m = n * k
        sp = torch.empty(m, dtype=torch.float64, device=dev); dsp = torch.empty_like(sp)
        ap = [g(np.repeat(tD, k), torch.float64), g(np.repeat(sv, k), torch.int32), g(np.repeat(rD, k), torch.float64),
              g(z, torch.float64), g(lay, torch.int32)]
        msp, all_p = timed(lambda: ub.eval_points_device(prm, *ap, sp, dsp), reps)
        res[f"points_x{k}"] = {"ms": msp, "us_per_screen": 1e3 * msp / n, "us_per_point": 1e3 * msp / m,
                               "all_ms": all_p}
    res["screen_over_one_point"] = res["screens"]["ms"] / (res["points_x2"]["ms"] / 2)
    line = json.dumps(res)
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
