"""Step time of BPR's shipped Adam training (K10, csrc/bpr_adam.cuh) at config C1's and C2's shapes; prints one JSON line.

    python tools/bpr_adam_probe.py [--steps 50] [--out FILE]

Per shape (synthetic power-law logs, B = 512 rows x K = 100 negatives, the reference's next_batch):
  * us per step as ONE call over `steps` steps (yue_bpr_adam_steps, losses copied back once), and as the class calls it:
    one step per call and its loss back on the host each time (host clock around calls that end in a device synchronise);
  * the dense Adam pass's byte model, 6 (m + n) ld 4 bytes per step (var, m and v of every row read and written), over the
    peak bandwidth: HBM bandwidth measured in the same run with a device-to-device copy of 4 GiB, and the data sheet's
    7.7 TB/s, each labelled; the step's time over that floor;
  * the GPU's name and power limit, read in the same run;
  * one step of the float64 oracle (oracle/bpr_adam_ref.py) on one host core at C1's shape, for context.
Needs a GPU; there is no CPU fallback.  Builds and caches nothing in the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("OMP_NUM_THREADS", "1")                  # the oracle's step on one host core

import numpy as np  # noqa: E402

DATASHEET_TBS = 7.7            # HGX B200 data sheet, one GPU, HBM3e
SHAPES = [dict(name="C1", users=4000, tracks=50000, plays=100000, d=10),
          dict(name="C2", users=1000000, tracks=200000, plays=50000000, d=64)]
B, K = 512, 100


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                   # noqa: BLE001
        pl = "unknown (%s)" % e
    return name, pl


def copy_bandwidth():
    """Device-to-device copy of 4 GiB (read + write), best of 5: bytes moved / time."""
    import torch
    n = 1 << 30
    a = torch.empty(n, dtype=torch.float32, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    best = None
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    del a, b
    torch.cuda.empty_cache()
    return 2 * 4 * n / (best * 1e-3) / 1e12


def measure(eng, shape, steps, tbs_measured):
    from yue_b200 import synth
    from yue_b200.lightgcn import truncated_normal
    log = synth.power_law_log_torch(shape["users"], shape["tracks"], shape["plays"], seed=20261020)
    eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    rng = np.random.default_rng(1)
    U, V = truncated_normal((log.m, shape["d"]), 0.005, rng), truncated_normal((log.n, shape["d"]), 0.005, rng)
    eng.set_factors(U, V)
    lr, reg, seed = 0.01, 0.01, 7
    eng.bpr_adam_steps(B, K, lr, reg, seed, 0, 3)                    # warm-up: modules, buffers
    s0 = 3
    t0 = time.perf_counter()
    loss = eng.bpr_adam_steps(B, K, lr, reg, seed, s0, s0 + steps)  # returns after the device is done (losses copied back)
    one_call = (time.perf_counter() - t0) / steps
    s0 += steps
    t0 = time.perf_counter()
    for s in range(s0, s0 + steps):
        eng.bpr_adam_steps(B, K, lr, reg, seed, s, s + 1)
    per_call = (time.perf_counter() - t0) / steps
    ld = (shape["d"] + 3) // 4 * 4
    ld = 128 if 64 < ld < 128 else ld
    dense = 6 * (log.m + log.n) * ld * 4
    out = dict(shape=shape["name"], users=log.m, tracks=log.n, train_events=int(log.ev_indptr[-1]), d=shape["d"], ld=ld,
               batch=B, negatives=K, steps=steps, us_per_step_one_call=round(one_call * 1e6, 1),
               us_per_step_one_call_per_step=round(per_call * 1e6, 1), dense_pass_bytes=dense,
               floor_us_measured_copy_bw=round(dense / (tbs_measured * 1e12) * 1e6, 1),
               floor_us_datasheet=round(dense / (DATASHEET_TBS * 1e12) * 1e6, 1),
               loss_first_last=[float(loss[0]), float(loss[-1])])
    out["step_over_floor_measured"] = round(out["us_per_step_one_call"] / out["floor_us_measured_copy_bw"], 2)
    return out, log


def oracle_step(log, d):
    from oracle import bpr_adam_ref as ba
    from yue_b200.lightgcn import truncated_normal
    rng = np.random.default_rng(1)
    U, V = truncated_normal((log.m, d), 0.005, rng), truncated_normal((log.n, d), 0.005, rng)
    t0 = time.perf_counter()
    ba.train(U, V, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, B, K, 0.01, 0.01, 7, 1)
    return round((time.perf_counter() - t0) * 1e6, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bpr_adam_probe: no CUDA device (this probe measures the GPU; there is no CPU fallback)")
    from yue_b200.engine import Engine
    name, power = gpu_info()
    tbs = copy_bandwidth()
    eng = Engine(0)
    res = dict(probe="bpr_adam", gpu=name, power_limit=power, hbm_tbs_measured_d2d_copy=round(tbs, 3),
               hbm_tbs_datasheet=DATASHEET_TBS, shapes=[])
    for sh in SHAPES:
        out, log = measure(eng, sh, a.steps, tbs)
        if sh["name"] == "C1":
            out["oracle_us_per_step_one_core"] = oracle_step(log, sh["d"])
        res["shapes"].append(out)
    eng.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
