#!/usr/bin/env python
"""bench.py -- BPR SGD triplets/s (headline) and top-N ranked users/s on B200.

    python bench.py [--gpus N --steps K --warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--steps K --warmup W]    # the reference's CPU path

A *step* is one SGD epoch of the hot path (recommender/cf/BPR.py:42-58) over the whole
synthetic play log of BASELINE.json configs[1] (C2: 1 M users x 200 K tracks x 50 M plays,
d = 64) resident in HBM; at N > 1 every rank owns its own C2-shaped user shard (weak scaling),
Q is replicated and the ranks reconcile Q deltas with one NCCL all-reduce per step
(SURVEY.md section 8e).  `value` times K steps on the device (CUDA events on the library's
stream, max over ranks).  `e2e` times the same step through the host-facing C ABI with host
buffers: upload of the log and of P/Q from pinned memory, one epoch, download of P/Q and the loss.
`roofline` is the SGD kernel against the measured HBM copy bandwidth with the algorithmic bytes
of SURVEY.md 8(d): 6*d*4 + 12 = 1548 B per triplet at d = 64.  `cpu_baseline` / `--impl
reference` time the oracle's port of the reference's numpy loop (the reference ships that loop
commented out and has nothing to compile, see DESIGN.md) on the host cores.
One JSON line on stdout (rank 0).  `--dump-outputs DIR` also writes the factor tables the last timed step left (see
dump_tables); the inputs are seeded, so runs with the same arguments start from the same log and tables.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bpr_sgd_triplets_per_sec"
UNIT = "triplets/s"
SEED = 20260103            # SEED_BASE + config# (C2 -> 2, +1 so that rank offsets never collide with C1)
LR, REG_U, REG_I = 0.02, 0.01, 0.01          # config/BPR.conf
D = 64                                       # set by --config (C2: 64, C3: 128)


def bytes_per_triplet(d):
    """SURVEY.md 8(d): 3 rows read + 3 rows written + positive id + amortised play-row probe."""
    return 6 * d * 4 + 12


def workload(small, config="C2", world=1):
    if config == "C3":
        # BASELINE.json configs[2]: ONE log of 10 M users x 2 M tracks x 1 B plays, d = 128, user-sharded over the ranks
        # (strong scaling: a rank holds 1/world of the users and of the plays; Q, 1.02 GB, is replicated)
        u, t, p = (10_000_000, 2_000_000, 1_000_000_000) if not small else (200_000, 50_000, 8_000_000)
        return dict(name="C3: BPR d=128, 10M users x 2M tracks x 1B plays, user-sharded over %d GPU(s) (synthetic power-law log, "
                         "each rank generates its shard)" % world, users=u // world, tracks=t, plays=p // world, d=128, scaling="strong")
    if small:
        return dict(name="C2-small (debug)", users=50_000, tracks=20_000, plays=2_000_000, d=64, scaling="weak")
    return dict(name="C2: BPR d=64, 1M users x 200K tracks x 50M plays (synthetic power-law log)",
                users=1_000_000, tracks=200_000, plays=50_000_000, d=64, scaling="weak")


def sgd_kernel_name(d):
    """The kernel yue_bpr_epoch launches in Hogwild mode for rows of d floats (yue_b200.cu: use_blk_kernel)."""
    ld = (d + 3) & ~3
    if ld > 128:
        return "bpr_sgd_kernel<%d, kAtomic>" % ((ld // 4 + 15) // 16)
    v = 1 if ld <= 32 else 2 if ld <= 64 else 4
    return "bpr_sgd_blk_kernel<%d, false, %s>" % (v, "true" if ld != 32 * v else "false")


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the SGD kernel on this workload, from the committed
    ncu --set full capture of the same command (profiles/ncu_traffic.json names the report each figure comes from).
    Not measurable inside a timed run (no profiler under a bench number); null when no capture exists for the config."""
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(tpath):
        return None, None
    ent = json.load(open(tpath)).get(key)
    if not ent:
        return None, None
    return ent.get("dram_bytes_per_launch"), ent.get("source")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), float(j.get("bf16_tflops", 1551.4)), "measured"
    return 6650.0, 1590.0, "fallback"


DUMP_TABLE_BYTES = 24 << 20     # --dump-outputs: at most this much of each factor table


def dump_tables(out_dir, P, Q):
    """--dump-outputs: the factor tables the timed steps left, i.e. what yue_get_factors hands a caller of the epoch, as
    out_dir/P.npy and out_dir/Q.npy in float32.  A table larger than DUMP_TABLE_BYTES is cut to a fixed sample of its rows
    (seeded, the same rows for the same shape, kept in row order), so that two builds can be compared row for row.
    The Hogwild epoch is not reproducible (warps read rows while others add to them, in an order the hardware picks), so
    two runs of ONE build differ too, although their inputs are byte-identical.  Measured on a B200 at config C2: one
    epoch from the same tables already differs by 2 % of the table norm (median row 0.1 % in P, 2 % in Q); after
    3 warm-up + 10 timed steps the median row differs by 0.2 % in P and 1.4 % in Q, the worst by 13 % and 26 %."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("P", P), ("Q", Q)):
        k = min(len(t), DUMP_TABLE_BYTES // (4 * t.shape[1]))
        if k < len(t):
            t = t[np.sort(np.random.default_rng(SEED).choice(len(t), k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(t, dtype=np.float32))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t_mark = index, [], None, None

    def start(self):
        """Started BEFORE the warm-up steps: nvidia-smi needs a few hundred ms to deliver its first line, more than a short
        timed region lasts (10 epochs of config C2 are 130 ms); mark() is called where the timed region begins."""
        if os.environ.get("YUE_BENCH_NO_CLOCKS"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("YUE_BENCH_CLOCKS_MS", "50")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [x.strip() for x in line.split(",")]))

    def wait_ready(self, timeout=2.0):
        """Block until nvidia-smi has delivered its first line (call BEFORE the barrier that precedes the timed region)."""
        t0 = time.monotonic()
        while self.proc and not self.rows and time.monotonic() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        self.t_mark = time.monotonic()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.monotonic()
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        t0 = self.t_mark if self.t_mark is not None else 0.0
        timed = [r for t, r in self.rows if t0 <= t <= t_end + 0.06]      # a line describes the ~50 ms before it arrived
        window = "timed region"
        if not timed:                                                     # region shorter than a sampling period
            timed, window = [r for _, r in self.rows], "warm-up + timed region (the timed region is shorter than a sampling period)"
        sm, mx, reasons = [], [], set()
        for r in timed:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle's port of BPR.py:31-62 on a bounded sample
# ------------------------------------------------------------------------------------------
def cpu_sample(log, n_triplets, d, seed):
    """A user-strided sample (keeps the degree mix) of about n_triplets events, as a sub-log."""
    from yue_b200 import synth
    deg = np.diff(log.ev_indptr)
    stride = max(1, int(log.train_size / max(n_triplets, 1)))
    users = np.arange(stride // 2, log.m, stride)
    keep_ev = np.concatenate([np.arange(log.ev_indptr[u], log.ev_indptr[u + 1]) for u in users])
    keep_uq = np.concatenate([np.arange(log.uq_indptr[u], log.uq_indptr[u + 1]) for u in users])
    ev_indptr = np.concatenate([[0], np.cumsum(deg[users])]).astype(np.int64)
    uq_indptr = np.concatenate([[0], np.cumsum(np.diff(log.uq_indptr)[users])]).astype(np.int64)
    P, Q = synth.init_factors(len(users), log.n, d, seed)
    return dict(ev_user=np.repeat(np.arange(len(users), dtype=np.int32), deg[users]),
                ev_items=log.ev_items[keep_ev], uq_indptr=uq_indptr, uq_items=log.uq_items[keep_uq],
                P=P, Q=Q, n=log.n, T=int(len(keep_ev)))


def cpu_epoch(sample, epoch):
    """One pass of the reference loop (oracle port: float32 numpy rows, Python scalars, per-triplet
    rejection sampling) -- 1 thread, the loop is inherently serial."""
    from oracle import bpr_ref, philox
    t0 = time.perf_counter()
    neg = philox.sample_negatives(SEED, epoch, sample["ev_user"], sample["n"], sample["uq_indptr"], sample["uq_items"])
    bpr_ref.sgd_epoch(sample["P"], sample["Q"], sample["ev_user"], sample["ev_items"], neg, LR, REG_U, REG_I)
    return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from yue_b200 import synth
    # C3: the sample is drawn from one of 8 shards of the log (generating 1 B plays to sample 60 K of them would take
    # longer than the whole arm); the degree mix and the catalog are the full config's
    wl = workload(args.small, args.config, 8 if args.config == "C3" else 1)
    D = wl["d"]
    per_step = 60_000                      # ~1.5-2 s of CPU per step at ~4e4 triplets/s
    log = synth.power_law_log_torch(wl["users"], wl["tracks"], wl["plays"], SEED) \
        if not args.small else synth.power_law_log(wl["users"], wl["tracks"], wl["plays"], SEED, test_ratio=0)
    sample = cpu_sample(log, per_step, D, SEED)
    for w in range(args.warmup):
        cpu_epoch(sample, w)
    t = sum(cpu_epoch(sample, args.warmup + k) for k in range(args.steps))
    if args.dump_outputs:
        dump_tables(args.dump_outputs, sample["P"], sample["Q"])
    value = sample["T"] * args.steps / t
    desc = "%d-triplet user-strided sample of the workload per step, oracle port of BPR.py:31-62" % sample["T"]
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload(args.small, args.config, max(1, args.gpus))["name"], "d": D, "triplets_per_step_per_gpu": wl["plays"], "lr": LR, "reg": [REG_U, REG_I],
                   "sgd_mode": "serial (the reference's loop order)", "parallelism": "1 host core (the loop is inherently serial)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc,
                         "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------
def run_native(args):
    import torch
    import torch.distributed as dist
    from yue_b200 import quality, sharding, synth
    from yue_b200.engine import MODE_HOGWILD, MODE_HOGWILD_STORE, MODE_SERIAL, Engine, PinnedArray

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "8")   # the exchange runs UNDER the next sub-epoch on the SMs the epoch kernel leaves free
        dist.init_process_group("nccl", device_id=dev)
    wl = workload(args.small, args.config, world)
    d = wl["d"]
    mode = MODE_HOGWILD_STORE if args.sgd_mode == "store" else MODE_HOGWILD
    hbm_peak, bf16_peak, peak_kind = peaks()
    bpt = bytes_per_triplet(d)

    log = synth.power_law_log_torch(wl["users"], wl["tracks"], wl["plays"], SEED + rank, device="cuda")
    T = log.train_size
    m, n = log.m, log.n
    torch.cuda.empty_cache()
    eng = Engine(local)
    # the host copy of the play log lives in pinned memory (DMA source of the e2e step)
    pins = []
    for name in ("ev_indptr", "ev_items", "uq_indptr", "uq_items"):
        a = getattr(log, name)
        pa = PinnedArray(a.shape, a.dtype)
        pa.array[:] = a
        setattr(log, name, pa.array)
        pins.append(pa)
    pP, pQ = PinnedArray((m, d), np.float32), PinnedArray((n, d), np.float32)
    P0, Q0 = synth.init_factors(m, n, d, SEED + 1000 + rank)
    if world > 1:                                   # Q is replicated: same init everywhere
        Q0 = synth.init_factors(1, n, d, SEED + 999)[1]
    pP.array[:], pQ.array[:] = P0, Q0
    # every rank owns its own users (weak scaling at C2: a C2-shaped shard each; strong at C3: 1/world of the one log);
    # global event indices keep the ranks' sampler streams apart
    user_begin, event_base = rank * m, rank * T
    local_counts = np.bincount(log.ev_items, minlength=n)

    def upload():
        eng.set_interactions(m, n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items,
                             user_begin=user_begin, event_base=event_base)
        eng.set_factors(pP.array, pQ.array)

    def barrier():
        eng.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def allmax(x):
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    upload()

    # ---- dominant kernel alone, one GPU's plain epochs (no collective): per-launch duration for the roofline ----
    for w in range(2):
        eng.bpr_epoch(LR, REG_U, REG_I, SEED, 900 + w, mode, want_loss=False)
    kms = []
    for k in range(max(3, min(args.steps, 10))):
        eng.sync()
        eng.timer_start()
        eng.bpr_epoch(LR, REG_U, REG_I, SEED, 1000 + k, mode, want_loss=False)
        kms.append(eng.timer_stop())
    k_ms = float(np.mean(kms))
    eng.set_factors(pP.array, pQ.array)             # the timed steps below start from the initial tables

    # ---- N > 1: N REPLICAS -- every GPU trains its own model on its own C2-shaped log (cross-validation folds, seeds,
    #      hyper-parameter points: host/driver.py maps -cv folds to devices), no collective.  Why not one sharded model:
    #      DESIGN.md section 6 -- at this log's skew any schedule that keeps Recall/NDCG within 0.5 points of the serial
    #      order is bound by how many updates of one row may be in flight, and N GPUs cannot beat one.  The sharded
    #      trainer is measured below (`sharded`), with its own quality verdict. ----
    ctl = sharding.TorchCtl(dist, dev) if world > 1 else None
    reduce_factory = quality.torch_reduce_factory(dist, dev) if world > 1 else None

    # config C3 IS the sharded one ("user-sharded SGD with Q-delta allreduce at 2/4/8 B200"): there the trainer is the headline,
    # with the quality caveat spelled out in the line
    headline_sharded = args.config == "C3" and world > 1

    def make_trainer():
        # plain sum of the tail deltas, the defaults of sharding.SharedHotTrainer (up to 248 shared rows, parts and asynchrony by
        # the number of ranks): the schedule that is inside the gate at this size on 2 and 4 GPUs (profiles/r2/quality_c2_n*_hot.log)
        return sharding.SharedHotTrainer(eng, ctl, local_counts, sub_epochs=args.sub_epochs, asynchrony=args.asynchrony or None,
                                         reduce=reduce_factory(eng), reserve_sms=args.reserve_sms)

    trainer = make_trainer() if headline_sharded else None

    def step(epoch, want_loss=False):
        if trainer is not None:
            return trainer.epoch(LR, REG_U, REG_I, SEED, epoch, want_loss=want_loss)
        return eng.bpr_epoch(LR, REG_U, REG_I, SEED, epoch, mode, want_loss=want_loss)

    # ---- value: K steps, inputs resident in HBM ---------------------------------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    clocks.wait_ready()
    for w in range(args.warmup):
        step(w)
    barrier()
    clocks.mark()
    l0 = eng.launch_count()
    eng.timer_start()
    for k in range(args.steps):
        step(args.warmup + k)
    if trainer is not None:
        trainer.finalize()                          # the exchange still in flight + the hot rows back into every rank's Q
    ms = eng.timer_stop()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    launches = eng.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_tables(args.dump_outputs, *eng.get_factors())
    ms = allmax(ms)
    value = T * world * args.steps / (ms * 1e-3)
    achieved = bpt * T / (k_ms * 1e-3) / 1e9
    tkey = args.config + ("-small" if args.small else "") + ("/%d" % world if args.config == "C3" else "")
    traffic, traffic_src = ncu_traffic(tkey)

    sched = None
    if trainer is not None:
        sched = dict(hot_rows=int(len(trainer.hot_tracks)), hot_share=float(trainer.hot_share_of_events), warps=int(trainer.n_warps),
                     ctas=int(trainer.n_ctas))
        trainer.close()
        eng.set_delta_weights(None)
        trainer = None

    # ---- config C5: APR epoch (adversarial BPR, fused per-triplet perturbation), APR.conf hyper-parameters ----
    apr = None
    if not args.no_apr and d == 64:
        ams = []
        for k in range(4):
            barrier()
            eng.timer_start()
            eng.apr_epoch(0.003, 0.002, 0.01, 0.5, 2.0, SEED, 3000 + k, 0, mode, want_loss=False)
            ams.append(allmax(eng.timer_stop()))
        apr = {"metric": "apr_triplets_per_sec", "value": T * world / (min(ams[1:]) * 1e-3), "ms_per_epoch": min(ams[1:]), "n_gpus": world,
               "workload": "C5: APR d=64 on the C2 log, eps 0.5, regA 2, lr 0.003 (config/APR.conf)", "kernel": "bpr_sgd_blk_kernel<2, APR>",
               "parallelism": ("%d replicas, like the headline" % world) if world > 1 else "single GPU"}

    # ---- the SHARDED trainer (one model over N GPUs: SURVEY 8e / north_star's partitioning), measured, not the headline ----
    sharded = None
    if world > 1 and not args.no_sharded and not headline_sharded:
        upload()
        tr = make_trainer()
        sms, ams = [], []
        try:
            for k in range(2 + min(args.steps, 4)):
                barrier()
                eng.timer_start()
                tr.epoch(LR, REG_U, REG_I, SEED, 4000 + k, finalize=True)
                sms.append(allmax(eng.timer_stop()))
            for k in range(3):
                barrier()
                eng.timer_start()
                tr.epoch(0.003, 0.002, 0.01, SEED, 4100 + k, apr=(0.5, 2.0), finalize=True)
                ams.append(allmax(eng.timer_stop()))
        finally:
            sinfo = dict(hot_rows=int(len(tr.hot_tracks)), hot_share_of_positives=float(tr.hot_share_of_events), warps_per_rank=int(tr.n_warps),
                         ctas_per_rank=int(tr.n_ctas), parts_per_epoch=args.sub_epochs, asynchrony=float(tr.asynchrony),
                         # what the shared rows put on NVLink, from the schedule (a model, not a counter: ncu is one process per
                         # call here): a positive in the shared table is on another rank for (N - 1) / N of the slots, and a touch
                         # is one row loaded and one row added
                         nvlink_bytes_per_triplet_model=float(tr.hot_share_of_events) * (world - 1) / world * 2 * d * 4)
            tr.close()
            eng.set_delta_weights(None)
        sharded = {"metric": METRIC, "value": T * world / (min(sms[2:]) * 1e-3), "unit": UNIT, "ms_per_step": min(sms[2:]), "scaling": "weak",
                   "apr_value": T * world / (min(ams[1:]) * 1e-3), "apr_ms_per_epoch": min(ams[1:]),
                   "schedule": "users sharded, P rows private; the most played tracks' rows live ONCE (slot s on rank s % N) and are loaded / "
                               "added over NVLink peer memory (CUDA IPC, ld/red .sys); the tail of Q is replicated, dQ all-reduced by NCCL on a "
                               "second stream UNDER the next part and applied one part late (plain sum); the ranks "
                               "together run `asynchrony` x the warps one GPU gives the whole log", **sinfo}

    # ---- SURVEY 8f row 4: WRMF (implicit ALS, recommender/cf/WRMF.py) on the same log and tables, d = 64 ----
    wrmf = None
    if world == 1 and not args.no_wrmf and d == 64:
        eng.sync()
        t0 = time.perf_counter()
        nnz = int(len(log.uq_items))
        eng.wrmf_pair_counts()                      # one-off: play counts per pair + the track-major copy of the pairs
        prep_s = time.perf_counter() - t0
        wms = {0: [], 1: []}
        for k in range(3):
            for side in (0, 1):
                eng.sync()
                eng.timer_start()
                eng.wrmf_sweep(side, 1.0, 10.0, want_loss=False)
                wms[side].append(eng.timer_stop())
        u_ms, t_ms = min(wms[0][1:]), min(wms[1][1:])
        flops = lambda rows: nnz * d * (d + 1) + rows * (d ** 3 / 3.0 + 2 * d * d)      # rank-1 terms (lower triangle) + LDL^T + substitutions
        wrmf = {"metric": "wrmf_iterations_per_sec", "value": 1e3 / (u_ms + t_ms), "ms_user_sweep": u_ms, "ms_track_sweep": t_ms,
                "unique_pairs": nnz, "pairs_per_sec": 2 * nnz / ((u_ms + t_ms) * 1e-3), "prepare_seconds": prep_s,
                "fp64_tflops_user_sweep": flops(m) / (u_ms * 1e-3) / 1e12, "fp64_tflops_track_sweep": flops(n) / (t_ms * 1e-3) / 1e12,
                "dtype": "f64 arithmetic on f32 tables (as the reference)", "kernel": "wrmf_solve_kernel<4, 16> + wrmf_light_kernel<64> (rows with <= 16 entries) + gram, chunk",
                "workload": "WRMF d=64, reg 1, alpha 10 on the C2 log (%d users x %d tracks, %d unique pairs)" % (m, n, nnz)}
        if not args.no_cpu:                         # the reference's per-row solve (oracle port of WRMF.py:36-57), one core
            from oracle import wrmf_ref
            Pn, Qn = eng.get_factors()
            rows = np.linspace(0, m - 1, 200).astype(np.int64)
            sub_ptr = np.zeros(len(rows) + 1, np.int64)
            np.cumsum(log.uq_indptr[rows + 1] - log.uq_indptr[rows], out=sub_ptr[1:])
            sub_idx = np.concatenate([log.uq_items[log.uq_indptr[r]:log.uq_indptr[r + 1]] for r in rows])
            out_rows = np.zeros((len(rows), d), np.float32)
            t0 = time.perf_counter()
            wrmf_ref.half_sweep(out_rows, Qn, sub_ptr, sub_idx, np.ones(len(sub_idx), np.int32), 1.0, gram="f32")
            dt = time.perf_counter() - t0
            wrmf["cpu_baseline"] = {"value": len(rows) / dt, "unit": "user rows/s", "cores": 1, "kind": "port",
                                    "sample": "200 evenly spaced users of the same log, oracle port of WRMF.py:36-57 incl. one YtY",
                                    "gpu_user_rows_per_sec": m / (u_ms * 1e-3)}

    # ---- WRMF over N GPUs: rows of a half-sweep are independent, every rank solves a range and broadcasts it -- exact,
    #      bit-identical to one GPU (tests/test_multigpu.py).  ONE log (rank 0's shape) held by every rank. ----
    if world > 1 and not args.no_wrmf and d == 64 and not headline_sharded:
        wlog = synth.power_law_log_torch(wl["users"], wl["tracks"], wl["plays"], SEED, device="cuda")      # the same log on every rank
        torch.cuda.empty_cache()
        wP, wQ = synth.init_factors(wlog.m, wlog.n, d, SEED + 1000)
        eng.set_interactions(wlog.m, wlog.n, wlog.ev_indptr, wlog.ev_items, wlog.uq_indptr, wlog.uq_items)
        eng.set_factors(wP * 10, wQ * 10)
        it_indptr = eng.wrmf_pair_counts()[1]
        wt = sharding.WrmfShardedTrainer(eng, dist, dev, wlog.uq_indptr, it_indptr)
        wts = []
        for k in range(4):
            barrier()
            eng.timer_start()
            wt.iteration(1.0, want_loss=False)
            wts.append(allmax(eng.timer_stop()))
        nnz = int(len(wlog.uq_items))
        wrmf = {"metric": "wrmf_iterations_per_sec", "value": 1e3 / min(wts[1:]), "ms_per_iteration": min(wts[1:]), "n_gpus": world, "scaling": "strong",
                "unique_pairs": nnz, "pairs_per_sec": 2 * nnz / (min(wts[1:]) * 1e-3),
                "parallelism": "every rank holds the log and both tables, solves a range of rows balanced by cost (sharding.shard_rows_by_cost: entries plus the factorisation every row pays) and broadcasts it (NCCL); "
                               "no reduction: bit-identical to one GPU",
                "workload": "WRMF d=64, reg 1, alpha 10 on ONE C2 log (%d users x %d tracks, %d unique pairs)" % (wlog.m, wlog.n, nnz)}
        del wlog, wP, wQ

    # ---- e2e: the job a user of the class API runs (IterativeRecommender.buildModel): the log and the tables go up ONCE
    #      from pinned host memory, num.max.iter = E epochs each return their loss (the lr schedule needs it), the tables
    #      come back.  Also: the same with the upload repeated before EVERY epoch (round 1's definition). ----
    E = args.e2e_epochs
    h2d = log.ev_indptr.nbytes + log.ev_items.nbytes + log.uq_indptr.nbytes + log.uq_items.nbytes + pP.nbytes + pQ.nbytes
    d2h = pP.nbytes + pQ.nbytes + 8 * E

    def e2e_job(epochs, base_epoch):
        upload()
        tr = make_trainer() if headline_sharded else None
        loss = 0.0
        for ep in range(epochs):
            if tr is not None:
                loss = tr.epoch(LR, REG_U, REG_I, SEED, base_epoch + ep, want_loss=True, finalize=True)
            else:
                loss = eng.bpr_epoch(LR, REG_U, REG_I, SEED, base_epoch + ep, mode, want_loss=True)
            p2, q2 = eng.frob2()
            loss += REG_U * p2 + REG_I * q2         # BPR.py:59 (per rank: its events, its P rows)
        if tr is not None:
            tr.close()
            eng.set_delta_weights(None)
        eng.get_factors(pP.array, pQ.array)
        return loss

    def timed(fn):
        barrier()
        t0 = time.perf_counter()
        r = fn()
        eng.sync()
        return r, allmax((time.perf_counter() - t0) * 1e3)

    e2e_job(1, 1900)                                # warm: allocations, pinned staging
    loss, job_ms = timed(lambda: e2e_job(E, 2000))
    e2e_value = T * world * E / (job_ms * 1e-3)
    _, one_ms = timed(lambda: e2e_job(1, 2100))
    e2e_every = T * world / (one_ms * 1e-3)

    # ---- north_star check 4 for THIS schedule: Recall@10 / NDCG@10 against the serial-order run of the same log ----
    qual = None
    if not args.no_quality:
        spec = dict(quality.QUALITY_LOG)
        if args.small:
            spec.update(users=20_000, tracks=5_000, plays=600_000)
        qlog, qP, qQ = quality.make_log(spec)
        torch.cuda.empty_cache()
        base = [0.0, 0.0, 0.0]
        if rank == 0:
            br, bn, bdt, _ = quality.single_gpu_run(local, qlog, qP, qQ, spec, MODE_SERIAL)
            base = [br, bn, bdt]
        bt = torch.tensor(base, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.broadcast(bt, 0)
        br, bn, bdt = (float(x) for x in bt)
        run = [0.0, 0.0, 0.0, 0.0]
        if rank == 0:
            run = list(quality.single_gpu_run(local, qlog, qP, qQ, spec, mode))
        rt = torch.tensor(run, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.broadcast(rt, 0)
        qual = quality.verdict(dict(recall=float(rt[0]), ndcg=float(rt[1]), seconds=float(rt[2]), last_epoch_loss=float(rt[3]), ranks=1), br, bn)
        qlog_desc = "%d users x %d tracks, %d training events (20 %% of %d plays held out), d=%d, %d epochs, lr %.2f" % (
            qlog.m, qlog.n, qlog.train_size, spec["plays"], spec["d"], spec["epochs"], spec["lr"])
        qref = ("serial-order mode on one GPU (reproduces BPR.py:40-62 to 1e-5), same tables and sampler seed: "
                "recall@10 %.4f ndcg@10 %.4f (%.1f s)" % (br, bn, bdt))
        qual.update(log=qlog_desc, reference=qref, schedule="yue_bpr_epoch, Hogwild mode on one GPU: the schedule of `value` (every replica runs it)")
        if sharded is not None:                     # the sharded trainer on ONE log, users interleaved over the ranks
            srun = quality.shared_hot_run(local, ctl, qlog, qP, qQ, spec, args.sub_epochs, args.asynchrony or None, reduce_factory=reduce_factory,
                                          reserve_sms=args.reserve_sms)
            sq = quality.verdict(srun, br, bn)
            sq.update(log=qlog_desc + "; ONE log, users interleaved over the ranks, plain sum of the tail deltas", reference=qref)
            sharded["quality"] = sq
            sharded["quality_at_bench_size"] = ("measured with tools/quality_mgpu.py at config C2's own size (1 M users x 200 K tracks, 50 M training events, 4 epochs; "
                                                "serial order 0.0978 / 0.0791) with this trainer's defaults -- up to 248 shared rows (239 = 47 % of the positives), "
                                                "asynchrony 0.25, plain sum: 2 GPUs, 32 parts: Recall@10 -0.0012 / NDCG@10 +0.0005; 4 GPUs, 64 parts: -0.0005 / +0.0049 -- "
                                                "8 GPUs, 256 parts: -0.0014 / +0.0030 -- inside the 0.5-point gate (profiles/r2/quality_c2_n2_async.log, quality_c2_n4_hot.log, "
                                                "quality_c2_n8_hot.log); with round 2's earlier 9 shared rows -0.026 / -0.016 at any asynchrony")
        del qlog, qP, qQ

    # ---- round 1's schedule, for continuity: replicas of ALL rows, saturation-weighted sum once per epoch ----
    tmode = None
    if world > 1 and not args.no_throughput_mode:
        upload()
        cnt = torch.from_numpy(local_counts).to("cuda")
        dist.all_reduce(cnt)
        w = sharding.saturation_weights(cnt.cpu().numpy(), world, 1, 0.05 * LR)
        old = sharding.ShardedTrainer(eng, dist, dev, sub_epochs=1, row_weights=w)
        for k in range(3):
            old.epoch(LR, REG_U, REG_I, SEED, 5000 + k, mode)
        barrier()
        eng.timer_start()
        for k in range(args.steps):
            old.epoch(LR, REG_U, REG_I, SEED, 5003 + k, mode)
        tms = allmax(eng.timer_stop())
        eng.set_delta_weights(None)
        tmode = {"value": T * world * args.steps / (tms * 1e-3), "unit": UNIT, "ms_per_step": tms / args.steps,
                 "schedule": "round 1: every row of Q replicated, full concurrency on every rank, ONE saturation-weighted all-reduce of dQ per epoch",
                 "quality": "outside the gate (profiles/quality_study_r1.md section E: Recall@10 +0.02 against the serial order on 2 GPUs, "
                            "unstable without the weights on 4) -- reported as a throughput ceiling, not as a result"}

    cune = None
    if world == 1 and args.config == "C2" and not args.no_cune:
        cune = bench_cune(eng, args)
    gcn = None
    if world == 1 and args.config == "C2" and not args.no_gcn:
        gcn = bench_lightgcn(eng, args)

    # ---- config C3's shard on one GPU: Q = 1 GB does not fit in L2, the honest HBM case (N = 1 line only) ----
    c3 = None
    if world == 1 and args.config == "C2" and not args.no_c3:
        c3 = bench_c3_shard(eng, args, hbm_peak)

    out = None
    if rank == 0:
        par = "single GPU"
        if headline_sharded:
            par = ("ONE model over %d GPUs: users sharded, P rows private; the %d most played tracks' rows (%.0f %% of the positives) live once "
                   "(slot s on rank s %% %d) and are loaded / added over NVLink peer memory; the tail of Q replicated, dQ all-reduced %d times "
                   "per epoch under the next part (plain sum), %d warps on %d CTAs per rank.  QUALITY: the same schedule is inside the 0.5-point "
                   "gate of the serial order at config C2's size on 2, 4 and 8 GPUs (`sharded.quality_at_bench_size`); not measured at C3's size; "
                   "the `quality` block is the one-GPU schedule" % (world, sched["hot_rows"], 100 * sched["hot_share"], world, args.sub_epochs,
                                                                    sched["warps"], sched["ctas"]))
        elif world > 1:
            par = ("%d replicas: every GPU trains its own model on its own C2-shaped log (folds / seeds / hyper-parameter points), no "
                   "collective on the path; one SHARDED model is measured in `sharded`: inside the 0.5-point gate, but slower than one GPU "
                   "(DESIGN.md section 6)" % world)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "d": d, "triplets_per_step_per_gpu": T, "lr": LR,
                       "reg": [REG_U, REG_I], "sgd_mode": "hogwild_" + ("store" if mode == MODE_HOGWILD_STORE else "atomic_delta"),
                       "l2": "inputs exceed L2 (P %d MB + log %d MB per step; Q %d MB %s)" % (
                           pP.nbytes >> 20, (log.ev_items.nbytes + log.uq_items.nbytes) >> 20, pQ.nbytes >> 20,
                           "is L2-resident by nature" if pQ.nbytes < (100 << 20) else "exceeds L2 too"),
                       "parallelism": par},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d // E), "d2h_bytes_per_step": int(d2h // E),
                    "steps": E, "ms_per_job": job_ms, "h2d_bytes_per_job": int(h2d), "d2h_bytes_per_job": int(d2h),
                    "what": "one buildModel through the C ABI with HOST buffers, as the class API runs it (num.max.iter = %d): set_interactions + "
                            "set_factors from pinned memory ONCE, then %d x (epoch + its loss + frob2 to the host: the lr schedule reads it), "
                            "then get_factors; value = %d epochs' triplets / the job's wall time" % (E, E, E),
                    "upload_before_every_epoch": {"value": e2e_every, "ms_per_step": one_ms, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h - 8 * (E - 1)),
                                                  "what": "round 1's definition: upload + one epoch + download, every step"}},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                         "kernel": sgd_kernel_name(d), "kernel_ms": k_ms,
                         "algorithmic_bytes_per_launch": bpt * T, "algorithmic_bytes_per_triplet": bpt,
                         "l2_bytes_per_triplet": 4 * d * 4 + 12,
                         "l2_note": "what a warp-per-user kernel must move through L2 per triplet: Q[i], Q[j] read and added (4 rows) + ids; "
                                    "P[u] lives in registers over a user's events.  Q (%d MB) %s, so DRAM traffic (`traffic`) is %s" % (
                                        pQ.nbytes >> 20, "fits in L2" if pQ.nbytes < (100 << 20) else "does not fit in L2",
                                        "a small fraction of the algorithmic bytes: the bound is L2 atomics + issue, see profiles/" if pQ.nbytes < (100 << 20)
                                        else "the real bound")},
            "final_loss": loss,
        }
        if qual:
            out["quality"] = qual
        if sharded:
            out["sharded"] = sharded
        if tmode:
            out["throughput_mode"] = tmode
        if apr:
            out["apr"] = apr
        if wrmf:
            out["wrmf"] = wrmf
        if cune:
            out["cune"] = cune
        if gcn:
            out["lightgcn"] = gcn
        if c3:
            out["c3"] = c3

    # ---- secondary metric: full-catalog masked top-10 (config C4 shape, bounded user block) --
    if not args.no_rank:
        rk = bench_ranking(eng, args, bf16_peak, rank, world, dist if world > 1 else None)
        if rank == 0:
            out["ranking"] = rk

    # ---- cpu_baseline (rank 0, N = 1 only) -----------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu:
        sample = cpu_sample(log, 400_000 if not args.small else 40_000, d, SEED)
        t = cpu_epoch(sample, 0)
        out["cpu_baseline"] = {"value": sample["T"] / t, "unit": UNIT, "cores": 1, "kind": "port",
                               "host_cores": os.cpu_count(),
                               "sample": "%d-triplet user-strided sample of the same log, one epoch of the oracle "
                                         "port of BPR.py:31-62 (float32 numpy rows, serial)" % sample["T"]}
    if rank == 0:
        emit(json.dumps(out))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def bench_cune(eng, args):
    """SURVEY 8f row 4: one epoch of CUNE's two-level BPR (recommender/advanced/CUNE.py:118-178, K8) on a tenth of config C2's
    shape -- the similar-user lists CUNE derives from its DeepWalk embedding are synthetic here (two other users per user,
    none for every fifth), the per-user implicit-positive sets are built from them as CUNE.py:95-113 does."""
    from yue_b200 import synth
    from yue_b200.cune import implicit_positive_lists
    from yue_b200.engine import MODE_HOGWILD
    users, tracks, plays, d = (100_000, 20_000, 5_000_000, 64) if not args.small else (10_000, 4_000, 300_000, 64)
    log = synth.power_law_log(users, tracks, plays, SEED + 8, test_ratio=0.0)
    m = log.m
    top = {u: [f for f in ((u * 7 + 3) % m, (u * 11 + 5) % m) if f != u] for u in range(m) if u % 5}
    ip_indptr, ip_items = implicit_positive_lists(m, log.uq_indptr, log.uq_items, top)
    P, Q = synth.init_factors(log.m, log.n, d, SEED + 9)
    eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    eng.set_factors(P, Q)
    eng.cune_set_implicit(ip_indptr, ip_items)
    T = log.train_size
    ms = []
    for ep in range(3):
        eng.sync()
        eng.timer_start()
        eng.cune_epoch(0.02, 0.01, 0.01, 2.0, SEED, ep, MODE_HOGWILD)
        ms.append(eng.timer_stop())
    t = min(ms[1:])
    return {"metric": "cune_events_per_sec", "value": T / (t * 1e-3), "unit": "events/s (3 repeats each)", "ms_per_epoch": t,
            "kernel": "cune_sgd_kernel<1, kAtomic>", "warps": int(max(1, min(148 * 16, T // 16384))),
            "workload": "CUNE d=64, s=2, lr 0.02, reg 0.01: %d users x %d tracks x %d events, %d implicit positives" % (m, log.n, T, len(ip_items)),
            "note": "the number of warps is bounded by the log (one per 16 384 events, like K2: profiles/cune_r2.md); the kernel is a chain of "
                    "7 dependent dot products + sigmoids per repeat (CUNE.py:134-159 re-evaluates every sigmoid), issue-latency bound"}


def bench_lightgcn(eng, args):
    """SURVEY 8f row 4: LightGCN (recommender/advanced/LightGCN.py:27-98, K9) at config/LightGCN.conf's settings (50 factors,
    batches of 128, lr 0.002, reg 0.001, 3 layers) on config C1's shape (the reference's own scale: every step propagates
    over the WHOLE graph), and on a log ten times larger.  A pass over the batches is one cooperative launch; a step is
    2 L + 2 = 8 graph-wide phases."""
    from yue_b200 import synth
    from yue_b200.lightgcn import truncated_normal
    out = {"metric": "lightgcn_steps_per_sec", "unit": "Adam steps/s (128 triplets, 3-layer propagation forward and backward over the whole graph)",
           "kernel": "gcn_steps_kernel<16, 1>: one cooperative launch per pass"}
    for name, (users, tracks, plays, steps) in (("c1_shape", (4_000, 50_000, 100_000, 0)), ("x10", (40_000, 100_000, 1_000_000, 600))):
        if args.small and name == "x10":
            continue
        log = synth.power_law_log(users, tracks, plays, SEED + 41, test_ratio=0.2)
        ev_user = np.repeat(np.arange(log.m, dtype=np.int32), np.diff(log.ev_indptr))
        perm = np.random.default_rng(SEED + 42).permutation(len(ev_user))
        rng = np.random.default_rng(SEED + 43)
        U, V = truncated_normal((log.m, 50), 0.005, rng), truncated_normal((log.n, 50), 0.005, rng)
        eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
        eng.set_factors(U, V)
        eng.gcn_set_events(ev_user[perm], log.ev_items[perm])
        n_steps = (log.train_size + 127) // 128
        end = min(n_steps, steps) if steps else n_steps
        eng.gcn_epoch(128, 0.002, 0.001, SEED, 0, step_end=min(end, 50))          # warm-up (also builds the row lists)
        ms, losses = [], None
        for ep in range(1, 4):
            eng.sync()
            eng.timer_start()
            losses = eng.gcn_epoch(128, 0.002, 0.001, SEED, ep, step_end=end)
            ms.append(eng.timer_stop())
        t = min(ms)
        nnz = int(log.uq_indptr[-1])
        if name == "c1_shape":
            c1 = (log, ev_user, perm, U, V)
        out[name] = {"users": log.m, "tracks": log.n, "train_events": log.train_size, "graph_edges": 2 * nnz, "steps": end,
                     "ms_per_pass": t, "us_per_step": 1e3 * t / end, "steps_per_sec": end / (t * 1e-3),
                     "gathered_GBps": 5 * 2 * nnz * 52 * 4 * end / (t * 1e-3) / 1e9,
                     "first_loss": float(losses[0]), "last_loss": float(losses[-1])}
    out["value"] = out["c1_shape"]["steps_per_sec"]
    # the CPU restatement of the same step (float64 scipy CSR products + numpy Adam), on the last log built, a few steps
    from oracle import lightgcn_ref as lg
    log, ev_user, perm, U, V = c1
    A = lg.adjacency(log.m, log.n, ev_user, log.ev_items)
    E0 = np.concatenate([U, V]).astype(np.float64)
    adam, neg = lg.Adam(E0.shape), rng.integers(0, log.n, 128)
    t0, n_cpu = time.perf_counter(), 0
    while n_cpu < 3 or time.perf_counter() - t0 < 5.0:
        sl = slice(128 * n_cpu, 128 * n_cpu + 128)
        _, g = lg.loss_and_grad(A, E0, log.m, ev_user[perm][sl], log.ev_items[perm][sl], neg, 0.001)
        adam.step(E0, g, 0.002)
        n_cpu += 1
    out["cpu_baseline"] = {"value": n_cpu / (time.perf_counter() - t0), "unit": "steps/s", "cores": 1, "kind": "port",
                           "sample": "%d steps on the c1_shape log (oracle/lightgcn_ref.py: scipy CSR products in float64, numpy Adam)" % n_cpu}
    out["note"] = ("gathered_GBps = 5 dense products per step x edges x 208-byte rows (the sixth product reads only the <= 384 rows the "
                   "batch touched); at C1's shape a step is bound by its 8 grid barriers, not by bandwidth")
    return out


def bench_c3_shard(eng, args, hbm_peak):
    """One GPU's share of config C3 at 8 GPUs: 1.25 M users x 2 M tracks x 125 M plays, d = 128.  Q is 1.02 GB -- ten times
    the L2 -- so this is the case where the SGD kernel really runs against HBM (SURVEY.md section 7 "roofline honesty")."""
    import torch
    from yue_b200 import synth
    from yue_b200.engine import MODE_HOGWILD
    users, tracks, plays, d = (1_250_000, 2_000_000, 125_000_000, 128) if not args.small else (60_000, 100_000, 3_000_000, 128)
    log = synth.power_law_log_torch(users, tracks, plays, SEED + 31, device="cuda")
    torch.cuda.empty_cache()
    P, Q = synth.init_factors(log.m, log.n, d, SEED + 32)
    eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    eng.set_factors(P, Q)
    T = log.train_size
    for k in range(2):
        eng.bpr_epoch(LR, REG_U, REG_I, SEED, k, MODE_HOGWILD, want_loss=False)
    times = []
    for k in range(4):
        eng.sync()
        eng.timer_start()
        eng.bpr_epoch(LR, REG_U, REG_I, SEED, 10 + k, MODE_HOGWILD, want_loss=False)
        times.append(eng.timer_stop())
    ms = float(np.mean(times))
    bpt = bytes_per_triplet(d)
    traffic, src = ncu_traffic("C3-shard" + ("-small" if args.small else ""))
    ach = bpt * T / (ms * 1e-3) / 1e9
    out = {"metric": METRIC, "value": T / (ms * 1e-3), "unit": UNIT, "ms_per_epoch": ms, "n_gpus": 1,
           "workload": "C3 shard (1 of 8): BPR d=128, %d users x %d tracks x %d plays; Q = %d MB" % (log.m, log.n, T, Q.nbytes >> 20),
           "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "kernel": sgd_kernel_name(d),
                        "kernel_ms": ms, "algorithmic_bytes_per_triplet": bpt, "traffic": traffic, "traffic_source": src,
                        "dram_gbs": (traffic / (ms * 1e-3) / 1e9) if traffic else None,
                        "dram_frac_of_peak": (traffic / (ms * 1e-3) / 1e9 / hbm_peak) if traffic else None}}
    return out


def bench_ranking(eng, args, bf16_peak, rank=0, world=1, dist=None):
    """Masked top-10 against a 2M-track catalog (config C4), users/s: one full wave of 148 CTAs x 128
    users, then all of C4's 1 M users.  Host ids in, host ids+scores out.  With N ranks the users are
    sharded by contiguous block, Q is replicated, no collective on the data path (SURVEY.md 8e); the time
    is the max over ranks."""
    import torch
    from yue_b200 import synth
    from yue_b200.engine import RANK_AUTO, PinnedArray
    n = 2_000_000 if not args.small else 100_000
    m_total = args.rank_users
    m = m_total * (rank + 1) // world - m_total * rank // world          # this rank's block of users
    indptr, uq = synth.mask_csr_torch(m, n, 50, SEED + 4 + 100 * rank)
    P, _ = synth.init_factors(m, 1, D, SEED + 4 + 100 * rank)
    _, Q = synth.init_factors(1, n, D, SEED + 4)
    eng.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), indptr, uq)
    eng.set_factors(P, Q)
    torch.cuda.empty_cache()
    users = np.arange(m, dtype=np.int32)
    ids, sc = PinnedArray((m, 10), np.int32), PinnedArray((m, 10), np.float32)
    ids20, sc20 = PinnedArray((min(m, 18944), 20), np.int32), PinnedArray((min(m, 18944), 20), np.float32)
    eng.rank_topn(users[:256], 10, RANK_AUTO, ids.array[:256], sc.array[:256])
    out = {"metric": "topn_ranked_users_per_sec", "unit": "users/s",
           "includes": "H2D of user ids, gather of P rows, tcgen05 candidate pass + exact re-score, D2H of ids+scores"}
    for key, B, N, reps in (("one_wave", min(m, 18944), 10, 3), ("one_wave_top20", min(m, 18944), 20, 3), ("c4_full", m, 10, 2)):
        oi, osc = (ids20.array, sc20.array) if N == 20 else (ids.array, sc.array)
        times = []
        for _ in range(reps):
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            eng.rank_topn(users[:B], N, RANK_AUTO, oi[:B], osc[:B])
            dt = time.perf_counter() - t0
            if dist is not None:                       # max over ranks
                tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
            times.append(dt)
        t = min(times)
        Ball = B * world if key != "c4_full" else m_total
        flops = 2.0 * Ball * n * D
        out[key] = {"users": Ball, "tracks": n, "topN": N, "seconds": t, "users_per_sec": Ball / t, "dense_tflops": flops / t / 1e12,
                    "frac_of_bf16_peak": flops / t / 1e12 / (bf16_peak * world), "fallback_and_spilled_rows_rank0": list(eng.rank_stats())}
    # K6: the metrics of those lists against a synthetic held-out set (5 tracks per user), on the device
    te_indptr, te_items = synth.mask_csr_torch(m, n, 5, SEED + 5)
    eng.set_test_set(te_indptr, te_items)
    t0 = time.perf_counter()
    sums, distinct = eng.rank_metrics([5, 10])
    out["metrics_seconds"] = time.perf_counter() - t0
    # the reference's per-user body of evalRanking (predict + mask + the shipped selection, IterativeRecommender.py:93-145)
    # as restated by the oracle, on one host core, for a few users of the same problem -- reported beside, not a target
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            from oracle import topn
            hp, hu = np.asarray(indptr), np.asarray(uq)
            nu = 20 if not args.small else 50
            t0 = time.perf_counter()
            for u in range(nu):
                topn.topn_ref_quirk(Q.dot(P[u]), hu[hp[u]:hp[u + 1]], 10)
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": nu / dt, "unit": "users/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
                                   "sample": "%d users of the same problem: Q.dot(P[u]) + mask + the reference's selection "
                                             "(oracle port of IterativeRecommender.py:93-145), serial" % nu}
        except Exception as exc:                      # a reported baseline must not cost the bench line
            out["cpu_baseline"] = {"error": repr(exc)}
    out["value"] = out["c4_full"]["users_per_sec"]
    out["workload"] = "C4: top-10 of %d users x %d tracks, d=64, ~50 masked tracks/user, %d GPU(s), users sharded by block" % (m_total, n, world)
    return out


_REAL_STDOUT = None


def quiet_stdout():
    """Native libraries write to fd 1 (NCCL prints its version there): keep stdout for the one JSON line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(line, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--small", action="store_true", help="debug-size workload (not a bench number)")
    ap.add_argument("--sgd-mode", default="atomic", choices=["atomic", "store"])
    ap.add_argument("--config", default="C2", choices=["C2", "C3"], help="BASELINE.json configs[1] (default) or configs[2]")
    ap.add_argument("--sub-epochs", type=int, default=0, help="multi-GPU: parts per epoch = exchanges of the tail of Q (0 = sharding.default_sub_epochs: 32 up to 2 GPUs, 4 N^2 above)")
    ap.add_argument("--asynchrony", type=float, default=0.0,
                    help="multi-GPU: the ranks together run this many times the warps one GPU gives the whole log (0 = sharding.default_asynchrony: 0.25)")
    ap.add_argument("--reserve-sms", type=int, default=8, help="multi-GPU: SMs the epoch kernel leaves to the NCCL kernels")
    ap.add_argument("--e2e-epochs", type=int, default=4, help="num.max.iter of the e2e job")
    ap.add_argument("--no-quality", action="store_true")
    ap.add_argument("--no-throughput-mode", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-c3", action="store_true")
    ap.add_argument("--no-cune", action="store_true")
    ap.add_argument("--no-gcn", action="store_true")
    ap.add_argument("--no-rank", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-apr", action="store_true")
    ap.add_argument("--no-wrmf", action="store_true")
    ap.add_argument("--rank-users", type=int, default=1_000_000)   # config C4: 1 M users
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the factor tables they left (rank 0's) to DIR as float32 .npy (see dump_tables)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and not args.small:
        args.warmup = 3
    quiet_stdout()
    if args.sub_epochs <= 0:
        from yue_b200.sharding import default_sub_epochs
        args.sub_epochs = default_sub_epochs(int(os.environ.get("WORLD_SIZE", args.gpus)))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
