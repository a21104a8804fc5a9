"""bench.py — DSA inputs prioritized / second on B200 (BASELINE.json metric), driver contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c1|c2|c3|c4|c5s]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic test traces.

Headline (`value`, `e2e`, `roofline`, `cpu_baseline`): C2, the configuration the metric is quoted on —
DSA, 10 000 test x 60 000 train x 128-d float32 Gaussian-cluster traces, 10 classes (SURVEY.md 8d,
seed 2).  With N GPUs the test batch grows to 10 000 x N ("scaling": "weak") and the default layout
is N_test sharding (every rank scores its own 10 000 inputs against a replicated 30.7 MB train set,
no data-path collective) — at C2's size the train set is too small for N_train sharding to pay
(`--shard train` measures it anyway).

Every line also carries (so that the driver records them, not only the builder):
  `n_train_sharded`  north_star's multi-GPU design on a C5-shaped slice: DSA, 10 000 test x 1.28 M
      train x 2048-d, 1000 classes, bf16-representable traces generated on the device by a counter
      RNG (oracle/synth_traces.py), N_train sharded over the N ranks (strong scaling: fixed problem),
      one exchange of packed (distance, index) keys per stage; ms per pass, inputs/s, fraction of
      N x the measured tensor peak, time of one exchange, and `parity_ok`: sampled inputs checked bit
      for bit against the CPU oracle on a host copy of the traces;
  `parity_ok` (N > 1)  C2 through the N_train-sharded DSA class vs the NumPy oracle, bit for bit;
  `other_configs` (N = 1)  C1 DeepGini, C3 LSA (+ per-class LSA, `device_call_graph_ms` = the CUDA-graph replay of a
      whole scoring call's device work), C4 KMNC, CAM: device ms, e2e, roofline and cpu_baseline each (also selectable
      alone with --workload);
  `fit_time_table` (N = 1)  the opt-in extension DSA.fit_other_class_table() — not what `value` measures;
  `stall_retries`  how many timed measurements were repeated because one step contained a host stall (Timer.timed).

`value` times the device-resident path (test traces already in HBM, result left in HBM); `e2e` times
the reference-facing call `DSA.__call__(numpy, numpy) -> numpy` from pinned host memory, host<->device
copies inside the timed region; `e2e_pageable` the same call from ordinary (pageable) NumPy memory —
what the reference's callers hold (handler_model.py:191).  Steps are timed individually with CUDA
events on the launching stream, L2 is flushed (256 MiB write) between steps, the sum over K steps is
max-reduced over ranks.  `--impl reference` times the reference's own NumPy algorithm (oracle port:
same NumPy expressions, same 5-thread badge pool, surprise.py:599) on the host.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

C2 = dict(n_train=60000, n_test=10000, d=128, classes=10, seed=2)
C5S = dict(n_train=1280000, n_test=10000, d=2048, classes=1000, seed=5)
METRIC = "dsa_inputs_prioritized_per_sec"


def c2_workload(n_test: int) -> str:
    return f"C2: DSA {n_test} test x 60000 train x 128-d float32, 10 classes (seed 2)"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


def _sustained_tflops():
    """cuBLAS bf16 under the power cap for seconds (the denominator for a kernel timed inside a long step)"""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        if "bf16_tflops_sustained" in p:
            return float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, "fallback (B200_PROFILING.md, sustained)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark(self):
        """the timed region starts now (nvidia-smi takes a few hundred ms to deliver its first row, so the sampler is
        started before the warm-up and only rows from here on count)"""
        self.t_mark = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        t0 = getattr(self, "t_mark", 0.0) - 0.1          # a row is up to one 100 ms period old when it is read
        inside = [r for t, r in self.rows if t >= t0]
        rows = inside if inside else [r for _, r in self.rows][-3:]
        sm = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 8 for i in range(4) if r[4 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "samples_inside_timed_region": len(inside)}


def pin_to_gpu_numa_node(gpu_index: int):
    """CPU affinity of this rank = the cores of its GPU's NUMA node, so that pinned staging buffers and
    the launching thread sit next to the GPU (SCALE's e2e swung 0.37-0.70 ms without it)."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        pass
    return None


# ----------------------------------------------------------------------------------------------
# reference arm / CPU baseline (the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------
def _ref_sample(xtr, ytr, xte, pte, n_inputs: int, threads: int = 5):
    from oracle import np_oracle

    t0 = time.perf_counter()
    np_oracle.dsa_oracle(xtr, ytr, xte[:n_inputs], pte[:n_inputs], badge_size=10, threads=threads)
    return time.perf_counter() - t0


def cpu_baseline(xtr, ytr, xte, pte, budget_inputs: int = 160):
    """Oracle port of the reference DSA (same NumPy expressions, 5 badge threads) on a bounded
    prefix of the same test set; cost is linear in the number of inputs (independent badges)."""
    from oracle import c_oracle

    dt = _ref_sample(xtr, ytr, xte, pte, budget_inputs)
    out = {"value": budget_inputs / dt, "unit": "inputs/s", "cores": 5, "kind": "port",
           "sample": f"first {budget_inputs} of the {xte.shape[0]} test inputs vs all {xtr.shape[0]} train rows, "
                     f"{dt:.1f} s; 5 badge threads as surprise.py:599; host has {os.cpu_count()} cpus"}
    try:  # stronger, non-reference CPU number for context: C/OpenMP port on all cores
        c_oracle.build()
        n_c = min(xte.shape[0], 2000)
        t0 = time.perf_counter()
        c_oracle.dsa(xtr, ytr, xte[:n_c], pte[:n_c])
        dc = time.perf_counter() - t0
        out["c_port_all_cores"] = {"value": n_c / dc, "cores": c_oracle.max_threads(),
                                   "sample": f"{n_c} inputs, {dc:.1f} s, OpenMP brute force in NumPy's summation order"}
    except Exception as e:  # pragma: no cover
        out["c_port_all_cores"] = {"error": str(e)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import np_oracle

    world = int(os.environ.get("WORLD_SIZE", "1"))
    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(**C2)
    per_step = 48                                   # bounded sample of the workload per step (~3-4 s)
    for _ in range(args.warmup):
        _ref_sample(xtr, ytr, xte, pte, per_step)
    t = [_ref_sample(xtr, ytr, xte, pte, per_step) for _ in range(args.steps)]
    total = float(np.sum(t))
    value = per_step * args.steps / total
    line = {"metric": METRIC, "value": value, "unit": "inputs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": c2_workload(C2["n_test"] * world)},
            "sample_inputs_per_step": per_step,
            "sample": f"bounded sample: {per_step} test inputs per step vs all 60000 train rows (cost is linear in the "
                      "number of inputs: independent badges of 10)",
            "cpu_baseline": {"value": value, "unit": "inputs/s", "cores": 5, "kind": "port",
                             "sample": f"{per_step} inputs per step; oracle port of surprise.py:558-651 (NumPy, "
                                       f"5 badge threads); host has {os.cpu_count()} cpus"},
            "e2e": {"value": value, "unit": "inputs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# shared timing helpers (our arm)
# ----------------------------------------------------------------------------------------------
class Timer:
    def __init__(self, dev, dist=None):
        import torch

        self.torch, self.dist = torch, dist
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, sync_ranks=True, flush=True):
        """per-step CUDA-event times (ms), L2 flushed before every step (flush=False: the caller's steps stream more
        than the L2 holds and alternate their buffers).  The events bracket host-issued launches, so a host stall
        between two launches (seen on the shared boxes: one step of ~80 ms among steps of 0.3 ms, e.g. while nvidia-smi
        holds the driver) lands in the step's time: a measurement with such an outlier (max > 8 x median) is repeated
        ONCE as a whole — still exactly `steps` steps — and the repeat is counted in `stall_retries`."""
        out = self._timed_once(fn, steps, sync_ranks, flush)
        if steps >= 5 and self.dist is None:
            med = sorted(out)[len(out) // 2]
            if med > 0 and max(out) > 8.0 * med:
                self.stall_retries += 1
                again = self._timed_once(fn, steps, sync_ranks, flush)
                if sum(again) < sum(out):
                    out = again
        return out

    stall_retries = 0

    def _timed_once(self, fn, steps, sync_ranks=True, flush=True):
        torch = self.torch
        out = []
        for _ in range(steps):
            if flush:
                self.flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if self.dist is not None and sync_ranks:
                self.dist.barrier()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            out.append(a.elapsed_time(b))
        return out

    def max_over_ranks(self, values, dev):
        torch = self.torch
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]


# ----------------------------------------------------------------------------------------------
# north_star multi-GPU design on a C5-shaped slice (every --gpus N, N = 1 included)
# ----------------------------------------------------------------------------------------------
def run_c5_slice(args, tm: Timer, dev, rank, world, comm, steps: int, cfg=None):
    """DSA, 10k test x 1.28M train x 2048-d, 1000 classes; N_train sharded over `world` ranks."""
    import torch

    from oracle import c_oracle, synth_traces as ST   # trace generator + parity checker only
    from simple_tip_b200 import engine as E

    cfg = dict(C5S if cfg is None else cfg)
    if os.environ.get("B200TIP_C5S_TRAIN"):          # profiling aid: one rank's share of the slice on one GPU
        cfg["n_train"] = int(os.environ["B200TIP_C5S_TRAIN"])
    n_train, n_test, d, classes, seed = cfg["n_train"], cfg["n_test"], cfg["d"], cfg["classes"], cfg["seed"]
    tflops_peak, _, peak_src = _peaks()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    # the whole training set in ORIGINAL order on every rank (replica: winners are gathered from it by index);
    # row i has class i % classes, so rank r's shard = rows whose rank within the class is r mod world
    full = torch.empty((n_train, d), dtype=torch.float32, device=dev)
    ST.fill(full, 0, d, classes, seed, 0)
    per_class = n_train // classes
    assert per_class * classes == n_train and per_class % world == 0
    mine = per_class // world
    cls = torch.arange(classes, device=dev).repeat_interleave(mine)
    k = torch.arange(mine, device=dev).repeat(classes)
    gid = (cls + classes * (rank + world * k)).to(torch.int64)         # class-major, ascending original index inside a class
    t_sorted = full.index_select(0, gid)
    class_off = np.arange(classes + 1, dtype=np.int64) * mine
    eng = E.NnEngine(t_sorted, class_off, gid.to(torch.int32))
    if world > 1:
        eng.t_full = full
    else:
        del full
    # test inputs: generated on the device too, identical on every rank; class-sorted for the device-resident path
    rows = torch.arange(n_test, dtype=torch.int64, device=dev)
    x = torch.empty((n_test, d), dtype=torch.float32, device=dev)
    ST.fill(x, 0, d, classes, seed, 1)
    yte = (rows % classes)
    order = torch.argsort(yte, stable=True)
    x_sorted = x.index_select(0, order).contiguous()
    q_off = np.concatenate([[0], np.cumsum(np.bincount(yte.cpu().numpy(), minlength=classes))]).astype(np.int64)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    tm.barrier()
    plan = E.dsa_plan(eng, n_test, q_off, torch.float32, True, comm if world > 1 else None)
    plan.load_sorted(x_sorted)
    for _ in range(3):
        plan.run()
    tm.barrier()
    t = tm.timed(plan.run, steps)
    (tot_ms,) = tm.max_over_ranks([sum(t)], dev)
    ms = tot_ms / steps
    out_dev = plan.out.clone()
    # one exchange in isolation (push + wait + reduce of n_test records), for "time spent in collectives"
    exch_ms, exch_kind = None, "none (1 GPU)"
    if world > 1:
        p2p = comm.p2p(dev, n_test)
        probe = torch.rand(n_test, device=dev)
        sink = torch.empty_like(probe)
        if p2p is not None:
            def one_exchange():
                p2p.push_nn(probe, None)
                p2p.min_into(sink)
            exch_kind = "peer-memory stores + flag wait fused into the consumer kernel (csrc/shard.cu)"
        else:
            def one_exchange():
                comm.reduce_min_nan(probe)
            exch_kind = "torch.distributed MIN all-reduce (NCCL)"
        for _ in range(3):
            one_exchange()
        tm.barrier()
        te = tm.timed(one_exchange, 10)
        (exch_tot,) = tm.max_over_ranks([sum(te)], dev)
        exch_ms = exch_tot / 10
    # parity: sampled inputs against the CPU oracle (brute force in NumPy's summation order) on a HOST
    # copy of the traces; and the device-side RNG against the same generator run on the host
    parity = {"checked_inputs": 0}
    if rank == 0:
        n_chk = int(args.parity_inputs)
        sel = np.sort(np.random.default_rng(7).choice(n_test, n_chk, replace=False))
        sel_t = torch.from_numpy(sel).to(dev)
        pos_in_sorted = torch.empty(n_test, dtype=torch.int64, device=dev)
        pos_in_sorted[order] = torch.arange(n_test, device=dev)
        got = out_dev[:, pos_in_sorted[sel_t]].cpu().numpy()
        host_train = (eng.t_full if world > 1 else None)
        if host_train is None:      # 1 GPU: un-sort the engine's class-major copy
            host_train = torch.empty((n_train, d), dtype=torch.float32, device=dev)
            host_train[gid] = eng.t
        t0 = time.perf_counter()
        train_np = host_train.cpu().numpy()
        labels_np = (np.arange(n_train) % classes).astype(np.int64)
        host_rows = ST.traces(torch.from_numpy(sel), d, classes, seed, 1).numpy()          # host-side regeneration
        rng_ok = bool(np.array_equal(host_rows, x[sel_t].cpu().numpy()))
        tr_rows = np.random.default_rng(8).choice(n_train, 64, replace=False)
        rng_ok = rng_ok and bool(np.array_equal(ST.traces(torch.from_numpy(tr_rows), d, classes, seed, 0).numpy(),
                                                train_np[tr_rows]))
        want = c_oracle.dsa(train_np, labels_np, host_rows, (sel % classes).astype(np.int64))
        ok = bool(np.array_equal(got[0].astype(np.float32), want["dist_a"]) and
                  np.array_equal(got[1].astype(np.float32), want["dist_b"]) and
                  np.array_equal(got[2].astype(np.int64), want["idx_a"]) and
                  np.array_equal(got[3], want["dsa"]))
        parity = {"checked_inputs": n_chk, "parity_ok": ok, "device_rng_equals_host_rng": rng_ok,
                  "oracle": "oracle/tip_oracle.c brute force (NumPy summation order, validated against the reference's "
                            "golden vectors in tests/test_oracle_golden.py)", "oracle_s": time.perf_counter() - t0}
        del train_np
    flops = 2.0 * d * n_test * n_train
    stats = eng.stats.cpu().numpy().tolist()
    if plan.speculative:         # the replayed graph has no exhaustive-scan launches: its overflow counter must be 0
        stats[0] = int(plan.overflow.item())
        assert stats[0] == 0, "a candidate list overflowed: the timed graph did not produce the result"
    cand = {}
    for mode, (cnt, _) in eng.last_cand_cnt_by_mode.items():
        c = cnt.float()
        cand["same_class" if mode == 0 else "other_classes"] = {"mean_chunks": float(c.mean()), "max_chunks": float(c.max())}
    block = {"workload": f"C5 slice: DSA {n_test} test x {n_train} train x {d}-d, {classes} classes, bf16-representable "
                         f"traces from a device-side counter RNG (seed {seed})",
             "layout": (f"N_train sharded over {world} GPUs ({n_train // world} rows per rank, every class dealt round-robin), "
                        "test inputs and raw training set replicated" if world > 1 else "1 GPU (no exchange)"),
             "scaling": "strong", "n_gpus": world, "steps": steps, "ms_per_pass": ms, "inputs_per_s": n_test / (ms * 1e-3),
             "algorithmic_tflops_aggregate": flops / (ms * 1e-3) / 1e12,
             # passes of tens of ms run back to back sit in the power-capped regime (ncu: tensor pipe 82 % active at
             # 1.45 GHz): the sustained cuBLAS figure is the matching denominator; the burst one is reported beside it
             "frac_of_n_x_tensor_peak": flops / (ms * 1e-3) / 1e12 / (_sustained_tflops()[0] * world),
             "peak_source": _sustained_tflops()[1],
             "frac_of_n_x_burst_peak": flops / (ms * 1e-3) / 1e12 / (tflops_peak * world), "burst_peak_source": peak_src,
             "exchange": exch_kind, "exchanges_per_pass": 0 if world == 1 else 2, "ms_per_exchange": exch_ms,
             "exchange_share_of_pass": None if exch_ms is None else 2 * exch_ms / ms,
             "torch_distributed_collectives_on_data_path": None if comm is None else comm.collectives,
             "generate_s": gen_s, "exhaustive_fallback_rows": stats[0], "candidates": cand}
    block.update(parity)
    # free the 10+ GB before the caller goes on
    del plan, eng, t_sorted, x, x_sorted
    torch.cuda.empty_cache()
    return block


# ----------------------------------------------------------------------------------------------
# our arm: C2 headline
# ----------------------------------------------------------------------------------------------
def step_outputs(out, plan, order, x_sorted, x_raw):
    """What one C2 device step computed, as a DSA caller receives it: float64 arrays with one entry per test input,
    in the order of the test inputs.  `out` is the step's result: the plan's [4, n] buffer, whose column r belongs to
    row r of the plan's landing buffer (class-sorted after load_sorted, the caller's rows after a DSA call), or, for
    an eager step, dist_a / dist_b of the class-sorted rows."""
    import torch

    if plan is None:
        named, rows = {"dsa": out}, order
    else:
        named = dict(zip(("dist_a", "dist_b", "winner_index", "dsa"), out))
        if torch.equal(plan.x_in, x_sorted):
            rows = order
        else:
            assert torch.equal(plan.x_in, x_raw), "the plan's landing buffer holds neither row order of the test inputs"
            rows = np.arange(order.size)
    res = {}
    for name, v in named.items():
        res[name] = np.empty(order.size)
        res[name][rows] = v.double().cpu().numpy()
    return res


def run_ours(args):
    import torch

    from oracle import np_oracle   # synthetic trace generator + cpu_baseline / parity only
    from simple_tip_b200 import _lib
    from simple_tip_b200 import engine as E
    from simple_tip_b200.core.surprise import DSA

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # the contract is ONE JSON line on stdout: anything libraries print there (NCCL's banner and its
    # NCCL_DEBUG=INFO lines) goes to stderr until the line is ready
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    affinity = pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None          # process group (timing barrier / max over ranks in every multi-GPU mode)
    comm = None
    # How the global batch of 10000 x N test inputs is spread over N GPUs:
    #   test  — every rank scores its own 10000 inputs against a replicated train set (30.7 MB at C2):
    #           independent units, no data-path collective;
    #   train — the train set is split 1/N per rank, every rank sees all 10000 x N inputs and the
    #           per-shard winners are exchanged (the layout C5 needs; measured in `n_train_sharded`).
    shard = args.shard if args.shard != "auto" else "test"
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
        comm = E.TrainShardComm()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    tm = Timer(dev, dist)

    cfg = dict(C2)
    cfg["n_test"] = C2["n_test"] * world           # weak scaling: 10000 test inputs per GPU
    xtr, ytr, xte_all, pte_all, _ = np_oracle.synth_clusters(**cfg)
    n_global = xte_all.shape[0]
    xte, pte = xte_all, pte_all
    if world > 1 and shard == "test":
        sl = slice(rank * C2["n_test"], (rank + 1) * C2["n_test"])
        xte, pte = np.ascontiguousarray(xte_all[sl]), np.ascontiguousarray(pte_all[sl])
    main_comm = comm if (world > 1 and shard == "train") else None
    sa = DSA(xtr, ytr, comm=main_comm)
    eng = sa._engine
    n_test = xte.shape[0]

    # first call through the public API: host planning + eager launches (plans are captured on the second
    # sighting of a batch shape)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sa(xte, pte)
    first_call_ms = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    sa(xte, pte)
    second_call_ms = 1e3 * (time.perf_counter() - t0)

    # device-resident inputs (value) and pinned / pageable host inputs (e2e)
    order, q_off = E.class_layout(pte, int(sa.num_classes))
    x_sorted = E.to_device(xte, dev).index_select(0, torch.from_numpy(order).to(dev))
    q_class = torch.from_numpy(pte[order].astype(np.int32)).to(dev)
    xte_pinned = torch.from_numpy(xte).pin_memory()
    xte_host = xte_pinned.numpy()
    xte_pageable = np.array(xte, copy=True)

    plan = None
    if sa.use_graphs:
        # steady-state path of DSA.__call__: the search replayed as CUDA graph(s)
        plan = E.dsa_plan(eng, n_test, q_off, x_sorted.dtype, sa.use_filter, main_comm)
        plan.load_sorted(x_sorted)

    def step_eager():
        a, b, _ = E.dsa_distances(eng, x_sorted, q_class, q_off, main_comm)
        return a / b

    last = {}

    def step_device():
        # keeps the step's result referenced: --dump-outputs reads what the last timed step computed
        last["out"] = step_eager() if plan is None else plan.run()

    def step_e2e():
        return sa(xte_host, pte)

    def step_e2e_pageable():
        return sa(xte_pageable, pte)

    xte_dev = E.to_device(xte, dev)

    def step_api_device():      # same public call with the traces already in HBM (torch CUDA tensor in)
        return sa(xte_dev, pte)

    def timed_profile(fn, steps):
        E.PROFILE = []
        t = tm.timed(fn, steps)
        prof, E.PROFILE = E.PROFILE, None
        return t, prof

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step_device()
        step_e2e()
        step_e2e_pageable()
        step_eager()
    tm.barrier()
    sampler.mark()
    t_dev = tm.timed(step_device, args.steps)
    if plan is not None and plan.speculative:
        # the replayed graph carries no exhaustive-scan launches; it is only valid if no candidate list overflowed
        assert int(plan.overflow.item()) == 0, "a candidate list overflowed: the timed graph did not produce the result"
    dumped = step_outputs(last["out"], plan, order, x_sorted, xte_dev) if (args.dump_outputs and rank == 0) else None
    t_e2e = tm.timed(step_e2e, args.steps)
    t_page = tm.timed(step_e2e_pageable, args.steps)
    step_api_device()
    t_api = tm.timed(step_api_device, args.steps)
    # per-kernel durations (roofline) and the launch census come from the same kernels launched
    # eagerly with CUDA events around the tensor-core launches; graph replays launch the same set
    launches0 = _lib.launch_count()
    _, prof = timed_profile(step_eager, args.steps)
    launches = (_lib.launch_count() - launches0) // max(1, args.steps)
    if plan is not None and plan.speculative:
        launches -= 2     # the replayed graph (what `value` times) carries no exhaustive-scan launches; the eager pass does
    tm.barrier()
    clocks = sampler.stop() if rank == 0 else None
    tot_dev_ms, tot_e2e_ms, tot_page_ms = tm.max_over_ranks([sum(t_dev), sum(t_e2e), sum(t_page)], dev)

    # ---- extension: dist_b tabulated per train row at fit time (not the headline: the per-call work changes) -------
    table = None
    if world == 1 and not args.no_others:
        want = [sa(xte_host, pte).copy(), sa.last_dist_a.copy(), sa.last_dist_b.copy(), sa.last_winner_index.copy()]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sa.fit_other_class_table()
        fit_ms = 1e3 * (time.perf_counter() - t0)
        sa(xte_host, pte)
        got = [sa(xte_host, pte).copy(), sa.last_dist_a.copy(), sa.last_dist_b.copy(), sa.last_winner_index.copy()]
        plan_t = E.dsa_plan(eng, n_test, q_off, x_sorted.dtype, sa.use_filter, None)
        plan_t.load_sorted(x_sorted)
        for _ in range(3):
            plan_t.run()
            sa(xte_host, pte)
        t_tab = tm.timed(plan_t.run, args.steps)
        t_tab_e2e = tm.timed(step_e2e, args.steps)
        table = {"what": "DSA.fit_other_class_table(): dist_b depends on the test input only through the train row that won "
                         "stage 1, so it is tabulated per train row once per training set (N_train x N_train pairs at fit "
                         "time) and a call runs stage 1 + a lookup; opt-in extension, not what `value` measures",
                 "fit_ms": fit_ms, "ms_per_step": sum(t_tab) / args.steps, "inputs_per_s": n_test * args.steps / (sum(t_tab) * 1e-3),
                 "e2e_ms_per_step": sum(t_tab_e2e) / args.steps,
                 "bit_identical_to_two_stage_call": bool(all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, want)))}
        del plan_t
        sa.drop_other_class_table()

    # ---- N > 1: the N_train-sharded DSA class against the NumPy oracle, bit for bit -----------------------
    parity = None
    if world > 1:
        n_p = 600
        sa_sh = sa if main_comm is not None else DSA(xtr, ytr, comm=comm)
        got = sa_sh(xte_all[:n_p], pte_all[:n_p])
        got2 = sa_sh(xte_all[:n_p], pte_all[:n_p])        # second call: the captured plan
        ok = None
        if rank == 0:
            want = np_oracle.dsa_oracle(xtr, ytr, xte_all[:n_p], pte_all[:n_p], threads=8)
            ok = bool(np.array_equal(got, want["dsa"]) and np.array_equal(got2, want["dsa"]) and
                      np.array_equal(sa_sh.last_winner_index, want["idx_a"]) and
                      np.array_equal(sa_sh.last_dist_a, want["dist_a"]) and np.array_equal(sa_sh.last_dist_b, want["dist_b"]))
        flag = torch.tensor([1 if (ok or ok is None) else 0], device=dev)
        same = torch.from_numpy(got).to(dev)
        ref = same.clone()
        dist.broadcast(ref, 0)
        flag &= torch.tensor([1 if torch.equal(torch.nan_to_num(ref, nan=-1.0), torch.nan_to_num(same, nan=-1.0)) else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = {"parity_ok": bool(flag.item()), "what": f"DSA(comm=N_train sharded over {world} ranks) on the first {n_p} C2 test "
                  "inputs == np_oracle.dsa_oracle (scores, dist_a, dist_b, winner index), identical on every rank",
                  "exchange": "peer-memory" if comm._p2p is not None else f"torch.distributed ({comm._p2p_failed or 'forced'})"}
        if sa_sh is not sa:
            del sa_sh

    # ---- north_star layout on the C5-shaped slice (all ranks) ---------------------------------------------
    c5 = None
    launch_mode = "CUDA-graph replay of the search" if plan is not None else "eager launches"
    if parity is not None and rank == 0:
        print("[bench] parity:", json.dumps(parity), file=sys.stderr, flush=True)
    if not args.no_c5:
        plan = None
        sa._engine._plans.clear()
        torch.cuda.empty_cache()
        try:
            c5 = run_c5_slice(args, tm, dev, rank, world, comm, steps=args.steps)
        except Exception as e:   # pragma: no cover - keep the headline line even if the big slice fails
            import traceback

            c5 = {"error": f"{type(e).__name__}: {e}", "traceback": traceback.format_exc()[-1500:]}
        if rank == 0:
            print("[bench] n_train_sharded:", json.dumps(c5), file=sys.stderr, flush=True)

    others = None
    if rank == 0 and world == 1 and not args.no_others:
        others = {}
        for wl in ("c1", "c3", "c4", "cam"):
            try:
                others[wl] = secondary(wl, args, tm, dev, steps=args.steps, with_cpu=not args.no_cpu)
            except Exception as e:   # pragma: no cover
                others[wl] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        value = n_global * args.steps / (tot_dev_ms * 1e-3)
        e2e = n_global * args.steps / (tot_e2e_ms * 1e-3)
        tflops_peak, hbm_peak, peak_src = _peaks()
        # dominant kernel: the stage-2 tcgen05 filter launch (other-class columns)
        roof = None
        if prof:
            by = {}
            for name, flops, ev0, ev1 in prof:
                by.setdefault(name, []).append((flops, ev0.elapsed_time(ev1)))
            name = max(by, key=lambda k: np.mean([t for _, t in by[k]]))
            flops = float(np.mean([f for f, _ in by[name]]))
            ms = float(np.mean([t for _, t in by[name]]))
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get(name)
            step_flops = float(sum(np.mean([f for f, _ in v]) for v in by.values()))
            roof = {"kernel": name, "bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": tflops_peak,
                    "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / tflops_peak, "traffic": traffic,
                    "peak_source": peak_src, "ms_per_launch": ms,
                    "algorithmic_flops_per_launch": flops,
                    "other_launches_ms": {k: float(np.mean([t for _, t in v])) for k, v in by.items() if k != name},
                    "whole_step": {"algorithmic_flops": step_flops, "ms": tot_dev_ms / args.steps,
                                   "frac": step_flops / (tot_dev_ms / args.steps * 1e-3) / 1e12 / tflops_peak}}
        n_ranks_copy = world if main_comm is None else 1
        line = {"metric": METRIC, "value": value, "unit": "inputs/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": tot_dev_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": c2_workload(n_global),
                           "parallelism": (f"N_train sharded over {world} GPU(s), every rank scores all 10000 x {world} "
                                           "inputs; per-shard winners exchanged once per stage" if main_comm is not None else
                                           f"N_test sharded over {world} GPU(s): 10000 inputs per GPU, train set "
                                           "replicated (30.7 MB), no data-path collective; the N_train-sharded design is "
                                           "measured in n_train_sharded" if world > 1 else "1 GPU"),
                           "filter": "bf16 tcgen05 candidate filter + exact fp32 re-rank (bit-identical to NumPy)",
                           "l2": "flushed between steps (256 MiB write)", "timing": "per-step CUDA events, summed",
                           "launch": launch_mode,
                           "cpu_affinity": affinity},
                "e2e": {"value": e2e, "unit": "inputs/s", "ms_per_step": tot_e2e_ms / args.steps,
                        "ms_per_step_median_rank0": float(np.median(t_e2e)), "ms_per_step_max_rank0": float(np.max(t_e2e)),
                        "source": "pinned host memory (caller-pinned NumPy array)",
                        "h2d_bytes_per_step": int((xte.nbytes + pte.shape[0] * 4) * n_ranks_copy),
                        # dist_a, dist_b, winner index, dsa as float64, summed over the ranks
                        "d2h_bytes_per_step": int(4 * n_test * 8 * n_ranks_copy)},
                "e2e_pageable": {"value": n_global * args.steps / (tot_page_ms * 1e-3), "unit": "inputs/s",
                                 "ms_per_step": tot_page_ms / args.steps,
                                 "source": "ordinary (pageable) NumPy arrays, as the reference's callers hold them "
                                           "(handler_model.py:191)"},
                "stall_retries": tm.stall_retries,
                "first_call_ms": first_call_ms, "second_call_ms": second_call_ms,
                "first_call_note": "first call of a batch shape = host planning + eager launches; the second captures the "
                                   "CUDA-graph plan, later calls replay it (wall clock, rank 0)",
                # the public call with device-resident traces (rank 0's own time, not max-reduced)
                "api_device_inputs": {"ms_per_step": float(np.mean(t_api)), "unit": "ms",
                                      "note": "DSA.__call__(torch CUDA tensor, labels) -> numpy scores"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof}
        if parity is not None:
            line.update({"parity_ok": parity["parity_ok"], "parity": parity})
        if c5 is not None:
            line["n_train_sharded"] = c5
        if table is not None:
            line["fit_time_table"] = table
        if others is not None:
            line["other_configs"] = others
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(xtr, ytr, xte, pte)
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, v in dumped.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), v)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if dist is not None:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
# secondary workloads (single GPU): same JSON shape; inside the default line as `other_configs`
# and selectable alone with --workload
# ----------------------------------------------------------------------------------------------
def secondary(wl, args, tm: Timer, dev, steps: int, with_cpu: bool = True):
    """c1 DeepGini 10k x 10 (+ APFD parity), c3 LSA 10k x 60k x 256 (bf16-stored traces; + per-class LSA),
    c4 KMNC 10k x 4096 x 1000 sections — BASELINE.json configs 1, 3, 4 on one B200."""
    import torch

    from oracle import c_oracle, np_oracle   # synthetic generators + cpu_baseline only
    from simple_tip_b200 import _lib
    from simple_tip_b200 import engine as E

    lib = _lib.load()
    tflops_peak, hbm_peak, peak_src = _peaks()
    extra = {}
    no_flush = False
    if wl == "c3":
        from simple_tip_b200.core.apfd import apfd_from_order
        from simple_tip_b200.core.surprise import LSA, MultiModalSA

        xtr, ytr, xte, pte, yte = np_oracle.synth_clusters(60000, 10000, 256, 10, seed=3, spread=1.0)
        rb = lambda a: torch.from_numpy(a).to(torch.bfloat16).to(torch.float32).numpy()   # bf16-stored traces
        xtr, xte = rb(xtr), rb(xte)
        sa = LSA(xtr)
        kde = sa.kde
        xd = E.to_device(xte, dev)
        pinned = torch.from_numpy(xte).pin_memory().numpy()
        n_units, metric = 10000, "lsa_inputs_prioritized_per_sec"
        sa(xte)                                    # the first call measures whether the one-segment fp16 pass is accurate enough
        fast = bool(kde._engine.fast_ok)
        scheme = kde.last_operands
        extra["operand_scheme"] = {"used": scheme, "check": getattr(kde, "last_fast_check", None),
                                   "note": "fp16 x1 = one tensor-core segment, accepted only after its -log density agreed with "
                                           "the split-bf16 x3 pass to rtol 4e-5 on 128 sampled inputs of this very batch; the "
                                           "e2e time includes that check on every call"}
        dtype = f"{scheme} tensor-core dot, fp32 log-sum-exp, f64 finish"
        workload = "C3: LSA Gaussian-KDE 10000 test x 60000 train x 256-d, traces stored in bf16 (seed 3)"
        # device step = whiten + pack + tensor-core log-sum-exp + merge for the whole batch, launched eagerly (as in
        # round 1).  A scoring call additionally verifies the fast pass on 128 sampled inputs (a three-segment pass) and
        # packs the partials; from the second sighting of a batch shape the product replays ALL of that as one CUDA
        # graph: `device_call_graph_ms` (and e2e) include it.
        step_device = lambda: kde._engine.log_kernel_sum(E.whiten(xd, None, kde._mu_dev, kde._w_dev), fast=fast)
        sa(xd)
        sa(xd)                                     # second sighting of the batch shape: captured
        plans = [p for k, p in getattr(kde, "_plans", {}).items() if k[0] == 10000]
        if plans:
            plans[0].x_in.copy_(xd)
            for _ in range(3):
                plans[0].graph.replay()
            torch.cuda.synchronize()
            extra["device_call_graph_ms"] = float(np.sum(tm.timed(plans[0].graph.replay, steps))) / steps
        step_e2e = lambda: sa(pinned)
        h2d, d2h = int(xte.nbytes), 2 * 10000 * 8
        flops = 2.0 * 256 * 10000 * 60000

        def roofline(ms):
            return {"kernel": "pair_kernel<MODE_LSE> + whiten/pack/merge (whole device step)", "bound": "tensor",
                    "achieved": flops / (ms * 1e-3) / 1e12, "peak": tflops_peak, "unit": "TFLOP/s",
                    "frac": flops / (ms * 1e-3) / 1e12 / tflops_peak, "traffic": None, "peak_source": peak_src,
                    "note": f"algorithmic 2*D flop per pair; operand scheme: {scheme}"}

        # parity at the full size: sampled rows against the float64 oracle (no absolute floor), APFD of the order
        sub = np.sort(np.random.default_rng(0).choice(10000, 256, replace=False))
        got_all = sa(xte)
        want = np_oracle.lsa_oracle(xtr, xte[sub], exact=True)
        rel = np.abs(got_all[sub] - want) / np.abs(want)
        extra["parity"] = {"rows": int(sub.size), "max_rel_err": float(rel.max()), "rtol_1e-4_ok": bool((rel <= 1e-4).all()),
                           "oracle": "np_oracle.lsa_oracle(exact=True): float64 restatement of scipy 1.4.1 gaussian_kde"}
        # what the study runs (handler_surprise.py:26): one LSA per predicted class
        pc = MultiModalSA.build_by_class(xtr, ytr, lambda x, y: LSA(x))
        for _ in range(3):                      # first sighting eager, second captures the per-class graphs, third replays
            pc(pinned, pte)
        t_pc = tm.timed(lambda: pc(pinned, pte), steps)
        pairs_pc = float(sum(int((pte == c).sum()) * int((ytr == c).sum()) for c in range(10)))
        extra["pc_lsa"] = {"ms_per_step_e2e": float(np.mean(t_pc)), "ms_per_step_e2e_median": float(np.median(t_pc)),
                           "inputs_per_s_e2e": 10000 / (np.mean(t_pc) * 1e-3),
                           "pairs": pairs_pc, "note": "MultiModalSA.build_by_class(LSA): 10 per-class KDEs, "
                           "sum_c N_test,c x N_train,c pairs; end to end from pinned host memory"}
        fault = pte != yte
        want_pc = np_oracle.pc_lsa_oracle(xtr, ytr, xte[sub], pte[sub])
        got_pc = pc(xte, pte)
        fin = np.isfinite(want_pc)
        rel_pc = np.abs(got_pc[sub][fin] - want_pc[fin]) / np.abs(want_pc[fin])
        extra["pc_lsa"]["max_rel_err_256_rows"] = float(rel_pc.max()) if fin.any() else None
        extra["pc_lsa"]["inf_pattern_equal"] = bool(np.array_equal(np.isinf(got_pc[sub]), np.isinf(want_pc)))
        extra["pc_lsa"]["inf_rows"] = int((~fin).sum())
        extra["apfd_lsa_order"] = float(apfd_from_order(fault, np.argsort(-got_all)))

        def cpu():
            n_s = 600          # ~10 s of single-threaded CPU work
            kf = np_oracle.KdeFit(xtr.T.astype(np.float64))
            w = np.linalg.cholesky(kf.inv_cov)
            p, q = kf.dataset.T @ w, xte[:n_s].astype(np.float64) @ w
            t0 = time.perf_counter()
            c_oracle.kde_eval(p, q, 1.0 / kf.n, 1.0, threads=1)
            dt = time.perf_counter() - t0
            return {"value": n_s / dt, "unit": "inputs/s", "cores": 1, "kind": "port",
                    "sample": f"{n_s} test inputs vs all 60000 train rows, {dt:.1f} s; literal loop nest of scipy 1.4.1 "
                              "gaussian_kernel_estimate (single-threaded, as in the reference)"}
    elif wl == "c4":
        from simple_tip_b200.core.neuron_coverage import KMNC

        act, mins, maxs = np_oracle.synth_relu(10000, 4096, seed=4)
        km = KMNC([mins], [maxs], 1000)
        pinned = torch.from_numpy(act).pin_memory().numpy()
        km.buckets([act[:8]])
        a_dev = E.to_device(act, dev)
        lo, jp = km._dev_stats
        bucket = torch.empty((10000, 4096), dtype=torch.int16, device=dev)
        score = torch.empty(10000, dtype=torch.int32, device=dev)
        n_units, metric, dtype = 10000, "kmnc_inputs_profiled_per_sec", "f32 compare, i16 bucket ids"
        workload = "C4: KMNC 10000 x 4096 ReLU traces, 1000 sections (seed 4); compact bucket ids + scores"
        # A second figure alternates between two input / output sets without the flush write (164 MB in + 82 MB out per
        # step exceed the 126 MB L2 anyway): there the dirty lines written back underneath the kernel are the previous
        # step's own bucket ids instead of the flush pattern.  Both are steady-state figures; ncu, which starts every
        # launch from a CLEAN L2, sees 45 us (profiles/r02_kmnc_strip_kernel_ncu_full.json).
        sets = [(a_dev, bucket), (a_dev.clone(), torch.empty_like(bucket))]
        turn = [0]

        def step_device():
            a, b = sets[turn[0] & 1]
            turn[0] += 1
            lib.tip_kmnc(E._p(a), 0, 10000, 4096, E._p(lo), E._p(jp), 0, 1000, E._p(b), 3, E._p(score), E._stream())

        step_e2e = lambda: km.buckets([pinned])
        no_flush = True
        h2d, d2h = int(act.nbytes), 10000 * 4096 * 2 + 10000 * 4
        nbytes = act.nbytes + 10000 * 4096 * 2 + 2 * 4096 * 4 + 10000 * 4

        def roofline(ms):
            return {"kernel": "kmnc_strip_kernel", "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm_peak,
                    "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": None, "peak_source": peak_src}

        def cpu():
            n_s, k_s = 2000, 50    # the dense N x D x k profile of the reference is 41 GB at k=1000
            t0 = time.perf_counter()
            np_oracle.kmnc_oracle([mins], [maxs], k_s, [act[:n_s]])
            dt = time.perf_counter() - t0
            per_section = dt / (n_s * k_s)
            return {"value": 1.0 / (per_section * 1000), "unit": "inputs/s", "cores": 1, "kind": "port",
                    "sample": f"{n_s} inputs at sections={k_s} ({dt:.2f} s), cost scaled linearly to 1000 sections "
                              "(the reference loops over sections, neuron_coverage.py:90-93)"}
    elif wl == "cam":
        # the step after every coverage score in the study (handler_coverage.py:122-124): CAM over NAC_0.75 profiles at
        # MNIST's 36 384 neurons (case_study_mnist.py:50-62) and over KMNC bucket ids at C4's shape, neither leaving HBM
        from simple_tip_b200.core.neuron_coverage import KMNC, NAC
        from simple_tip_b200.core.prioritizers import cam_from_bits, cam_from_buckets

        rng = np.random.default_rng(6)
        n, d = 10000, 36384
        act = torch.clamp(torch.randn((n, d), device=dev, generator=torch.Generator(device=dev).manual_seed(6)) * 0.5 + 0.1, min=0)
        nac = NAC(0.75)
        score_d, bits = nac.packed(act)
        score = score_d.cpu().numpy()
        order = np.array(list(cam_from_bits(score, bits)))
        chk = np.sort(rng.choice(n, 300, replace=False))          # a sub-problem small enough for the NumPy restatement
        s_s, b_s = nac.packed(act[torch.from_numpy(chk).to(dev)][:, :4096].contiguous())
        _, p_s = nac(act[torch.from_numpy(chk).to(dev)][:, :4096].contiguous())
        ok_bits = bool(np.array_equal(np.array(list(cam_from_bits(s_s.cpu().numpy(), b_s))),
                                      np_oracle.cam_oracle(s_s.cpu().numpy(), p_s)))
        st = torch.zeros(4, dtype=torch.int32)
        t0 = time.perf_counter()
        greedy_rounds = 0
        for _ in range(3):
            greedy_rounds = sum(1 for _ in cam_from_bits(score, bits))
        torch.cuda.synchronize()
        dt_bits = (time.perf_counter() - t0) / 3
        words = int(bits.shape[1])
        # rounds actually run by the greedy loop: samples yielded before the tail = picks with positive gain
        from simple_tip_b200.core import prioritizers as P
        picks_bits, dev_ms_bits = int(P.LAST_GREEDY_PICKS), float(P.LAST_GREEDY_MS)
        actk, mins, maxs = np_oracle.synth_relu(10000, 4096, seed=4)
        km = KMNC([mins], [maxs], 1000)
        ks, kb = km.buckets([torch.from_numpy(actk).to(dev)], device_out=True)
        ksn = ks.cpu().numpy()
        t0 = time.perf_counter()
        n_b = sum(1 for _ in cam_from_buckets(ksn, kb, 1000))
        torch.cuda.synchronize()
        dt_bk = time.perf_counter() - t0
        picks_bk = int(P.LAST_GREEDY_PICKS)
        sub = kb[:200, :512].contiguous()
        ss = ((sub >= 0).sum(dim=1)).cpu().numpy()
        ok_bk = bool(np.array_equal(np.array(list(cam_from_buckets(ss, sub, 1000))),
                                    np_oracle.cam_from_buckets_oracle(ss, sub.cpu().numpy().astype(np.int32), 1000)))
        return {"metric": "cam_greedy_rounds_per_sec", "unit": "rounds/s", "data": "synthetic", "n_gpus": 1,
                "bits": {"workload": f"CAM over NAC_0.75 profiles, {n} samples x {d} neurons, bit-packed in HBM ({words} words per sample)",
                         "kernel": "cam_bits_kernel (one persistent cooperative launch for all rounds)", "greedy_rounds": picks_bits,
                         "ms_total": 1e3 * dt_bits, "ms_device_greedy_loop": dev_ms_bits,
                         "rounds_per_s": picks_bits / (dev_ms_bits * 1e-3) if dev_ms_bits > 0 else None,
                         "us_per_round": 1e3 * dev_ms_bits / max(1, picks_bits),
                         "bytes_per_round_worst_case": int(n * words * 4), "order_is_a_permutation": bool(sorted(order.tolist()) == list(range(n))),
                         "sub_problem_equals_numpy_restatement": ok_bits,
                         "note": "a round reads only the non-zero words of the pick's new coverage for samples with gain left, "
                                 "so the worst-case bytes are an upper bound"},
                "buckets": {"workload": "CAM over KMNC bucket ids, 10000 x 4096, 1000 sections (C4's profile: 41 GB dense)",
                            "kernel": "cam_pick / cam_collect / cam_update (3 launches per round)", "greedy_rounds": picks_bk,
                            "ms_total": 1e3 * dt_bk, "rounds_per_s": picks_bk / dt_bk if dt_bk > 0 else None,
                            "sub_problem_equals_numpy_restatement": ok_bk},
                "value": picks_bits / (dev_ms_bits * 1e-3) if dev_ms_bits > 0 else None, "higher_is_better": True}
    else:   # c1
        from simple_tip_b200.core.apfd import apfd_from_order
        from simple_tip_b200.core.deepgini import DeepGini

        p, truth = np_oracle.synth_softmax(10000, 10, seed=1)
        pinned = torch.from_numpy(p).pin_memory().numpy()
        p_dev = E.to_device(p, dev)
        pred_d = torch.empty(10000, dtype=torch.int32, device=dev)
        gini_d = torch.empty(10000, dtype=torch.float32, device=dev)
        n_units, metric, dtype = 10000, "deepgini_inputs_prioritized_per_sec", "f32"
        workload = "C1: DeepGini on 10000 x 10 softmax outputs (seed 1) + APFD"
        step_device = lambda: lib.tip_deepgini(E._p(p_dev), 0, 10000, 10, E._p(pred_d), E._p(gini_d), E._stream())
        step_e2e = lambda: DeepGini.calculate(pinned)
        h2d, d2h = int(p.nbytes), 10000 * 8
        nbytes = p.nbytes + 10000 * 8
        pred, gini = DeepGini.calculate(p)
        wp, wg = np_oracle.deepgini_oracle(p)
        fault = wp != truth
        extra["apfd"] = {"ours": float(apfd_from_order(fault, np.argsort(-gini))),
                         "oracle": float(np_oracle.apfd_oracle(fault, np.argsort(-wg))),
                         "scores_bit_identical": bool(np.array_equal(gini, wg) and np.array_equal(pred, wp))}

        def roofline(ms):
            return {"kernel": "gini_small_kernel", "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm_peak,
                    "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": None, "peak_source": peak_src,
                    "note": "480 KB problem: one launch, latency-bound by construction (the roofline time is 0.07 us)"}

        def cpu():
            t0 = time.perf_counter()
            for _ in range(200):
                np_oracle.deepgini_oracle(p)
            dt = (time.perf_counter() - t0) / 200
            return {"value": 10000 / dt, "unit": "inputs/s", "cores": 1, "kind": "port",
                    "sample": "whole 10000 x 10 batch, NumPy expressions of deepgini.py:33-34, mean of 200 runs"}

    for _ in range(max(3, args.warmup)):
        step_device()
        step_e2e()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    t_dev = float(np.sum(tm.timed(step_device, steps)))
    launches = (_lib.launch_count() - l0) // max(1, steps)
    l2_note = "flushed between steps (256 MiB write)"
    if no_flush:
        extra["ms_per_step_alternating_sets_no_flush"] = float(np.sum(tm.timed(step_device, steps, flush=False))) / steps
    t_e2e_steps = tm.timed(step_e2e, steps)
    t_e2e = float(np.sum(t_e2e_steps))
    line = {"metric": metric, "value": n_units * steps / (t_dev * 1e-3), "unit": "inputs/s", "n_gpus": 1,
            "steps": steps, "warmup": max(3, args.warmup), "ms_per_step": t_dev / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {"workload": workload, "l2": l2_note, "timing": "per-step CUDA events, summed"},
            "e2e": {"value": n_units * steps / (t_e2e * 1e-3), "unit": "inputs/s", "ms_per_step": t_e2e / steps,
                    "ms_per_step_median": float(np.median(t_e2e_steps)), "ms_per_step_max": float(np.max(t_e2e_steps)),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "roofline": roofline(t_dev / steps)}
    line.update(extra)
    line["stall_retries_so_far"] = tm.stall_retries
    if with_cpu:
        line["cpu_baseline"] = cpu()
    return line


def run_secondary(args):
    import torch

    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    tm = Timer(dev)
    sampler = ClockSampler(0)
    sampler.start()
    if args.workload == "c5s":
        line = run_c5_slice(args, tm, dev, 0, 1, None, steps=args.steps)
    else:
        line = secondary(args.workload, args, tm, dev, args.steps, with_cpu=not args.no_cpu)
    line["clocks"] = sampler.stop()
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs (profiling runs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the n_train_sharded block (C5-shaped slice)")
    ap.add_argument("--no-others", action="store_true", help="skip other_configs (C1 / C3 / C4)")
    ap.add_argument("--parity-inputs", type=int, default=48, help="inputs of the C5 slice checked against the CPU oracle")
    ap.add_argument("--shard", default="auto", choices=["auto", "test", "train"],
                    help="multi-GPU layout of the C2 headline: test = N_test sharded, train replicated (default: the "
                         "train set is 30.7 MB); train = N_train sharded (what C5 needs; always measured on the C5-shaped "
                         "slice in n_train_sharded)")
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5s", "cam"],
                    help="c2 (default) = the configuration the headline metric is quoted on (its line also carries the "
                         "others); c1/c3/c4/c5s = one of the other configurations alone, single GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed C2 step computed as DIR/<name>.npy: dsa, "
                         "dist_a, dist_b, winner_index, float64, one entry per test input (rank 0's), in input order")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs writes the outputs of the C2 headline (--impl ours --workload c2)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload != "c2":
        assert args.gpus == 1, "secondary workloads are single-GPU"
        run_secondary(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
