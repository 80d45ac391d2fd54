#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): training throughput of ``federated_multi`` — ResNet18, FedAvg over
parameter blocks, one worker per GPU, batch 128 per worker, synthetic CIFAR10, random init.

    python bench.py --gpus N --steps K --warmup W            # N=1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W               # N>1, one rank per GPU
    python bench.py --impl reference --gpus N ...            # the unmodified reference through an offline shim
    python bench.py --driver consensus --bb ...              # BASELINE config 3 (adaptive ADMM); --driver fedprox
                                                             # --optimizer lbfgs (config 4); --driver vae | cpc (config 5)
    python bench.py ... --dump-outputs DIR                   # also save what the last step computed (see dump_outputs)

A *step* is one minibatch optimizer step on every worker (128*N images): zero-grad, forward, CE loss, backward,
fused Adam on the active block, and the reference's post-step diagnostics forward; block aggregation (fused
NVLink kernel) happens every ``steps_per_round`` = 49 steps exactly as in the training schedule (K=8-sized shards).
Weak scaling: the per-GPU work is fixed.

THE TIMED WINDOW STRADDLES A ROUND BOUNDARY: the K timed steps are placed so that the aggregation after step 98 (the second
of the run; the first one, after step 49, is warm-up) and every later one the window reaches is inside it — untimed steps
before the window are warm-up.  So every printed number contains at least one fused aggregation (cross-rank kernel at
N > 1) plus the host's one 32-byte read of it.

ONE engine is built per process (dataset synthesis, model, symmetric heap, graph capture happen once); the same
engine then runs the device-timed window (dataset resident in HBM) and, two rounds later, the end-to-end window
(dataset in pinned host memory: every step copies its uint8 batch + labels host->device through the native batch
assembler and the step's loss is copied device->host and read by the host).

Printed JSON (rank 0, one line): ``value`` = images/s of the whole job, device-timed (CUDA events, barrier +
synchronize on both sides, max over ranks); ``e2e`` as described; ``collective`` (N > 1): device time and bus GB/s of
one FedAvg aggregation at each of the ten ResNet18 block sizes for the fused kernel (NVLS and P2P variants, one-shot
vs two-shot) next to NCCL ``all_reduce`` + the ATen epilogue, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

T_PROCESS_START = time.perf_counter()

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STEPS_PER_ROUND = 49      # ceil(6249 / 128): the K=8 shard of the BASELINE config
PRIME_STEPS = 4           # eager warm-up + CUDA-graph capture of the step, before the W warm-up steps
# The device window straddles the SECOND round boundary: the first aggregation of a run is warm-up like the first minibatches are
# (first cross-GPU touch of the block's peer-mapped pages; on one 8-GPU box it cost 9 ms once, the next ones 0.7 ms — r2_scaling.md).
TIMED_BOUNDARY = 2 * STEPS_PER_ROUND
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, eng) -> None:
    """Write what a caller of the training step receives once the run's last step is done: that step's loss
    (``loss.npy``) and the trained model, every ``state_dict`` entry of replica 0 as ``<model>.<key>.npy`` in its logical
    shape.  Inputs (synthetic data, initialisation) are seeded, so two builds run with the same arguments can be compared
    file for file."""
    import numpy as np

    arrays = {"loss": eng.last_loss1.detach().float().reshape(1)}
    for model, net in eng.replicas[0].nets.items():
        for key, t in net.state_dict().items():
            arrays["%s.%s" % (model, key)] = t.detach().float() if t.is_floating_point() else t.detach().double()
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of %d bytes exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().contiguous().numpy())


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self) -> int:
        """Index of the next sample: ``window(mark_at_open, mark_at_close)`` summarises only what was sampled in between."""
        return len(self.rows)

    def window(self, i0: int, i1: int) -> dict:
        return self._summarise(self.rows[max(0, i0 - 1): i1 + 1])      # include the samples that bracket the window

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        return self._summarise(self.rows)

    def _summarise(self, rows) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _max_over_ranks(x: float, device) -> float:
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)
    return x


def straddle_window(K: int, W: int, earliest: int, boundary: int) -> int:
    """First step of a K-step window that contains the aggregation after step ``boundary`` (i.e. steps boundary-1 and
    boundary are both inside), starts no earlier than ``earliest`` and leaves at least W warm-up steps before it."""
    first = boundary - K // 2
    if K >= 2 * STEPS_PER_ROUND or first < earliest + W:
        first = earliest + W          # a window this long (or this early) reaches the boundary anyway / as soon as allowed
    return first


# ----------------------------------------------------------------------------------------------
def _collective_table(coll, topo, eng, iters: int = 20, warm: int = 3):
    """Device time (max over ranks) of ONE FedAvg aggregation at every ResNet18 block size on the replicas' own
    arenas: fused kernel (auto = NVLS when bound, two-shot >= 256 KB), fused with P2P loads/stores only, fused forced
    one-shot, and the NCCL baseline (all_reduce + div + dual norm + write-back: what ``--impl nccl`` runs)."""
    import torch.distributed as dist

    from federated_pytorch_test_b200.parallel.collective import TorchCollective

    dev, Wd = topo.device, topo.world_size
    rep = eng.replicas[0]
    arena = rep.arenas["net"]
    blocks = rep.nets["net"].train_order_block_ids()
    base = TorchCollective(topo)
    rows = []

    def timed(fn):
        for _ in range(warm):
            fn()
        if Wd > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return _max_over_ranks(a.elapsed_time(b) * 1e3 / iters, dev)

    heap_mc = bool(coll.heap.locate(arena.data)[0].get("mc_ptr", 0)) if hasattr(coll, "heap") else False
    for ci, (lo, hi) in enumerate(blocks):
        x = arena.block(lo, hi)
        n = x.numel()
        z = coll.zeros_like_block(x, "z")
        row = {"block": ci, "floats": n, "bytes": 4 * n}
        dflt = bool(getattr(coll, "default_multimem", True))      # multimem (NVLS) from 4 ranks on, P2P loads / stores between 2
        variants = [("fused", dflt, "auto")]
        if Wd > 1:
            variants += [("fused_p2p", False, "auto"), ("fused_nvls", True, "auto"), ("fused_oneshot", dflt, "0")]
        for label, mc, mode in variants:
            coll.use_multimem, coll.two_shot_mode = mc, mode
            row[label + "_us"] = timed(lambda: coll._launch(0, [x], None, z, 0.0))
            row[label + "_two_shot"] = bool(coll.last_two_shot)
        coll.use_multimem, coll.two_shot_mode = dflt, "auto"
        coll.read_record()
        if Wd > 1:
            xr, zr = x.clone(), z.clone()
            row["nccl_us"] = timed(lambda: base.fedavg_([xr], zr, True))
            raw = x.clone()
            row["nccl_allreduce_only_us"] = timed(lambda: dist.all_reduce(raw))
            f = 2.0 * (Wd - 1) / Wd * 4 * n / 1e3          # bytes -> GB/s with us: bus bandwidth convention of nccl-tests
            for k in ("fused", "fused_p2p", "fused_nvls", "fused_oneshot", "nccl", "nccl_allreduce_only"):
                row[k + "_busGBs"] = f / row[k + "_us"]
            row["fused_frac_of_900GBs"] = row["fused_busGBs"] / 900.0
            row["speedup_vs_nccl"] = row["nccl_us"] / row["fused_us"]
            row["speedup_vs_bare_allreduce"] = row["nccl_allreduce_only_us"] / row["fused_us"]
        rows.append(row)
    return {"world": Wd, "multicast_bound": heap_mc, "fused_default": "nvls multimem" if getattr(coll, "default_multimem", True) else "p2p loads/stores", "transport": getattr(getattr(coll, "heap", None), "transport", "n/a"),
            "timing": "CUDA events around %d back-to-back launches after %d warm-up, max over ranks; no host read inside" % (iters, warm),
            "rows": rows}


# ----------------------------------------------------------------------------------------------
def run_ours(args) -> dict:
    from federated_pytorch_test_b200.algo.engine import Engine
    from federated_pytorch_test_b200.algo.strategies import ADMM, BBConfig, FedAvg, FedProx
    from federated_pytorch_test_b200.api import common, consensus_multi, federated_multi, fedprox_multi
    from federated_pytorch_test_b200.ops import cuda_ops

    N, K, W = args.gpus, args.steps, args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == N or (N == 1 and world == 1), "launch with torchrun --nproc-per-node N for N > 1"

    # window placement (see module docstring)
    first_d = straddle_window(K, W, PRIME_STEPS, TIMED_BOUNDARY)
    last_d = first_d + K
    b_host = -(-last_d // STEPS_PER_ROUND) * STEPS_PER_ROUND          # first step served by the host-resident loader
    first_e = straddle_window(K, W, b_host, b_host + STEPS_PER_ROUND)
    last_e = first_e + K
    if args.no_e2e:
        last_e = last_d
    # block 0 (full-depth backward, the most expensive block) stays active for the whole measurement
    nadmm = max(3, -(-last_e // STEPS_PER_ROUND) + 1)

    mod = {"federated": federated_multi, "consensus": consensus_multi, "fedprox": fedprox_multi}[args.driver]
    kw = dict(K=N, use_resnet=True, Nloop=1000, Nadmm=nadmm, Nepoch=1, check_results=False, save_model=False, be_verbose=False,
              biased_input=True, data_on_device=True, graphs=not args.no_graphs, fast=not args.no_fast,
              collective=args.collective, diagnostics=args.diagnostics, max_minibatches=STEPS_PER_ROUND, seed=69,
              optimizer=args.optimizer)
    if args.driver == "consensus":
        kw["bb_update"] = bool(args.bb)
    cfg = mod.Config(**kw)
    topo, coll = common.setup_runtime(cfg)
    task = common.ClassifierTask(cfg, topo, cfg.lambda1, cfg.lambda2)
    if args.driver == "federated":
        strat = FedAvg(coll, topo)
    elif args.driver == "fedprox":
        strat = FedProx(coll, topo, len(task.blocks), cfg.admm_rho0)
    else:
        strat = ADMM(coll, topo, len(task.blocks), cfg.admm_rho0, BBConfig(enabled=bool(args.bb)), log=lambda m: None)
    eng = Engine(task, topo, strat, coll, common.engine_config(cfg), log=lambda m: None)
    dev = topo.device
    t_built = time.perf_counter()

    ev_d = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    ev_e = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    st = {"d": {}, "e": {}, "t_first_step": None, "loss": None, "wait": 0.0, "aggs0": 0}
    # D2H read of every step's loss (e2e window): async copy into a pinned slot right after the step is enqueued, consumed
    # one step later (the host stays one step ahead of the GPU, so host jitter does not idle the device).
    slots = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    slot_ev = [torch.cuda.Event(), torch.cuda.Event()]
    pending = []
    # ONE nvidia-smi sampler for the whole run, started before the first step: its start-up (NVML attaches to every GPU of the
    # box) stalls CUDA launches of ALL ranks for tens of ms on an 8-GPU node — inside a 50 ms window that contains a cross-rank
    # aggregation this was measured as a 30 ms "step" (profiles/r2_scaling.md).  The windows only mark sample indices.
    smi = ClockSampler(dev.index or 0) if (topo.is_root and os.environ.get("FEDB200_BENCH_NO_SMI", "0") != "1") else None
    if smi:
        smi.start()

    import gc

    gc.collect()
    gc.freeze()           # everything built so far is long-lived: keep it out of the collector's generations

    def open_window(tag, ev):
        gc.collect()
        gc.disable()      # a cyclic-GC pause (~10 ms with this heap) inside a 50 ms window is 20 % noise; re-enabled at close
        topo.barrier()
        torch.cuda.synchronize(dev)
        st[tag]["smi0"] = smi.mark() if smi else 0
        st[tag].update(l0=cuda_ops.launch_count(), g0=getattr(eng, "graph_kernel_launches", 0), a0=eng.aggregations_done,
                       t0=time.perf_counter())
        st["wait"] = 0.0
        ev.record()

    def close_window(tag, ev):
        ev.record()
        torch.cuda.synchronize(dev)
        topo.barrier()
        gc.enable()
        s = st[tag]
        s["t1"] = time.perf_counter()
        s["launches"] = (cuda_ops.launch_count() - s["l0"]) + (getattr(eng, "graph_kernel_launches", 0) - s["g0"])
        s["aggregations"] = eng.aggregations_done - s["a0"]
        s["wait_ms"] = st["wait"] * 1e3
        s["clocks"] = smi.window(s["smi0"], smi.mark()) if smi else None

    def swap_to_host_loaders():
        """From the next round on, batches come from pinned host memory through the native batch assembler."""
        host = task.data_host if getattr(task, "data_host", None) is not None else None
        if host is None:
            from federated_pytorch_test_b200.data.cifar import CifarData

            d = task.data
            host = CifarData(d.train_images.cpu(), d.train_labels.cpu(), d.test_images.cpu(), d.test_labels.cpu()).to(dev, pin=True)
        task.data = host
        task._loaders.clear()

    step_ev = {"d": [], "e": []}   # one CUDA event per step of a timed window: is a slow window uniform, or one long step?

    def stamp(tag):
        evn = torch.cuda.Event(enable_timing=True)
        evn.record()
        step_ev[tag].append(evn)

    def hook(e: Engine):
        n = e.steps_done
        if first_d < n <= last_d:
            stamp("d")
        elif (not args.no_e2e) and first_e < n <= last_e:
            stamp("e")
        if n == 1 and st["t_first_step"] is None:
            torch.cuda.synchronize(dev)
            st["t_first_step"] = time.perf_counter() - T_PROCESS_START
        in_e2e = (not args.no_e2e) and first_e <= n - 1 < last_e          # the step just finished was an e2e step
        if in_e2e and e.last_loss1 is not None:
            i = n & 1
            slots[i].copy_(e.last_loss1.detach().reshape(()), non_blocking=True)     # D2H of this step's result
            slot_ev[i].record()
            pending.append(i)
            tw = time.perf_counter()
            while len(pending) > (0 if n >= last_e else 1):          # consume the previous step's value (all at the end)
                j = pending.pop(0)
                slot_ev[j].synchronize()
                st["loss"] = float(slots[j])
            st["wait"] += time.perf_counter() - tw
        if n == first_d:
            open_window("d", ev_d[0])
        elif n == last_d:
            close_window("d", ev_d[1])
            if args.no_e2e:
                e.stop_requested = True
            else:
                swap_to_host_loaders()
        elif n == first_e and not args.no_e2e:
            open_window("e", ev_e[0])
        elif n == last_e and not args.no_e2e:
            close_window("e", ev_e[1])
            e.stop_requested = True

    eng.step_hook = hook
    eng.run()
    if args.dump_outputs and topo.is_root:
        dump_outputs(args.dump_outputs, eng)
    ms_d = _max_over_ranks(ev_d[0].elapsed_time(ev_d[1]), dev)
    images = 128 * N * K
    value = images / (ms_d / 1e3)
    loader = task.loader(topo.local_workers[0])
    out = {
        "metric": "train_images_per_sec", "value": value, "unit": "images/s", "n_gpus": N, "steps": K, "warmup": W,
        "ms_per_step": ms_d / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32" if not args.no_fast else "fp32(tf32 conv)", "data": "synthetic", "impl": args.impl,
        "config": {"model": "ResNet18", "algo": {"federated": "fedavg", "consensus": "admm" + ("+bb" if args.bb else ""), "fedprox": "fedprox"}[args.driver],
                   "optimizer": args.optimizer, "global_batch": 128 * N, "per_gpu_batch": 128, "K": N,
                   "parallelism": "fed%d (one replica per GPU, block aggregation over NVLink)" % N,
                   "steps_per_round": STEPS_PER_ROUND, "rounds_per_block_visit": nadmm, "diagnostics_forward": args.diagnostics,
                   "cuda_graphs": not args.no_graphs, "collective": coll.name,
                   "symmetric_heap": getattr(getattr(coll, "heap", None), "transport", "n/a"),
                   "timed_steps": [first_d, last_d], "aggregations_in_window": st["d"].get("aggregations"),
                   "aggregation_two_shot": bool(getattr(coll, "last_two_shot", False)),
                   "warmup_steps_before_window": first_d,
                   "l2": "per-step working set (~1 GB of fp32 activations) exceeds the 126 MB L2; no explicit flush",
                   "timing": "CUDA events on the step stream, barrier+synchronize both sides, max over ranks"},
        "clocks": st["d"].get("clocks"),
        "gpu_launches": st["d"].get("launches"),
        "time_to_first_step_s": st["t_first_step"], "build_s": t_built - T_PROCESS_START,
    }
    def per_step(tag, ev0):
        evs = [ev0] + step_ev[tag]
        if len(evs) < 3:
            return None
        per = [round(a.elapsed_time(b), 3) for a, b in zip(evs[:-1], evs[1:])]
        return {"min": min(per), "median": statistics.median(per), "max": max(per), "argmax_step": per.index(max(per)),
                "note": "this rank's CUDA event after every step of the window; the step that contains the aggregation (waiting for "
                        "the slowest rank included) and the host's read of its record is the max"}

    out["config"]["per_step_ms"] = per_step("d", ev_d[0])
    if smi:
        smi.stop()
    if not args.no_e2e:
        ms_e = _max_over_ranks(ev_e[0].elapsed_time(ev_e[1]), dev)
        wall_e = _max_over_ranks((st["e"]["t1"] - st["e"]["t0"]) * 1e3, dev)
        out["e2e"] = {"value": images / (max(ms_e, wall_e) / 1e3), "unit": "images/s", "ms_per_step": max(ms_e, wall_e) / K,
                      "h2d_bytes_per_step": loader.h2d_bytes_per_batch * (1 if loader.host_resident else 0), "d2h_bytes_per_step": 4,
                      "device_ms_per_step": ms_e / K, "wall_ms_per_step": wall_e / K,
                      "host_wait_ms_per_step": st["e"]["wait_ms"] / K, "host_cpus": len(os.sched_getaffinity(0)),
                      "timed_steps": [first_e, last_e], "aggregations_in_window": st["e"].get("aggregations"),
                      "last_loss_read_by_host": st["loss"],
                      "note": "same engine, dataset moved to pinned host memory: native batch assembler, async H2D of each uint8 batch, "
                              "every step's loss copied D2H into pinned memory and read by the host one step later; "
                              "per-rank bytes (x N for the job)",
                      "per_step_ms": per_step("e", ev_e[0]),
                      "clocks": st["e"].get("clocks"), "gpu_launches": st["e"].get("launches")}
    if not args.no_collective_table and hasattr(coll, "_launch") and "ResNet" in task.model_name:
        try:
            out["collective"] = _collective_table(coll, topo, eng)
        except Exception as exc:      # the table must never cost the headline number
            out["collective"] = {"error": repr(exc)}
    return out if topo.is_root else {}


# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"],
                    help="ours | reference (unmodified reference via shim) | nccl (BASELINE 'ref-nccl': ATen model + NCCL all-reduce)")
    ap.add_argument("--driver", default="federated", choices=["federated", "consensus", "fedprox", "vae", "vae_cl", "cpc"],
                    help="which entry point is benchmarked (default: the headline federated_multi / FedAvg)")
    ap.add_argument("--algo", default=None, choices=[None, "fedavg", "admm"], help="alias: admm = --driver consensus")
    ap.add_argument("--bb", action="store_true", help="consensus: Barzilai-Borwein adaptive rho (BASELINE config 3)")
    ap.add_argument("--optimizer", default="adam", choices=["adam", "lbfgs"])
    ap.add_argument("--collective", default="auto", choices=["auto", "fused", "torch"])
    ap.add_argument("--diagnostics", default="post", choices=["post", "pre"])
    ap.add_argument("--no-graphs", dest="no_graphs", action="store_true")
    ap.add_argument("--no-fast", dest="no_fast", action="store_true")
    ap.add_argument("--no-e2e", dest="no_e2e", action="store_true")
    ap.add_argument("--no-collective-table", dest="no_collective_table", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss and the trained model to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.algo == "admm":
        args.driver = "consensus"
    if args.impl == "nccl":   # the "baseline, not the product": stock ATen ops, eager, NCCL all-reduce on the flat block
        args.no_fast, args.no_graphs, args.collective = True, True, "torch"

    if args.dump_outputs and (args.impl == "reference" or args.driver in ("vae", "vae_cl", "cpc")):
        ap.error("--dump-outputs is supported for the ResNet18 drivers (federated, consensus, fedprox) of this implementation")
    if args.impl == "reference":
        from baseline.ref_shim import run_reference_bench

        res = run_reference_bench(args.gpus, args.steps, args.warmup, driver=args.driver, bb=args.bb, optimizer=args.optimizer)
    elif args.driver in ("vae", "vae_cl", "cpc"):
        from baseline.bench_aux import run_aux_bench

        res = run_aux_bench(args)
    else:
        res = run_ours(args)
    if res:
        print(json.dumps(res), flush=True)
    try:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
