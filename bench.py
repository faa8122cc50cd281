#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): samples/sec of the 2-layer-1024 LSTM, seq_len 128, batch 256 per GPU, bf16,
per-step gradient allreduce, synthetic sequences / random-init weights.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference|baseline] [--dump-outputs DIR]

N > 1 is launched by the driver under torchrun (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from the env), one rank
per GPU.  Rank 0 prints ONE JSON line.  ``value`` is the whole-job aggregate (sum over GPUs); timing is CUDA events
on the launching stream bracketed by barrier + synchronize, max over ranks.

  --impl ours       this framework through its public API (lstm_tensorspark_b200.engine.TrainEngine)
  --impl reference  the unmodified reference from baseline/_ref — it is Python-2 / TF-1.0 / PySpark source without
                    packaging metadata and cannot be installed here (DESIGN.md §Reference arm) -> "unavailable"
  --impl baseline   our stand-in for "the reference's own NCCL(+cuBLAS) build" (BASELINE.md §2): cuDNN nn.LSTM +
                    NCCL all_reduce + torch fused Adam, same model / schedule (baseline/harness.py)
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = dict(hidden_units="1024,1024", in_features=1024, seq_len=128, batch_size=256, num_classes=10)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "baseline"])
    ap.add_argument("--comm", default="auto", help="ours: fused (default for N>1) | nccl")
    ap.add_argument("--optimizer", default="adam")
    ap.add_argument("--cuda_graph", type=int, default=-1, help="-1 auto (capture the step when there is one rank), 0 eager, 1 force")
    ap.add_argument("--no_baseline", action="store_true", help="ours: skip timing the cuDNN+NCCL stand-in arm afterwards")
    ap.add_argument("--baseline_variant", default="tuned", choices=["stock", "tuned"], help="--impl baseline: which stand-in")
    ap.add_argument("--grad_buckets", type=int, default=1, help="ours, N>1: per-layer gradient buckets overlapped with backward")
    ap.add_argument("--hidden_units", default=MODEL["hidden_units"])
    ap.add_argument("--in_features", type=int, default=MODEL["in_features"])
    ap.add_argument("--seq_len", type=int, default=MODEL["seq_len"])
    ap.add_argument("--batch_size", type=int, default=MODEL["batch_size"])
    ap.add_argument("--no_e2e", action="store_true")
    ap.add_argument("--e2e_depth", type=int, default=2, help="staging slots of the end-to-end loader (copy enqueued depth-1 steps ahead)")
    ap.add_argument("--bind_inputs", type=int, default=1, help="1 = CUDA graphs captured on the input buffers themselves (no staging copy)")
    ap.add_argument("--config", type=int, default=3, choices=[3, 4],
                    help="BASELINE.json config: 3 = 2x1024 T=128 B=256 per-step grad allreduce (headline); "
                         "4 = 4x2048 T=512 B=64 per-epoch parameter average (one average inside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="ours: after the device-timed steps, write the loss of the last step and the model variables it left as "
                         "DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write ``arrays`` (name -> numpy array) as ``out_dir/<name>.npy`` ("/" in a name becomes "."), float64 kept, anything
    else as float32, ``budget`` bytes in all: every array gets an equal share, and one larger than its share is stored as a
    fixed, seeded sample of its elements (flattened, the same indices on every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays) - 256                      # room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        cap = share // a.itemsize
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name.replace("/", ".") + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []          # (arrival time, csv line)
        self.proc = None
        self.nvml = None
        self.gpu = gpu_index
        self.t_mark = None

    def start(self):
        # NVML in-process (10 ms period: the timed region of a short run is ~100 ms); nvidia-smi -lms as the fallback
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.stop_evt = threading.Event()
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        bits = ((0x8, "Active"), (0x40, "Active"), (0x20, "Active"), (0x4, "Active"))     # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        while not self.stop_evt.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = 0.0
                flags = ",".join(("Active" if mask & b else "Not Active") for b, _ in bits)
                self.rows.append((time.time(), f"{self.gpu}, {sm}, {mx}, {pw:.1f}, {flags}"))
            except Exception:
                pass
            self.stop_evt.wait(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        """Start of the timed region: samples before this are warm-up."""
        self.t_mark = time.time()

    def stop(self):
        if getattr(self, "nvml", None) is not None:
            self.stop_evt.set()
            self.t.join(1.0)
        elif self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        else:
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        timed = [r for (t, r) in self.rows if self.t_mark is None or t >= self.t_mark]
        window = "timed region"
        if len(timed) < 2:                       # run shorter than the sampling period: use the samples under load
            timed = [r for (_, r) in self.rows[1:]] or [r for (_, r) in self.rows]
            window = "warm-up + timed region"
        for r in timed:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


def run_reference(args):
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    why = ("reference is Python-2/TensorFlow-1.0/PySpark source with no setup.py/pyproject (pip install fails: "
           "'neither setup.py nor pyproject.toml found'); tensorflow and pyspark are not in this image")
    if os.path.isdir(ref_dir) and any(f.endswith(".py") for _, _, fs in os.walk(ref_dir) for f in fs):
        why = "reference sources present under baseline/_ref but need python2 + tensorflow 1.0 + pyspark (absent)"
    rank, _, _ = dist_env()
    if rank == 0:
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def timed_loop(torch, dist, world, device, step_fn, steps, warmup, clocks=None):
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize(device)
    if clocks is not None:
        clocks.mark()
    if world > 1:
        dist.barrier(device_ids=[device.index])
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for _ in range(steps):
        last = step_fn()
    e1.record()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier(device_ids=[device.index])
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, last


def measure(torch, dist, world, device, local, step_dev, step_e2e, steps, warmup, no_e2e, B, n_gpus, h2d, d2h, after_timed=None):
    """Device-timed loop (+ clocks sampled during it) and the end-to-end loop of one arm.  ``after_timed(last)`` runs between
    the two with what the last device-timed step returned."""
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)
    ms, last = timed_loop(torch, dist, world, device, step_dev, steps, warmup, clocks)
    clk = clocks.stop()
    if after_timed is not None:
        after_timed(last)
    e2e = None
    if not no_e2e:
        ms_e2e, _ = timed_loop(torch, dist, world, device, step_e2e, steps, max(3, warmup // 2))
        e2e = {"value": B * n_gpus * steps / (ms_e2e / 1e3), "unit": "samples/s", "ms_per_step": ms_e2e / steps,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
    return ms, clk, e2e


def run_baseline_arm(torch, dist, args, hidden, D, C, B, T, rank, world, device, local, variant):
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import harness
    runner = harness.BaselineRunner(hidden, D, C, B, T, rank, world, device, optimizer=args.optimizer, variant=variant)
    runner.bind_inputs = bool(args.bind_inputs) and args.config == 3      # same input binding as our arm
    step_dev, step_e2e, h2d, d2h, launches, cfg_extra = runner.make_steps()
    ms, clk, e2e = measure(torch, dist, world, device, local, step_dev, step_e2e, args.steps, args.warmup, args.no_e2e, B, world, h2d, d2h)
    res = {"value": B * world * args.steps / (ms / 1e3), "ms_per_step": ms / args.steps, "clocks": clk, "e2e": e2e, "config": cfg_extra}
    del runner, step_dev, step_e2e
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return res


def verify_fused_step(torch, dist, eng, comm, world, rank, device):
    """N > 1: correctness evidence for the fused allreduce + Adam kernel on the box that produced the numbers - replicas
    bit-identical after the timed steps, and one extra fused step on known gradients against the closed-form Adam update."""
    flat, opt = eng.flat, eng.optimizer
    n = flat.padded_numel
    torch.cuda.synchronize(device)
    # (1) replicas identical: compare 64-bit checksums of the raw fp32 bit patterns
    bits = flat.data.view(torch.int32).to(torch.int64)
    chk = torch.stack([bits.sum(), (bits * (torch.arange(n, device=device, dtype=torch.int64) % 8191 + 1)).sum()])
    allc = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    identical = all(bool(torch.equal(allc[0], c)) for c in allc)
    # (2) one fused step from a clean Adam state on rank-dependent gradients
    out = {"replicas_identical": identical}
    if opt.kind == "adam" and hasattr(comm, "grad_step_"):
        w0 = flat.data.clone()
        opt.m.zero_(); opt.v.zero_(); opt.step_count = 0
        if opt.step_dev is not None:
            opt.step_dev.zero_()
        idx = torch.arange(n, device=device, dtype=torch.float32)
        gs = [1.0 + 0.5 * torch.sin(idx * 0.01 * (r + 1)) for r in range(world)]
        flat.grad.copy_(gs[rank])
        torch.cuda.synchronize(device)
        dist.barrier(device_ids=[device.index])
        comm.grad_step_(flat, opt)
        torch.cuda.synchronize(device)
        g = gs[0].clone()
        for r in range(1, world):
            g += gs[r]
        g /= world
        lr_t = opt.lr * (1 - opt.beta2) ** 0.5 / (1 - opt.beta1)
        m1, v1 = (1 - opt.beta1) * g, (1 - opt.beta2) * g * g
        exp = w0 - lr_t * m1 / (v1.sqrt() + opt.eps)
        err = float((flat.data - exp).abs().max())
        t = torch.tensor([err], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["fused_adam_max_abs_err"] = float(t.item())
        out["fused_adam_ok"] = bool(t.item() < 1e-5)
    return out


def main():
    args = parse()
    if args.config == 4:
        args.hidden_units, args.in_features, args.seq_len, args.batch_size = "2048,2048,2048,2048", 2048, 512, 64
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    rank, world, local = dist_env()
    if world != args.gpus and rank == 0 and world > 1:
        sys.stderr.write(f"[bench] WORLD_SIZE={world} != --gpus {args.gpus}; using WORLD_SIZE\n")
    n_gpus = world
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29512")

    B, T, D = args.batch_size, args.seq_len, args.in_features
    C = MODEL["num_classes"]
    hidden = [int(h) for h in args.hidden_units.split(",")]
    sync_label = ("per-step gradient allreduce" if args.config == 3 else "per-epoch parameter average") if n_gpus > 1 else "none"
    extra_out = {}

    if args.impl == "baseline":
        variant = args.baseline_variant
        res = run_baseline_arm(torch, dist, args, hidden, D, C, B, T, rank, world, device, local, variant)
        ms, clk, e2e, launches, cfg_extra = res["ms_per_step"] * args.steps, res["clocks"], res["e2e"], 0, res["config"]
        model_name = f"cudnn-lstm-{len(hidden)}x{hidden[0]}"
        par = f"dp{n_gpus}-nccl"
        sync_label = "per-step gradient allreduce (DDP)" if n_gpus > 1 else "none"
    else:
        from lstm_tensorspark_b200.config import Config
        from lstm_tensorspark_b200.engine import TrainEngine
        from lstm_tensorspark_b200.parallel.comm import make_communicator
        from lstm_tensorspark_b200 import data as Dm
        from lstm_tensorspark_b200.ops import cuda_lstm
        comm_kind = args.comm if args.comm != "auto" else "fused"
        cfg = Config(hidden_units=args.hidden_units, in_features=D, seq_len=T, batch_size=B, num_classes=C,
                     partitions=world, sync_mode="grad_allreduce" if args.config == 3 else "param_avg",
                     sync_every=0 if args.config == 3 else args.steps, average_scope="all", optimizer=args.optimizer, init="scaled",
                     learn_initial_state=False, comm=comm_kind, dtype="bf16", device="cuda", learning_rate=1e-3, quiet=True,
                     grad_buckets=bool(args.grad_buckets))
        comm = make_communicator(comm_kind if world > 1 else "auto", rank, world, device)
        eng = TrainEngine(cfg, rank, world, comm, batch_size=B, device=device, dtype=torch.bfloat16)
        # synthetic shard: 4 distinct device-resident batches (inputs >> L2 together with the activations)
        nb = 4
        xs, ys = Dm.synthetic_sequences(nb * B, T, D, C, seed=1234 + rank)
        dev_x = torch.as_tensor(xs).to(device=device, dtype=torch.bfloat16)
        dev_y = torch.as_tensor(ys).to(device)
        it = {"i": 0}

        def step_dev():
            i = it["i"] % nb
            it["i"] += 1
            loss = eng.step(dev_x[i * B:(i + 1) * B], dev_y[i * B:(i + 1) * B])
            eng.maybe_average()                       # config 4: the per-epoch parameter average (every `steps` steps)
            return loss

        loader = Dm.PinnedHostLoader(xs, ys, B, device, dtype=torch.bfloat16, shuffle=False, seed=rank, depth=args.e2e_depth)
        e2e_dbg = os.environ.get("LSTM_TS_E2E_DEBUG", "")              # diagnostics: "nocopy" (no H2D DMA), "lagN" (read the loss N steps late)
        loader.debug_skip_copy = "nocopy" in e2e_dbg
        lag = int(e2e_dbg.split("lag")[1][0]) if "lag" in e2e_dbg else 1
        nslot = lag + 1
        loss_host = torch.empty(nslot, dtype=torch.float32, pin_memory=True)
        loss_evt = [torch.cuda.Event() for _ in range(nslot)]
        e2e_state = {"i": 0, "last": float("nan")}

        def step_e2e():
            # every step: H2D of this step's batch (pinned, double-buffered on a copy stream) and a D2H read of its loss.
            # The read-back is asynchronous (pinned buffer + event) and consumed one step later, so the host is already
            # enqueueing step k+1 while step k runs - a blocking .item() per step would expose ~50 launch latencies.
            i = e2e_state["i"]
            x, y = loader.next()
            loss = eng.step(x, y)
            eng.maybe_average()
            loss_host[i % nslot].copy_(loss.float(), non_blocking=True)
            loss_evt[i % nslot].record()
            if i >= lag:
                loss_evt[(i - lag) % nslot].synchronize()
                e2e_state["last"] = float(loss_host[(i - lag) % nslot])     # the previous step's loss, on the host
            e2e_state["i"] = i + 1
            return loss_host

        from lstm_tensorspark_b200.ops import cuda_ext
        step_dev()
        k0 = cuda_ext.LAUNCHES["n"]
        step_dev()
        torch.cuda.synchronize(device)
        launches = cuda_ext.LAUNCHES["n"] - k0          # our kernels per step (counted at the binding layer, eager step)
        graphed, graph_err = False, None
        want_graph = args.cuda_graph != 0           # default: capture the whole step (fwd + bwd + fused allreduce/update) once, replay it
        if want_graph:
            try:
                # graphs captured directly on the buffers the batches arrive in (the 4 device batches of the device-timed loop,
                # the loader's 2 staging slots of the end-to-end loop): no 67 MB staging copy per step.  Config 4: 10 GB of
                # activations per graph and a 50 ms step - not worth seven graphs.
                bind = ([(dev_x[i * B:(i + 1) * B], dev_y[i * B:(i + 1) * B]) for i in range(nb)] + list(loader.dev)) \
                    if (args.bind_inputs and args.config == 3) else []
                try:
                    eng.capture(dev_x[:B], dev_y[:B], bind=bind)
                except Exception as e:                  # noqa: BLE001  (e.g. out of memory for seven graphs): one staged graph
                    if not bind:
                        raise
                    graph_err = "bound capture failed, staged graph instead: " + repr(e)[:160]
                    eng._graph, eng._bound = None, {}
                    torch.cuda.synchronize(device)
                    eng.capture(dev_x[:B], dev_y[:B])
                graphed = True
            except Exception as e:                      # noqa: BLE001
                graph_err = repr(e)[:200]
                eng._graph, eng._bound = None, {}
                torch.cuda.synchronize(device)
        h2d, d2h = loader.bytes_per_batch, 4

        def write_outputs(loss):
            # what a caller of the step receives (its loss) and the variables it leaves behind, as a checkpoint names them
            arrays = {"loss": loss.float().cpu().numpy()}
            arrays.update((k, v.float().numpy()) for k, v in eng.model.reference_state_dict().items())
            dump_outputs(args.dump_outputs, arrays)

        ms, clk, e2e = measure(torch, dist, world, device, local, step_dev, step_e2e, args.steps, args.warmup, args.no_e2e, B, n_gpus, h2d, d2h,
                               after_timed=write_outputs if (args.dump_outputs and rank == 0) else None)
        cuda_lstm.check_kernel_errors(device)
        if hasattr(comm, "check_errors"):
            comm.check_errors()
        cfg_extra = {"comm": comm.name, "fast_path": cuda_lstm.STATS["fast_fwd"] > 0, "cuda_graph": graphed, "optimizer": args.optimizer,
                     "graph_inputs": "bound (one graph per input buffer, no staging copy)" if (graphed and eng._bound) else "staged",
                     "e2e_loader_depth": args.e2e_depth,
                     "grad_buckets": bool(eng._bucket_plan)}
        if graph_err:
            cfg_extra["cuda_graph_error"] = graph_err
        model_name = f"lstm-{len(hidden)}x{hidden[0]}"
        par = f"dp{n_gpus}" + ("" if world == 1 else f"-{comm.name}")
        if world > 1 and comm.name == "fused" and args.config == 3:
            eng._graph = None
            extra_out["multi_gpu_check"] = verify_fused_step(torch, dist, eng, comm, world, rank, device)

    value = B * n_gpus * args.steps / (ms / 1e3)
    out = {"metric": "samples/sec", "value": value, "unit": "samples/s", "n_gpus": n_gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "impl": args.impl,
           "config": {"model": model_name, "global_batch": B * n_gpus, "per_gpu_batch": B, "seq_len": T, "in_features": D,
                      "num_classes": C, "parallelism": par, "sync": sync_label,
                      "l2": "per-step working set (activations+inputs, >1 GB) exceeds the 126 MB L2; 4 rotating input batches",
                      **cfg_extra},
           "clocks": clk, "gpu_launches": launches * args.steps}
    if e2e is not None:
        out["e2e"] = e2e
    out.update(extra_out)

    if args.impl == "ours" and not args.no_baseline:
        # The reference itself cannot run here (BASELINE.md §2), so the only same-box anchor is the stand-in for "the reference's
        # NCCL(+cuBLAS) build": cuDNN nn.LSTM + NCCL DDP + fused Adam (baseline/harness.py, library parts only).  Timed HERE, in
        # the same process / box / N / steps / warm-up, with its own clock record; the better of the stock and the tuned variant is
        # the bar.  (BASELINE.md publishes no number, so there is nothing else to divide by.)
        del eng, dev_x, dev_y, loader
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        arms = {}
        for variant in ("stock", "tuned"):
            try:
                arms[variant] = run_baseline_arm(torch, dist, args, hidden, D, C, B, T, rank, world, device, local, variant)
            except Exception as e:                      # noqa: BLE001
                arms[variant] = {"error": repr(e)[:300]}
                torch.cuda.synchronize(device)
        ok = {k: v for k, v in arms.items() if "value" in v}
        if ok:
            best = max(ok, key=lambda k: ok[k]["value"])
            bv = ok[best]
            out["vs_baseline"] = value / bv["value"]
            detail = {"what": "cuDNN nn.LSTM + NCCL DDP + fused Adam stand-in (baseline/harness.py), same process/box/N/steps/warm-up; "
                              "the reference (Py2/TF1/PySpark) cannot run and publishes no number",
                      "ratio": value / bv["value"], "baseline_variant": best, "baseline_value": bv["value"],
                      "baseline_ms_per_step": bv["ms_per_step"], "baseline_clocks": bv["clocks"],
                      "variants": {k: ({"value": v["value"], "ms_per_step": v["ms_per_step"], "clocks": v["clocks"], "config": v["config"],
                                        "e2e_value": (v["e2e"] or {}).get("value")} if "value" in v else v) for k, v in arms.items()}}
            if e2e is not None and bv.get("e2e"):
                be = max((v["e2e"]["value"] for v in ok.values() if v.get("e2e")), default=None)
                if be:
                    detail["e2e_ratio"] = e2e["value"] / be
                    detail["baseline_e2e_value"] = be
            out["vs_baseline_detail"] = detail
        else:
            out["vs_baseline_detail"] = {"error": arms}

    if rank == 0:
        print(json.dumps(out))
    if world > 1 and dist.is_initialized():
        try:
            dist.destroy_process_group()
        except Exception:
            pass
    return 0


if __name__ == "__main__":
    sys.exit(main())
