#!/usr/bin/env python
"""bench.py — waveforms/s of the seist_m_dpk training step (fwd + BCE + bwd + Adam) on (B,3,8192)
synthetic seismograms; see DESIGN.md §5 for what each JSON key means.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "waveforms/sec (B,3,8192) seist_m_dpk fwd+bwd"
UNIT = "waveforms/s"


def synthetic(n, length, seed, head="dpk"):
    """SURVEY §8d: i.i.d. N(0,1) per-trace standardised waveforms; Gaussian-bump P/S labels + detection box."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 3, length, generator=g)
    x = (x - x.mean(-1, keepdim=True)) / x.std(-1, keepdim=True)
    if head != "dpk":
        return x, torch.rand(n, 1, generator=g) * 8.0
    t = torch.arange(length, dtype=torch.float32)[None, :]
    p = torch.randint(length // 8, length // 2, (n, 1), generator=g).float()
    s = p + torch.randint(length // 32, length // 4, (n, 1), generator=g).float()
    tgt = torch.zeros(n, 3, length)
    tgt[:, 1] = torch.exp(-((t - p) ** 2) / 200.0)
    tgt[:, 2] = torch.exp(-((t - s) ** 2) / 200.0)
    tgt[:, 0] = ((t >= p) & (t <= s + 2 * (s - p))).float()
    return x.contiguous(), tgt.contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def summary(self, t0, t1):
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 and len(r) >= 8] or [r for _, r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = []
        for i, nm in ((4, "hw_slowdown"), (5, "hw_thermal_slowdown"), (6, "sw_thermal_slowdown"), (7, "sw_power_cap")):
            if any(r[i].lower().startswith("active") for r in rows):
                reasons.append(nm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


def reference_step_rate(model_name, batch, length, steps, warmup, threads, device="cpu"):
    """The reference's training step (training/train.py:87-111: forward, BCELoss / HuberLoss, zero_grad, backward,
    Adam.step) timed on `device`.  kind "reference": the UNMODIFIED reference modules staged by oracle/build_ref.py
    (models/seist.py + models/loss.py, default drop rates, torch's own kernels); kind "port": the pinned oracle
    restatement (dropout identity) when the staged copy is absent.  Returns (waveforms/s, seconds, kind)."""
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    from oracle import build_ref
    dev = torch.device(device)
    head = "dpk" if model_name.endswith("dpk") else "reg"
    x, tgt = synthetic(batch, length, 99, head)
    x, tgt = x.to(dev), tgt.to(dev)

    def sync():
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)

    if build_ref.available():
        M = build_ref.import_models()
        model = M.create_model(model_name, in_channels=3, in_samples=length).to(dev).train()
        loss_fn = (M.BCELoss(weight=[[0.5], [1], [1]]) if head == "dpk" else M.HuberLoss()).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=8e-5)
        kind = "reference"

        def step():
            out = model(x)
            loss = loss_fn(out, tgt)
            opt.zero_grad()
            loss.backward()
            opt.step()
    else:
        from oracle import seist_ref as R
        from seist_b200.models import create_model
        m = create_model(model_name, in_channels=3, in_samples=length)
        sd = {k: (v.detach().clone().to(dev).requires_grad_(True) if v.dtype.is_floating_point and "running" not in k
                  else v.detach().clone().to(dev)) for k, v in m.state_dict().items()}
        opt = torch.optim.Adam([v for v in sd.values() if v.requires_grad], lr=8e-5)
        spec = R.spec_for(model_name)
        kind = "port"

        def step():
            y, bufs = R.forward(sd, x, spec, training=True)
            loss = R.bce_loss(y, tgt) if spec.head == "dpk" else R.huber_loss(y, tgt)
            opt.zero_grad()
            loss.backward()
            opt.step()
            for k, b in bufs.items():
                sd[k] = b
    times = []
    for i in range(warmup + steps):
        sync()
        t0 = time.perf_counter()
        step()
        sync()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return batch * len(times) / sum(times), sum(times), kind


DUMP_BYTES = 60 << 20      # bound on the arrays of one --dump-outputs directory (under 64 MB with the file headers)
DUMP_ROWS = 64             # waveforms of the predictions kept in a dump, a fixed seeded sample of the batch


def dump_outputs(out_dir, trainer):
    """Writes what the last Trainer.step() computed, as its caller sees it, to out_dir/<name>.npy (float32): the loss,
    the model's predictions (rows listed in prediction_rows.npy), the parameter gradients, and the parameters and
    BatchNorm running statistics after the Adam update.  Two builds run with the same arguments can be compared
    array by array."""
    import numpy as np
    y = trainer.plan.y_out.x
    arrays = {"loss": trainer.loss_out, "gradients": trainer.last_grads, "parameters": trainer.flat.P,
              "bn_running_stats": trainer.flat.RB}
    row_bytes = y[0].numel() * 4
    budget = DUMP_BYTES - sum(t.numel() * 4 for t in arrays.values())
    n = min(y.shape[0], DUMP_ROWS, budget // row_bytes)
    if n < 1:
        raise ValueError(f"--dump-outputs: the outputs of one step exceed {DUMP_BYTES >> 20} MB")
    rows = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:n].sort().values
    arrays["predictions"] = y[rows.to(y.device)]
    arrays["prediction_rows"] = rows
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to("cpu", torch.float32).numpy())


def _kind_text(kind):
    return ("unmodified reference modules staged in oracle/_ref, default drop rates" if kind == "reference"
            else "oracle port of the reference step, dropout identity")


def main():
    # stdout carries exactly ONE JSON line: everything else (NCCL banner, library prints) goes to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--model", default="seist_m_dpk")
    ap.add_argument("--batch", type=int, default=512, help="waveforms per GPU")
    ap.add_argument("--length", type=int, default=8192)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--op-times", default="", help="write the per-op device-time table (JSON) here")
    ap.add_argument("--cpu-batch", type=int, default=32)
    ap.add_argument("--cpu-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = min(os.cpu_count() or 1, 32)      # host threads used by the CPU arm (torch intra-op pool)
    workload = f"{args.model} train step (fwd+BCE+bwd+Adam), batch {args.batch}/GPU x (3,{args.length}) fp32"
    config = {"workload": workload, "model": args.model, "per_gpu_batch": args.batch, "in_samples": args.length,
              "global_batch": args.batch * max(args.gpus, 1), "parallelism": f"dp{max(args.gpus, 1)}",
              "l2": "per-step working set (GBs of activations) far exceeds the 126 MB L2; no explicit flush",
              "dropout": "reference default rates, counter-based RNG"}

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps                       # ~0.5 s per 32-waveform CPU step
        warm = max(1, min(args.warmup, 2))
        rate, secs, kind = reference_step_rate(args.model, args.cpu_batch, args.length, steps, warm, cores)
        config["cpu_sample_batch"] = args.cpu_batch
        config["workload"] += f"; this arm: the reference's CPU step on {cores} host threads, bounded sample of {args.cpu_batch} waveforms/step"
        line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": 1e3 * secs / steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
                                 "sample": f"{steps} train steps of {args.cpu_batch} waveforms ({_kind_text(kind)})"},
                "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch.distributed as dist
    from seist_b200 import _lib
    from seist_b200.models import create_model
    from seist_b200.roofline import STEP_BYTES_PER_WAVEFORM, time_ops
    from seist_b200.train import Trainer, cyclic_lr

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    torch.manual_seed(0)
    model = create_model(args.model, in_channels=3, in_samples=args.length).to(dev)
    if world > 1:      # reference training/train.py:374
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
    head = model.hp.head
    x_h, t_h = synthetic(args.batch, args.length, 1234 + rank, head)
    x_h, t_h = x_h.pin_memory(), t_h.pin_memory()
    x_d, t_d = x_h.to(dev), t_h.to(dev)
    trainer = Trainer(model, lr_schedule=lambda it: cyclic_lr(it), use_graph=not args.no_graph)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident inputs ------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        trainer.step(x_d, t_d)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    profiling = os.environ.get("SEIST_PROFILE") == "1"     # ncu --profile-from-start off: capture the timed steps only
    if profiling:
        torch.cuda.profiler.start()
    t0 = time.time()
    ms = timed(lambda: trainer.step(x_d, t_d), args.steps)
    t1 = time.time()
    if profiling:
        torch.cuda.profiler.stop()
    clocks = sampler.summary(t0, t1) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer)
    loss_val = float(trainer.loss_out.item())
    value = args.batch * world * args.steps / (ms / 1e3)

    # ---- end to end: pinned host inputs in, loss out, every step ----------------------------------
    loss_host = torch.zeros((), pin_memory=True)

    # every step: one pinned-host -> device copy of a full batch (issued on the trainer's copy stream right after
    # the step that consumes the previous one was launched, so it overlaps that step - the job of a data loader's
    # prefetcher) and one device -> host read of the step's loss, waited for before the next step starts
    def e2e_step():
        loss = trainer.step()                      # consumes the staged batch
        trainer.prefetch(x_h, t_h)                 # H2D of the next batch, overlapping the step just launched
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    trainer.prefetch(x_h, t_h)
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e_value = args.batch * world * args.steps / (ms_e2e / 1e3)

    arena_gb = trainer.plan.arena_bytes / 1e9
    launches_per_step, used_graph = trainer.launches_per_step, trainer.graph is not None
    # ---- dominant kernel roofline (rank 0) ---------------------------------------------------------
    roofline, step_roofline, cpu_baseline, reference_gpu = None, None, None, None
    if rank == 0:
        rows = time_ops(trainer.plan, reps=2)
        tot = sum(r["ms"] for r in rows)
        rows.sort(key=lambda r: -r["ms"])
        # the dominant kernel FAMILY of the step: ops aggregated by (op kind, kernel template family), measured live
        # (every op launched alone, CUDA events on the launching stream, L2-evicting write in between)
        fams = {}
        for r in rows:
            f = fams.setdefault(r.get("family", str(r["kind"])), {"ms": 0.0, "bytes": 0, "flops": 0.0, "ops": 0})
            f["ms"] += r["ms"]; f["bytes"] += r["bytes"]; f["flops"] += r.get("flops", 0.0); f["ops"] += 1
        fam_name, fam = max(fams.items(), key=lambda kv: kv[1]["ms"])
        ach = fam["bytes"] / (fam["ms"] * 1e-3) / 1e9
        top = max((r for r in rows if r.get("family", str(r["kind"])) == fam_name), key=lambda r: r["ms"])
        # DRAM traffic of the family's largest op from the committed `ncu --set full` capture (profiles/dram_traffic.json:
        # dram__bytes_read.sum + dram__bytes_write.sum per launch at this batch size), null if not captured
        traffic = None
        try:
            cap = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
            ent = cap.get("ops", {}).get(top["name"])
            if ent and cap.get("model") == args.model and cap.get("batch") == args.batch:
                traffic = ent["dram_bytes"]
        except Exception:
            pass
        tensor_pct = None
        try:
            tp = json.load(open(os.path.join(ROOT, "profiles", "tensor_pipe.json")))
            tensor_pct = tp.get("families", {}).get(fam_name)
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": fam_name, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": traffic, "traffic_op": top["name"], "ms": fam["ms"],
                    "algorithmic_bytes": fam["bytes"], "ops": fam["ops"], "share_of_step": fam["ms"] / tot,
                    "tflops": fam["flops"] / (fam["ms"] * 1e-3) / 1e12, "tensor_pipe_pct": tensor_pct,
                    "peak_source": peak_src,
                    "families": {k: {"ms": round(v["ms"], 3), "share": round(v["ms"] / tot, 4),
                                     "GBps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1), "ops": v["ops"]}
                                 for k, v in sorted(fams.items(), key=lambda kv: -kv[1]["ms"])}}
        if args.op_times:
            os.makedirs(os.path.dirname(os.path.abspath(args.op_times)), exist_ok=True)
            json.dump({"total_ms_isolated": tot, "step_ms": ms / args.steps, "rows": rows}, open(args.op_times, "w"))
        bpw = STEP_BYTES_PER_WAVEFORM.get(args.model)
        if bpw and args.length == 8192:
            a = value / world * bpw / 1e9
            step_roofline = {"bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak,
                             "bytes_per_waveform": bpw, "model": "6 accesses per BN-input element + I/O (SURVEY 8d)"}
        if world == 1 and not args.no_cpu_baseline:
            rate, secs, kind = reference_step_rate(args.model, args.cpu_batch, args.length, args.cpu_steps, 1, cores)
            cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
                            "sample": f"{args.cpu_steps} train steps of {args.cpu_batch} waveforms "
                                      f"({secs:.1f} s; {_kind_text(kind)})"}
            # informational, same box: the reference's modules under stock PyTorch eager on this B200 (SURVEY 8d)
            try:
                del trainer
                torch.cuda.empty_cache()
                gb = min(args.batch, 128)
                grate, gsecs, gkind = reference_step_rate(args.model, gb, args.length, 6, 3, cores, device=f"cuda:{local_rank}")
                reference_gpu = {"value": grate, "unit": UNIT, "kind": gkind, "batch": gb,
                                 "how": "stock PyTorch eager (cuDNN/cuBLAS, TF32 convs allowed as by default), fp32, "
                                        "same train step, 6 timed steps after 3 warm-up"}
            except Exception as e:      # noqa: BLE001
                reference_gpu = {"unavailable": repr(e)[:200]}
    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": (x_h.numel() + t_h.numel()) * 4, "d2h_bytes_per_step": 4,
                        "d2h": "the step's loss only; the model outputs stay on the device (the reference's train() copies "
                               "them to the host every step for its CPU metrics, training/train.py:141 - out of this path)",
                        "h2d": "pinned host batch copied every step on a copy stream, one step ahead (Trainer.prefetch)"},
                "gpu_launches": launches_per_step * args.steps,
                "launches_per_step": launches_per_step, "cuda_graph": used_graph,
                "loss": loss_val, "clocks": clocks, "roofline": roofline, "step_roofline": step_roofline,
                "cpu_baseline": cpu_baseline, "reference_gpu_eager": reference_gpu, "arena_gb": arena_gb}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
