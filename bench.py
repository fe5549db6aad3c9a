#!/usr/bin/env python
"""bench.py — train_step throughput of the data-parallel hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this backend (libedb.so kernels)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)

Workload (config.workload): GPT-2 medium (L24 H1024 16 heads), bf16 params/activations, 512-token
synthetic sequences, 8 sequences per GPU (weak scaling), SGD(momentum 0.9, foreach) — BASELINE.json
configs[1] ("GPT-2 medium auto-SPMD, bf16, synthetic 512-seq batches").  One step = forward +
backward + optimizer update of one global batch through `easydist_compile`'s compiled graph.

Printed keys (one JSON line from rank 0): see the bench contract in the task statement;
`value` = samples/s with inputs resident in HBM, `e2e` = the same through the public API with
pinned-host inputs copied H2D and the loss read back D2H every step, `roofline` = the dominant
kernel (tcgen05 GEMM) against the measured bf16 peak, `cpu_baseline` = the oracle port on the
host cores (bounded sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="edb", choices=["edb", "reference", "torch-nccl"],
                    help="edb: this backend; reference: the reference's CPU path (oracle port); "
                         "torch-nccl: stock eager PyTorch + DDP/NCCL + cuBLAS on the same GPUs (what "
                         "the reference's lowering runs on: SURVEY.md 8(d) 'the real competitor')")
    ap.add_argument("--model", default="gpt2-medium")
    ap.add_argument("--mode", default="zero3", choices=["ddp", "zero2", "zero3", "auto"],
                    help="auto: BASELINE.json config 1 (the reference's GPT example, fp32) in auto-SPMD "
                         "mode with the plan the reference's solver recorded for this mesh "
                         "(tools/bench_c1_auto.py; needs 2, 4 or 8 GPUs)")
    ap.add_argument("--batch-per-gpu", type=int, default=8)
    ap.add_argument("--seq", type=int, default=512)
    ap.add_argument("--attn", default="sdpa", choices=["sdpa", "unfused"])
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-fuse", action="store_true",
                    help="keep all-gather / reduce-scatter as separate kernels (no AG+GEMM, GEMM+RS)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-seqs", type=int, default=2)
    ap.add_argument("--heap-gb", type=float, default=12.0)
    ap.add_argument("--no-roofline", action="store_true",
                    help="skip the GEMM launch-list replay (multi-billion-parameter models: the replay "
                         "allocates fresh operands for every launch)")
    ap.add_argument("--no-parity", action="store_true",
                    help="skip the pre-timing parity leg (compiled N-GPU steps vs vanilla fp32)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                         "(its loss; the parameters and momentum buffers it left, sampled), so that "
                         "two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "edb" or args.mode == "auto"):
        ap.error("--dump-outputs covers this backend's data-parallel path (--impl edb, --mode "
                 "ddp / zero2 / zero3)")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "hbm_gbs": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe's clocks line)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names)
                   if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---- the reference arm / cpu baseline: oracle port on host cores ------------------------------------


def cpu_train_step_throughput(args, n_seqs, steps=1, warmup=0):
    """The reference's path on CPU is ATen-CPU compute + gloo collectives driven by the FX graph
    (SURVEY.md §8d).  The oracle port runs the same train step (same model, fp32 on CPU — the
    reference's CPU runs are fp32) on the host cores; at world 1 there is no collective."""
    import torch
    from oracle import train_oracle
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    # eager PyTorch on CPU stops scaling (and oversubscribes cgroup-limited boxes) well before
    # 128 threads: measured 88 s/step with 128 threads vs 4 s with 8 for the same sequence
    cores = max(1, min(avail, int(os.environ.get("EDB_CPU_THREADS", "32"))))
    torch.set_num_threads(cores)
    t, loss = train_oracle.time_cpu_train_step(args.model, args.attn, n_seqs, args.seq, steps,
                                               warmup=warmup)
    return {"value": n_seqs * steps / t, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": f"{steps} timed step(s) (+{warmup} warm-up) of {n_seqs} x {args.seq}-token "
                      f"sequences each (bounded sample of the {args.batch_per_gpu}-sequence "
                      f"per-GPU batch), fp32, torch CPU eager, single process ({cores} threads), "
                      f"{t:.1f} s", "loss": loss, "seconds": t}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # exactly --warmup untimed and --steps timed steps, each a bounded sample (--cpu-sample-seqs
    # sequences) of the per-GPU batch: ~2 s per step on 32 threads, so the default 20 + 5 steps end
    # within about a minute.  At N > 1 this is still ONE process on rank 0's host cores (the
    # reference itself cannot travel to the GPU box; DESIGN.md §4).
    base = cpu_train_step_throughput(args, args.cpu_sample_seqs, steps=max(1, args.steps),
                                     warmup=max(0, args.warmup))
    line = {
        "impl": "reference", "metric": "train_step_throughput", "value": base["value"],
        "unit": "samples/s", "n_gpus": args.gpus, "steps": max(1, args.steps),
        "warmup": max(0, args.warmup),
        "ms_per_step": 1e3 * base["seconds"] / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"{args.model} train_step (fwd+bwd+SGD-momentum), bf16, seq {args.seq}, "
                        f"{args.batch_per_gpu} seq/GPU",
            "global_batch": args.batch_per_gpu * world, "seq_len": args.seq,
            "parallelism": f"{args.mode} dp{world}", "attention": args.attn,
            "l2_policy": "per-step working set (weights+activations > 2 GB) exceeds the 126 MB L2",
            "cuda_graph": not args.no_cuda_graph}


# ---- this backend -----------------------------------------------------------------------------------------


def gemm_roofline(torch, gemm, calls, peaks, sustained, fused_calls=(), rank=0, pf_map=None):
    """Dominant kernel = the tcgen05 GEMM.  Replays the step's GEMM launches (exact shapes, operand
    layouts and strides recorded from the compiled graph) back to back from a CUDA graph with CUDA
    events around the whole list on the launching stream; operands of consecutive launches differ
    and sum to far more than L2.  achieved = algorithmic FLOPs (2*M*N*K per launch) / measured time."""
    if not calls and not fused_calls:
        return None
    ops = []
    flops = 0
    for (M, N, K, a_k, b_k, a_stride, b_stride) in calls:
        # same extents AND strides as in the step (e.g. the LM-head gradient arrives with a padded,
        # TMA-legal row stride from the cross-entropy kernel; an unaligned one is staged by gemm.mm)
        a = torch.empty_strided((M, K), a_stride, device="cuda", dtype=torch.bfloat16).normal_()
        b = torch.empty_strided((K, N), b_stride, device="cuda", dtype=torch.bfloat16).normal_()
        ops.append((a, b))
        flops += 2 * M * N * K
    # the fused collective GEMMs of the step (N > 1): the REAL kernels, replayed with their real
    # symmetric buffers on every rank at once — epoch-mode AG+GEMM pulls the peers' (static) weight
    # shards, the push GEMM stores into the peers' receive slots (scratch between steps), neither
    # needs a handshake, so the replay carries the step's NVLink traffic
    from easydist_b200 import reshard, runtime as _rtm
    from easydist_b200.runtime import SymmBuffer
    fused_ops = []
    for c in fused_calls:
        M, N, K = c["M"], c["N"], c["K"]
        if c["kind"] == "ag":
            x = torch.empty_strided((M, K), c["a_stride"], device="cuda", dtype=torch.bfloat16).normal_()
            n = len(c["group"])
            w = SymmBuffer(_rtm.get_runtime(), c["buf"][0], N // n * K * 2).tensor(torch.bfloat16, (N // n, K))
            fused_ops.append(("ag", x, w, c))
        else:
            a = torch.empty_strided((M, K), c["a_stride"], device="cuda", dtype=torch.bfloat16).normal_()
            b = torch.empty_strided((K, N), c["b_stride"], device="cuda", dtype=torch.bfloat16).normal_()
            fused_ops.append(("push", a, b, c))
        flops += 2 * M * N * K

    def run_fused():
        for kind, u, v, c in fused_ops:
            if kind == "ag":
                reshard.ag_mm(u, v, c["group"], c["N"], c["K"], None, _buf=c["buf"], _epoch=1)
            else:
                reshard.mm_push(u, v, c["group"], _buf=c["buf"])

    pf_map = pf_map or {}

    def run_plain(mm):
        for i, (a, b) in enumerate(ops):
            if mm is gemm.mm and i in pf_map:
                gemm.mm(a, b, _pf=pf_map[i])  # with its all-gather prefetch passengers
            else:
                mm(a, b)

    run_plain(gemm.mm)
    run_fused()
    torch.cuda.synchronize()
    # replayed from a CUDA graph like the step itself: eager launches of 30-us kernels would measure
    # the host (ctypes + tensor-map encode per call), not the kernel
    def graph_ms(mm, reps=3):
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                run_plain(mm)
                if mm is gemm.mm:
                    run_fused()
            graph.replay()
            side.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(reps):
                graph.replay()
            e1.record(side)
            side.synchronize()
        torch.cuda.current_stream().wait_stream(side)
        del graph
        return e0.elapsed_time(e1) / reps

    ms = graph_ms(gemm.mm)
    achieved = flops / ms / 1e9  # TFLOP/s
    n_launch = len(calls) + len(fused_ops)
    # context only: what cuBLAS reaches on the plain GEMMs of the list (same operands, same graph
    # replay); shapes cuBLAS cannot align (LM head, vocab 50257) hit its sm_75-class `align1` kernels
    cublas_tf = None
    if ops and not fused_ops and not pf_map:
        for a, b in ops:
            torch.mm(a, b)
        torch.cuda.synchronize()
        cublas_tf = flops / graph_ms(torch.mm) / 1e9
    # the replay is a ~10-20 ms burst timed on its own, so the burst peak is the denominator
    # (the sustained figure is reported beside it)
    peak = peaks["bf16_tflops_sustained"] if sustained else peaks["bf16_tflops"]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_gemm_dram_traffic.json")
    if os.path.exists(tpath) and not fused_ops and not pf_map:
        with open(tpath) as f:
            traffic = json.load(f)
    return {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"],
            "traffic": (traffic or {}).get("dram_bytes_per_launch"),
            "traffic_algorithmic_bytes_per_launch": (traffic or {}).get("algorithmic_bytes_per_launch"),
            "traffic_source": (traffic or {}).get("source"),
            "kernel": "edb::k_gemm_bf16 (plain" + (", with all-gather prefetch CTAs" if pf_map else "")
                      + (", push-fused" if fused_ops else "") + ")",
            "launches_per_step": n_launch, "fused_launches_per_step": len(fused_ops),
            "prefetch_carrying_launches_per_step": len(pf_map),
            "avg_launch_us": 1e3 * ms / n_launch,
            "gemm_ms_per_step": ms, "flops_per_step": flops,
            "cublas_same_launch_list_tflops": cublas_tf,
            "peak_source": peaks["source"] + (", sustained figure" if sustained else
                                              ", burst figure (the launch list is replayed on its own)")}


def parity_leg(torch, dist, args, cfg, GPT2, step_fn, model, opt, state0, par_host, first_loss,
               rank, world):
    """Pre-timing parity (outside every timed region): the compiled N-GPU train step against
    vanilla fp32 PyTorch on the same global batches — loss of every step, EVERY parameter and
    EVERY momentum buffer (the reference's comparator, tests/test_torch/test_spmd.py:97-113).
    The first compiled call already ran the first batch twice (eager warm-up + first CUDA-graph
    replay, the same as the reference's wrapper, api.py:183-222), so the vanilla run does too."""
    from tools import parity as P
    B, S = args.batch_per_gpu, args.seq
    n_par = len(par_host)
    losses = [first_loss]
    for b in range(1, n_par):
        t, y = par_host[b][rank]
        losses.append(float(step_fn(t.cuda(), y.cuda(), model, opt)))
    torch.cuda.synchronize()
    graph_on = not args.no_cuda_graph
    sched = ([0, 0] if graph_on else [0]) + list(range(1, n_par))
    steps = [par_host[b] for b in sched]
    mk_opt = lambda ps: torch.optim.SGD(ps, lr=1e-3, momentum=0.9, foreach=True)
    ref_losses, ref_p, ref_s = P.vanilla_run(lambda: GPT2(cfg), state0, steps, mk_opt,
                                             torch.float32, "cuda")
    van_losses, van_p, van_s = P.vanilla_run(lambda: GPT2(cfg), state0, steps, mk_opt,
                                             torch.bfloat16, "cuda")
    got_p, got_s = P.compiled_state(step_fn.compiled_func, ref_p, ref_s, world)
    ours = P.compare(got_p, got_s, ref_p, ref_s, low_precision=True)
    van = P.compare({k: v.to(torch.bfloat16) for k, v in van_p.items()},
                    {k: {kk: vv.to(torch.bfloat16) for kk, vv in st.items()} for k, st in van_s.items()},
                    ref_p, ref_s, low_precision=True)
    # our losses are the local (per-rank) means of each call; with a CUDA graph the first call
    # returns the loss of its replay = the second vanilla step on batch 0
    idx = [1 if graph_on else 0] + list(range(2 if graph_on else 1, len(sched)))
    loss_rel = max(abs(l - ref_losses[i][rank]) / abs(ref_losses[i][rank])
                   for l, i in zip(losses, idx))
    van_loss_rel = max(abs(van_losses[i][rank] - ref_losses[i][rank]) / abs(ref_losses[i][rank])
                       for i in idx)
    tol_state = max(2e-2, 2.0 * van["state_rel_l2"])
    tol_ulp = max(2.0, 2.0 * van["param_max_ulp"])
    ok = loss_rel <= 2e-2 and ours["state_rel_l2"] <= tol_state and ours["param_max_ulp"] <= tol_ulp
    res = {"ok": bool(ok), "checks": ours["checks"] + len(losses),
           "max_rel_err": max(ours["state_rel_l2"], loss_rel),
           "loss_rel_err": loss_rel, "momentum_rel_l2": ours["state_rel_l2"],
           "param_max_bf16_ulp": ours["param_max_ulp"], "worst": ours["worst"],
           "vanilla_bf16_vs_fp32": {"loss_rel_err": van_loss_rel, "momentum_rel_l2": van["state_rel_l2"],
                                    "param_max_bf16_ulp": van["param_max_ulp"]},
           "tolerance": {"loss_rel": 2e-2, "momentum_rel_l2": tol_state, "param_bf16_ulp": tol_ulp},
           "what": f"{len(sched)} optimisation steps ({n_par} calls) of the compiled {world}-GPU "
                   f"{args.mode} step vs vanilla fp32 PyTorch on the same global batches: loss per "
                   "call, every parameter, every momentum buffer"}
    if world > 1:
        # the reshard-kernel battery of tests/mgpu_worker.py (every collective / dtype / dim, P2P
        # boxes, the epoch-protocol kernels and the all-gather prefetch) bit for bit against the
        # oracle, so that multi-rank kernel parity is part of every N > 1 bench record
        try:
            from tests import mgpu_worker as W
            group = list(range(world))
            stages = [("cases", lambda: W.run_cases(rank, world, group, tag="bench")),
                      ("p2p", lambda: W.run_p2p(rank, world, group)),
                      ("epoch", lambda: W.run_epoch(rank, world, group)),
                      ("prefetch", lambda: W.run_prefetch(rank, world, group)),
                      ("push", lambda: W.run_push_cases(rank, world, group, passes=2, big=False))]
            # wall-clock bound on this pre-timing leg (host-side oracle work grows with N): a stage
            # starts only while every rank is inside the budget (MAX over ranks: one decision for all)
            budget_s = float(os.environ.get("EDB_BENCH_BATTERY_S", "90"))
            t_b, n_resh, skipped = time.time(), 0, []
            for name, stage in stages:
                el = torch.tensor([time.time() - t_b], device="cuda")
                dist.all_reduce(el, op=dist.ReduceOp.MAX)
                if el.item() > budget_s:
                    skipped.append(name)
                    continue
                n_resh += stage()
            res["reshard_checks_bit_exact"] = n_resh
            res["reshard_battery_s"] = time.time() - t_b
            if skipped:
                res["reshard_battery_skipped"] = skipped
            res["checks"] += n_resh
        except AssertionError as e:
            ok = False
            res["ok"] = False
            res["reshard_failure"] = str(e)[:300]
        flags = torch.tensor([0.0 if ok else 1.0, res["max_rel_err"], res["param_max_bf16_ulp"]],
                             device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MAX)
        res["ok"] = bool(flags[0].item() == 0.0)
        res["max_rel_err"] = flags[1].item()
        res["param_max_bf16_ulp"] = flags[2].item()
    return res


def dump_outputs(torch, step_fn, loss, full_shapes, world, rank, out_dir):
    """The last timed step's results as out_dir/<name>.npy: `loss` (float64) and, in float32, every
    parameter (`param.<name>`) and optimizer state (`<key>.<name>`) it left, gathered to full size.
    Tensors above `per` elements are sampled at `per` positions drawn with a fixed seed, which keeps
    the files under 64 MB in all."""
    import numpy as np
    from tools import parity as P
    params, _, states = step_fn.compiled_func.get_state()
    tensors = []
    for name, shape in full_shapes.items():
        tensors.append((f"param.{name}", params[name], shape))
        for key, t in states.get(name, {}).items():
            if isinstance(t, torch.Tensor) and t.dim() > 0:
                tensors.append((f"{key}.{name}", t, shape))
    per = min(16384, (60 << 20) // (4 * len(tensors)))
    arrays = {"loss": np.float64(loss)}
    for fname, t, shape in tensors:
        full = P.gather_full(t.detach(), shape, world).flatten()
        if full.numel() > per:
            idx = np.sort(np.random.default_rng(0).choice(full.numel(), per, replace=False))
            full = full[torch.from_numpy(idx).to(full.device)]
        arrays[fname] = full.float().cpu().numpy()
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)


def run_edb(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from easydist_b200 import gemm, runtime
    from easydist_b200.api import easydist_compile
    from easydist_b200.device_mesh import set_device_mesh
    from easydist_b200.workloads import (GPT2, GPT2_CONFIGS, gpt2_train_step, synthetic_tokens,
                                         train_flops_per_step)
    import dataclasses
    rt = runtime.init(rank, world, local, heap_bytes=int(args.heap_gb * (1 << 30)))
    set_device_mesh(list(range(world)), ["dp"], rank=rank)
    if args.model.startswith("llama"):
        # BASELINE.json config 4: Llama-2 (RMSNorm / rotary / SwiGLU, untied head); "-lN" = N layers
        from easydist_b200.workloads import LLAMA_CONFIGS, Llama
        base, _, nl = args.model.partition("-l")
        cfg = dataclasses.replace(LLAMA_CONFIGS["llama2-7b"], block_size=max(args.seq, 2048),
                                  **({"n_layer": int(nl)} if nl else {}))
        GPT2 = Llama
    else:
        cfg = dataclasses.replace(GPT2_CONFIGS[args.model], attn=args.attn,
                                  block_size=max(args.seq, GPT2_CONFIGS[args.model].block_size))
    torch.manual_seed(0)
    if args.model.startswith("llama"):
        with torch.device("cuda"):  # 7 B fp32 parameters per rank must not be built in host memory
            model = GPT2(cfg)
        model = model.to(torch.bfloat16)
    else:
        model = GPT2(cfg).to(device="cuda", dtype=torch.bfloat16)
    opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, foreach=True)
    full_shapes = {n: p.shape for n, p in model.named_parameters()}
    B, S = args.batch_per_gpu, args.seq
    n_batches = 4
    host = [synthetic_tokens(cfg, B, S, seed=1000 * b + rank) for b in range(n_batches)]
    host = [(t.pin_memory(), y.pin_memory()) for t, y in host]
    dev = [(t.cuda(), y.cuda()) for t, y in host]
    step_fn = easydist_compile(gpt2_train_step, parallel_mode=args.mode, tracing_mode="fake",
                               cuda_graph=not args.no_cuda_graph, fuse=not args.no_fuse)
    state0 = None if args.no_parity else {k: v.detach().clone() for k, v in model.state_dict().items()}
    # parity batches: one per (step, rank); every rank can rebuild all of them for the reference
    n_par = 3
    par_host = [[synthetic_tokens(cfg, B, S, seed=7000 + 1000 * b + r) for r in range(world)]
                for b in range(n_par)]
    first = par_host[0][rank] if not args.no_parity else host[0]
    first = (first[0].cuda(), first[1].cuda())
    launches0 = rt.launch_count()
    gemm.reset_stats()
    t0 = time.time()
    loss = step_fn(first[0], first[1], model, opt)  # compile + eager warm-up (+ graph capture)
    torch.cuda.synchronize()
    compile_s = time.time() - t0
    info = step_fn.compiled_func.info
    # kernels of ours per step: counted on the eager warm-up step (graph replays launch the same)
    stats = gemm.stats()
    passes = 1 if args.no_cuda_graph else 2  # warm-up + capture both go through the host calls
    launches_per_step = (rt.launch_count() - launches0) // passes
    gemm_calls_per_step = stats["edb_gemm"] // passes
    aten_mm_per_step = stats["aten_mm"] // passes
    # the step's GEMM launch list, frozen now (the parity battery below issues GEMMs of its own)
    step_calls = gemm.recorded_calls()[:gemm_calls_per_step]
    fused_all = gemm.recorded_fused_calls()
    step_fused = fused_all[:len(fused_all) // passes]
    step_pf = {i: d for i, d in gemm.recorded_prefetches().items() if i < len(step_calls)}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps, e2e):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        last = None
        for i in range(n_steps):
            if e2e:
                t_h, y_h = host[i % n_batches]
                t_d = t_h.to("cuda", non_blocking=True)
                y_d = y_h.to("cuda", non_blocking=True)
                last = step_fn(t_d, y_d, model, opt)
                last = float(last)  # device -> host read of the step's result
            else:
                t_d, y_d = dev[i % n_batches]
                last = step_fn(t_d, y_d, model, opt)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), float(last)

    parity = None
    if not args.no_parity:
        parity = parity_leg(torch, dist, args, cfg, GPT2, step_fn, model, opt, state0, par_host,
                            float(loss), rank, world)
    # clocks / throttle reasons are sampled from the warm-up steps on (the same workload): the timed
    # region alone lasts only ~0.3 s, one or two nvidia-smi samples
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # its first sample arrives ~0.1 s later: the GPU is already under load
    for _ in range(max(3, args.warmup)):
        step_fn(dev[0][0], dev[0][1], model, opt)
    torch.cuda.synchronize()
    ms_total, loss_v = timed(args.steps, e2e=False)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, loss_last = timed(args.steps, e2e=True)
    errs = rt.error_flags()
    assert not any(errs), f"collective spin-wait timeouts: {errs}"
    if args.dump_outputs:
        dump_outputs(torch, step_fn, loss_last, full_shapes, world, rank, args.dump_outputs)
    gbatch = B * world
    value = gbatch * args.steps / (ms_total / 1e3)
    e2e_value = gbatch * args.steps / (ms_e2e / 1e3)
    ms_per_step = ms_total / args.steps
    peaks = measured_peaks()
    # GEMM shapes of one step, recorded by the dispatcher during the eager warm-up
    calls, fused_calls = step_calls, step_fused
    # every rank replays (the fused kernels talk to the peers); rank 0 reports
    barrier()
    pf_map = step_pf
    roof = None if args.no_roofline else gemm_roofline(torch, gemm, calls, peaks, sustained=False,
                                                       fused_calls=fused_calls, rank=rank, pf_map=pf_map)
    barrier()
    if args.model.startswith("llama"):
        p_mm = sum(p.numel() for n_, p in model.named_parameters() if p.dim() == 2 and "tok" not in n_)
        step_flops = 6 * p_mm * B * S + 12 * cfg.n_layer * cfg.n_embd * S * B * S
    else:
        step_flops = train_flops_per_step(cfg, B, S)
    line = {
        "metric": "train_step_throughput", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(args, world),
        "tokens_per_s": value * S,
        "model_tflops_per_gpu": step_flops / (ms_per_step / 1e3) / 1e12,
        "e2e": {"value": e2e_value, "unit": "samples/s",
                "h2d_bytes_per_step": 2 * B * S * 8, "d2h_bytes_per_step": 2,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
        "dispatch": {"edb_gemm_per_step": gemm_calls_per_step, "aten_mm_per_step": aten_mm_per_step,
                     "comm_nodes": info.get("comm_nodes"), "fused": info.get("fused"),
                     "symm_bytes": info.get("symm_bytes"), "epoch_check": info.get("epoch_check")},
        "clocks": clocks, "loss": loss_v, "compile_s": compile_s,
    }
    if parity is not None:
        line["parity"] = parity
    if world > 1 and not args.no_parity:
        # the other half of BASELINE.json's metric: reshard bus bandwidth (nccl-tests convention)
        # against NVLink-5 peak, 64 MiB bf16, push-protocol kernels vs NCCL on the same GPUs
        # (tests/mgpu_worker.py bench2: CUDA-graph timed, max over ranks; outside the timed region)
        try:
            from tests import mgpu_worker as W
            rows = W.bench2(rank, world, list(range(world)), sizes=[1 << 26], dtypes=("bfloat16",),
                            quiet=True)
            r0 = next(r for r in rows if r["dim"] == "0")
            nb, f = r0["bytes"], (world - 1) / world
            line["reshard_bus"] = {
                "bytes": nb, "dtype": "bf16", "unit": "GB/s", "nvlink_peak": 900.0,
                "all_gather": r0["ag_edb_GBs"], "reduce_scatter": r0["rs_edb_GBs"],
                "all_reduce": r0.get("ar_edb_GBs"), "all_to_all": r0.get("a2a_edb_GBs"),
                "nccl_all_gather": nb * f / r0["ag_nccl_us"] / 1e3,
                "nccl_reduce_scatter": nb * f / r0["rs_nccl_us"] / 1e3,
                "nccl_all_reduce": 2 * nb * f / r0["ar_nccl_us"] / 1e3 if "ar_nccl_us" in r0 else None,
                "frac_of_nvlink_peak": r0["ag_edb_GBs"] / 900.0}
        except Exception as e:  # the microbench must never sink the throughput line
            line["reshard_bus"] = {"error": repr(e)[:200]}
    if roof:
        roof["share_of_step"] = roof["gemm_ms_per_step"] / ms_per_step
        line["roofline"] = roof
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = {k: v for k, v in cpu_train_step_throughput(
                    args, args.cpu_sample_seqs).items() if k != "loss"}
            except Exception as e:  # the baseline must never sink the measurement
                line["cpu_baseline"] = {"error": repr(e)}
        print(json.dumps(line, default=str), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        raise SystemExit("parity leg failed: " + json.dumps(parity, default=str))


def run_torch_nccl(args):
    """GPU baseline on the same box: the same model / batches / optimizer in stock eager PyTorch
    (bf16, cuBLAS GEMMs, cuDNN attention, ATen elementwise) with DistributedDataParallel over NCCL
    for N > 1 — none of this repository's kernels, graph passes or runtime."""
    import dataclasses
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from easydist_b200.workloads import GPT2, GPT2_CONFIGS, synthetic_tokens
    cfg = dataclasses.replace(GPT2_CONFIGS[args.model], attn=args.attn,
                              block_size=max(args.seq, GPT2_CONFIGS[args.model].block_size))
    torch.manual_seed(0)
    model = GPT2(cfg).to(device="cuda", dtype=torch.bfloat16)
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
    opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, foreach=True)
    B, S = args.batch_per_gpu, args.seq
    dev = [tuple(t.cuda() for t in synthetic_tokens(cfg, B, S, seed=1000 * b + rank)) for b in range(4)]

    def step(i):
        t, y = dev[i % 4]
        loss = net(t, y)
        loss.backward()
        opt.step()
        opt.zero_grad(True)
        return loss

    for i in range(max(3, args.warmup)):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        value = B * world * args.steps / (ms.item() / 1e3)
        cfgd = workload_config(args, world)
        cfgd["parallelism"] = f"DistributedDataParallel dp{world}" if world > 1 else "single GPU"
        cfgd["cuda_graph"] = False
        print(json.dumps({"impl": "torch-nccl", "metric": "train_step_throughput", "value": value,
                          "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                          "warmup": max(3, args.warmup), "ms_per_step": ms.item() / args.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "bf16", "data": "synthetic", "config": cfgd,
                          "loss": float(loss)}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.mode == "auto" and args.impl == "edb":
        from tools import bench_c1_auto
        bench_c1_auto.run(argparse.Namespace(mesh="", steps=args.steps, warmup=max(3, args.warmup),
                                             no_cuda_graph=args.no_cuda_graph))
        return
    if args.impl == "torch-nccl":
        run_torch_nccl(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_edb(args)


if __name__ == "__main__":
    main()
