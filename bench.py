#!/usr/bin/env python
"""Benchmark of the MAML / MAML++ hot path (BASELINE.json metric: meta-tasks/sec, 5-way, 5 inner steps).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--impl ours|reference]

One "step" = one ``run_train_iter`` over one meta-batch of synthetic episodes: inner-loop unroll for every
task, second-order meta-gradient, (all-reduce over ranks), clamp + Adam, running-stat EMA.
  value      whole-job tasks/s with the episode tensors already resident in HBM, per-step CUDA-event timing,
             L2 flushed between steps, max over ranks;
  e2e        the same metric through the public API ``MAMLFewShotClassifier.run_train_iter`` with HOST
             tensors: pinned H2D of the episodes and D2H of loss / accuracy / logits inside the timed region;
  roofline   the dominant kernel class (3x3 implicit-GEMM convolutions): algorithmic conv FLOPs per launch
             (SURVEY.md section 8d) / mean launch duration from CUDA events on the launching stream, against the
             measured tensor peak (MEASURED_PEAKS.json bf16 / 2 = TF32, / 3 for the fp32-faithful 3xTF32 split);
  cpu_baseline  the reference's CPU path restated (oracle "port": same torch.nn.functional ops + autograd as
             the reference -- the reference itself is Python and cannot travel to the GPU box), timed on the
             host cores on a bounded sample of the same workload.
``--impl reference`` prints the CPU arm as its own line (rank 0 only under torchrun).
Weak scaling: every rank holds ``batch_size`` tasks (tasks are sharded over GPUs, one all-reduce of the flat
meta-gradient per iteration); the global meta-batch is N x batch_size.
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

METRIC = "meta-tasks/sec (5-way, 5 inner steps, second order)"
DEFAULT_CONFIG = "omniglot_mamlpp_5w1s"          # BASELINE.json configs[1]: the 1xB200 headline workload
SCALING = {}                                      # config -> "weak" / "strong" (filled by main from the CLI)


def workload_desc(name, args, n_gpus):
    return {
        "workload": "%s: %d-way %d-shot, %d target/class, %dx%dx%d, %d filters, %d inner steps, meta-batch %d per GPU"
                    % (name, args.num_classes_per_set, args.num_samples_per_class, args.num_target_samples,
                       args.image_height, args.image_width, args.image_channels, args.cnn_num_filters,
                       args.number_of_training_steps_per_iter, args.batch_size),
        "config": name, "tasks_per_gpu": int(args.batch_size), "global_meta_batch": int(args.batch_size) * n_gpus,
        "second_order": bool(args.second_order), "multi_step_loss": bool(args.use_multi_step_loss_optimization),
        "per_step_bn": bool(args.per_step_bn_statistics), "parallelism": "task-sharded dp%d" % n_gpus,
        "l2": "flushed between steps (256 MiB memset outside the per-step event pair); 8 distinct episode batches cycled through the two staging slots",
        "inputs": "bernoulli(0.93) 28x28x1" if args.image_channels == 1 else "normal(0,1) 84x84x3",
    }


def flops_per_task(args):
    """Algorithmic conv FLOPs per task (SURVEY.md section 8d)."""
    h, w, c = args.image_height, args.image_width, args.image_channels
    F = args.cnn_num_filters
    fl = []
    for _ in range(args.num_stages):
        fl.append(2.0 * h * w * F * c * 9)
        h, w, c = h // 2, w // 2, F
    n_s = args.num_classes_per_set * args.num_samples_per_class
    n_t = args.num_classes_per_set * args.num_target_samples
    S = args.number_of_training_steps_per_iter
    sup2 = 4 * fl[0] + 9 * sum(fl[1:])
    sup1 = 2 * fl[0] + 3 * sum(fl[1:])
    tgt = 2 * fl[0] + 3 * sum(fl[1:])
    n_tp = S if args.use_multi_step_loss_optimization else 1
    return S * n_s * (sup2 if args.second_order else sup1) + n_tp * n_t * tgt


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def _cpu_port_iteration_times(args, iters, warmup, threads):
    import torch
    from oracle import maml_oracle as O
    torch.set_num_threads(threads)
    state = O.init_state(args)
    names = O.trainable_names(args)
    m = {n: torch.zeros_like(state[n]) for n in names}
    v = {n: torch.zeros_like(state[n]) for n in names}
    step, times = 0, []
    for it in range(warmup + iters):
        batch = O.synthetic_batch(args, iteration=it)
        t0 = time.perf_counter()
        res = O.autograd_train_iter(state, args, batch, 0)
        clamp = [n for n in names if n.startswith("classifier.")] if "imagenet" in args.dataset_name else None
        newp, m, v, step = O.adam_step({n: state[n] for n in names}, res["grads"], m, v, step, O.cosine_lr(args, 0), clamp=clamp)
        state.update(newp)
        state.update(res["running"])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return times


def cpu_port_tasks_per_sec(args, iters, warmup, threads=None):
    """The reference's CPU path (restated: same torch.nn.functional ops + autograd.grad(create_graph) + one reverse
    sweep as reference few_shot_learning_system.py:170-263,325-336) on the host cores.  The thread count is tuned
    (1 probe iteration each over 8/16/32/64/all cores -- these ops are small, more threads is not faster) and the
    best is used; ``cores`` reports the threads actually used.  Returns (tasks/s, cores, sample, times)."""
    ncpu = os.cpu_count() or 1
    if threads is None:
        cands = sorted(set(c for c in (8, 16, 32, 64, ncpu) if c <= ncpu)) or [ncpu]
        best, best_t = cands[0], None
        for c in cands:
            t = _cpu_port_iteration_times(args, 1, 1, c)[0]
            if best_t is None or t < best_t:
                best, best_t = c, t
            if t > 4.0 * best_t:
                break
        threads = best
    times = sorted(_cpu_port_iteration_times(args, iters, warmup, threads))
    med = times[len(times) // 2]
    sample = "%d timed iterations of %d tasks (median), %d warm-up, %d of %d host threads (tuned)" % (
        iters, args.batch_size, warmup, threads, ncpu)
    return args.batch_size / med, threads, sample, times


def torch_gpu_port_tasks_per_sec(args, dev, iters=3, warmup=1):
    """SURVEY.md section 8d "library kernels to beat": the same call-for-call restatement of the reference
    (torch.nn.functional convs / batch_norm / max_pool2d + autograd.grad(create_graph) + one reverse sweep), but on the
    GPU through PyTorch's own CUDA kernels (cuDNN / ATen), strict fp32 (TF32 off).  This is what the reference does when
    it sees a GPU (few_shot_learning_system.py:73-81).  A baseline beside the line, never the thing measured."""
    import torch
    from oracle import maml_oracle as O
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        state = {k: v.to(dev) for k, v in O.init_state(args).items()}
        names = O.trainable_names(args)
        m = {n: torch.zeros_like(state[n]) for n in names}
        v = {n: torch.zeros_like(state[n]) for n in names}
        step, times = 0, []
        for it in range(warmup + iters):
            batch = tuple(t.to(dev) for t in O.synthetic_batch(args, iteration=it))
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            res = O.autograd_train_iter(state, args, batch, 0)
            clamp = [n for n in names if n.startswith("classifier.")] if "imagenet" in args.dataset_name else None
            newp, m, v, step = O.adam_step({n: state[n] for n in names}, res["grads"], m, v, step, O.cosine_lr(args, 0), clamp=clamp)
            state.update(newp)
            state.update(res["running"])
            torch.cuda.synchronize(dev)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        times.sort()
        med = times[len(times) // 2]
        return {"value": args.batch_size / med, "unit": "tasks/s", "ms_per_step": 1e3 * med,
                "kind": "port on PyTorch CUDA library kernels (cuDNN / ATen eager autograd), fp32, inputs resident",
                "sample": "%d timed iterations of %d tasks (median), %d warm-up" % (iters, args.batch_size, warmup)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def _visible_gpu_token(local_rank):
    """What CUDA_VISIBLE_DEVICES must be for a child process to see exactly this rank's GPU."""
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        toks = [t.strip() for t in vis.split(",") if t.strip()]
        if local_rank < len(toks):
            return toks[local_rank]
    return str(local_rank)


def run_unmodified_reference(config, batch_size, device, steps, warmup, local_rank=0, tune=True, max_seconds=240.0):
    """Run ``baseline/run_reference.py`` (the UNMODIFIED reference staged under baseline/_ref, its own public API and
    stock code path) in a child process and return its JSON dict, or {"unavailable": why}."""
    script = os.path.join(ROOT, "baseline", "run_reference.py")
    cmd = [sys.executable, script, "--config", config, "--device", device, "--steps", str(steps), "--warmup", str(warmup),
           "--max-seconds", str(max_seconds)]
    if batch_size:
        cmd += ["--batch-size", str(batch_size)]
    if tune and device == "cpu":
        cmd += ["--tune-threads"]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)                    # the reference is a single-process program; torchrun pins OMP_NUM_THREADS=1
    env["CUDA_VISIBLE_DEVICES"] = "" if device == "cpu" else _visible_gpu_token(local_rank)
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=max_seconds + 600)
    except subprocess.TimeoutExpired:
        return {"unavailable": "reference run timed out"}
    for line in reversed(r.stdout.strip().splitlines()):
        line = line.strip()
        if line.startswith("{"):
            try:
                return json.loads(line)
            except ValueError:
                continue
    return {"unavailable": ("reference run failed (rc %d): %s" % (r.returncode, (r.stderr or r.stdout)[-300:])).replace("\n", " | ")}


def reference_cpu_baseline(cli, args, steps, warmup):
    """cpu_baseline dict (+ raw run) from the unmodified reference on the host cores; falls back to the oracle port
    (stated in ``kind``) only when baseline/_ref was not staged."""
    ref = run_unmodified_reference(cli.config, int(args.batch_size), "cpu", steps, warmup)
    if "unavailable" not in ref:
        sample = "%d timed iterations of %d tasks (median), %d warm-up, %d of %d host threads (1 probe iteration each at 8/16/32/64/all, fastest kept)" % (
            len(ref["times_s"]), ref["batch_size"], ref["warmup"], ref["threads"], ref["host_threads"])
        return {"value": ref["tasks_per_sec"], "unit": "tasks/s", "cores": ref["threads"], "kind": "reference",
                "sample": sample, "cpu_model": ref["cpu_model"], "host_threads": ref["host_threads"],
                "reference_commit": ref.get("commit"), "ms_per_step": ref["ms_per_iter"],
                "thread_probe_s": ref.get("thread_probe_s")}, ref
    tps, cores, sample, times = cpu_port_tasks_per_sec(args, iters=min(steps, 8), warmup=min(warmup, 2))
    return {"value": tps, "unit": "tasks/s", "cores": cores, "kind": "port",
            "sample": sample + " -- FALLBACK: " + ref["unavailable"], "ms_per_step": 1e3 * sorted(times)[len(times) // 2]}, ref


def run_reference_arm(cli, args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (unmodified, baseline/_ref) on the host
    cores, same config / metric / unit; rank 0 only."""
    if rank != 0:
        return
    steps = max(1, min(cli.steps, 20))
    warm = max(1, min(cli.warmup, 2))
    t0 = time.perf_counter()
    cb, raw = reference_cpu_baseline(cli, args, steps, warm)
    n_timed = len(raw["times_s"]) if "times_s" in raw else steps
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "tasks/s", "n_gpus": world, "steps": n_timed,
        "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": SCALING.get(cli.config, "weak"),
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "config": workload_desc(cli.config, args, 1),
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "tasks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = the unmodified reference's run_train_iter (few_shot_learning_system.py:338-369) imported from "
                "baseline/_ref with CUDA_VISIBLE_DEVICES='' (BASELINE.md section 4); one step = one meta-batch of %d tasks; "
                "wall %.1f s" % (int(args.batch_size), time.perf_counter() - t0),
    }
    _emit(line)


def _stats(xs):
    xs = sorted(xs)
    return {"min": xs[0], "median": xs[len(xs) // 2], "max": xs[-1]}


def measure_device_loop(model, args, dev, rank, world, K, W, flush, n_pool=8, sampler=None, sync_each_step=False):
    """`value` leg: K steps with the episode tensors resident in HBM, no host sync inside the loop, L2 flushed between
    steps (outside the per-step CUDA-event pair).  Returns per-rank timing; the caller takes the max over ranks."""
    import torch
    import torch.distributed as dist
    from howtotrainyourmamlpytorch_b200 import synthetic_batch
    host_batches = [synthetic_batch(args, iteration=1000 * rank + i) for i in range(n_pool)]
    dev_batches = [(hb[0].to(dev), hb[1].to(dev), hb[2].long().to(dev), hb[3].long().to(dev)) for hb in host_batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_step(i):
        model._current_lr = model._cosine_lr(0)
        return model._run(dev_batches[i % n_pool], 0, training_phase=True, apply_update=True)

    for i in range(max(W, 4)):      # warm-up: >= W steps, and both staging slots (one CUDA graph per slot) captured
        device_step(i)
    barrier()
    if sampler is not None:
        sampler.start()
        time.sleep(0.3)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    loop0, loop1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.perf_counter()
    loop0.record()
    last = None
    for i in range(K):
        if flush is not None:
            flush.zero_()
        ev[i][0].record()
        last = device_step(W + i)
        ev[i][1].record()
        if sync_each_step:
            torch.cuda.synchronize()
    loop1.record()
    barrier()
    wall = time.perf_counter() - wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    return {"step_ms": step_ms, "sum_ms": sum(step_ms), "loop_ms": loop0.elapsed_time(loop1), "wall_s": wall,
            "host_batches": host_batches, "device_step": device_step, "barrier": barrier, "last": last}


def dump_outputs(model, last, out_dir, rank):
    """Write what the last timed step handed back (loss, accuracy, logged learning rate, multi-step loss weights and
    the per-task target logits, i.e. what ``run_train_iter`` returns) as ``<out_dir>/<name>.npy`` so that two builds
    can be compared output for output.  Must run before anything else reuses the engine's result buffers."""
    import numpy as np
    losses, preds = model._finish(*last)
    losses["learning_rate"] = model._logged_lr(0)
    arrays = {k: np.asarray(v, dtype=np.float64 if isinstance(v, float) else np.float32) for k, v in losses.items()}
    arrays["logits"] = np.stack(preds).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if rank == 0 else "_rank%d" % rank
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def gather_rank_stats(step_ms, loop_ms, coll_us, dev, world):
    """[per rank: min / median / max step ms, loop ms, median collective us] on every rank (tiny all_gather)."""
    import torch
    import torch.distributed as dist
    st = _stats(step_ms)
    t = torch.tensor([st["min"], st["median"], st["max"], loop_ms, coll_us], dtype=torch.float64, device=dev)
    if world == 1:
        return [t.tolist()]
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [o.tolist() for o in out]


def roofline_from_profile(prof, prof_steps, peaks, peak_src, value, fpt, world, traffic):
    conv_ms, conv_fl, conv_n = prof["conv_igemm"]
    wg_ms, wg_fl, wg_n = prof["wgrad"]
    c0_ms, c0_fl, c0_n = prof["conv_first_block"]
    w0_ms, w0_fl, w0_n = prof["wgrad_first_block"]
    tot_prof_ms = sum(v[0] for v in prof.values())
    # dominant kernel class = every 3x3 conv contraction of blocks >= 1 (forward / tangent / dgrad implicit GEMMs + wgrad)
    dom_ms, dom_fl, dom_n = conv_ms + wg_ms, conv_fl + wg_fl, conv_n + wg_n
    tf32_peak = peaks["bf16_tflops"] / 2.0            # dense TF32 = half of dense bf16 (measured burst)
    peak_3x = tf32_peak / 3.0                         # fp32-faithful 3xTF32 operand split
    achieved = dom_fl / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
    all_ms, all_fl = dom_ms + c0_ms + w0_ms, dom_fl + c0_fl + w0_fl
    return {
        "bound": "tensor", "kernel": "3x3 conv contractions of blocks >= 1: conv_tc_kernel (forward / dgrad / tangent) + wgrad_tc_kernel (weight gradient), both tcgen05 3xTF32 fed by TMA",
        "achieved": achieved, "peak": peak_3x, "unit": "TFLOP/s", "frac": achieved / peak_3x,
        "traffic": traffic,
        "peak_source": peak_src + ": bf16_tflops %.1f / 2 (tf32) / 3 (3xTF32 split)" % peaks["bf16_tflops"],
        "launches_profiled": int(dom_n), "mean_launch_us": 1e3 * dom_ms / max(dom_n, 1),
        "share_of_step": dom_ms / tot_prof_ms if tot_prof_ms > 0 else None,
        "all_convs_incl_first_block": {"achieved": all_fl / (all_ms * 1e-3) / 1e12 if all_ms > 0 else 0.0,
                                       "share_of_step": all_ms / tot_prof_ms if tot_prof_ms > 0 else None},
        "whole_iteration": {"alg_tflops": value * fpt / 1e12, "frac_of_peak": value * fpt / 1e12 / (peak_3x * world)},
        "by_class_ms_per_step": {k: v[0] / prof_steps for k, v in prof.items()},
        "by_class_tflops": {k: (v[1] / (v[0] * 1e-3) / 1e12 if v[0] > 0 and v[1] > 0 else None) for k, v in prof.items()},
    }


def profile_classes(model, device_step, steps=3):
    eng = model._engine
    eng.profile(True)
    for i in range(steps):
        device_step(i)
    prof = eng.profile_read()
    eng.profile(False)
    return prof


def extra_config_line(name, tasks_per_gpu, scaling, dev, rank, world, local_rank, flush, peaks, peak_src, K=6, W=3):
    """Short measurement of another BASELINE configuration (value + roofline by kernel class), same method as the
    headline's `value` leg."""
    import torch
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier, make_args
    args = make_args(name, batch_size=tasks_per_gpu)
    model = MAMLFewShotClassifier(im_shape=(2, args.image_channels, args.image_height, args.image_width), device=dev, args=args)
    r = measure_device_loop(model, args, dev, rank, world, K, W, flush, n_pool=2)
    t = torch.tensor([r["sum_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t[0])
    prof = profile_classes(model, r["device_step"], steps=2)
    value = tasks_per_gpu * world * K / (total_ms * 1e-3)
    fpt = flops_per_task(args)
    roof = roofline_from_profile(prof, 2, peaks, peak_src, value, fpt, world, None)
    out = {"config": name, "tasks_per_gpu": tasks_per_gpu, "global_meta_batch": tasks_per_gpu * world, "scaling": scaling,
           "value": value, "unit": "tasks/s", "ms_per_step": total_ms / K, "steps": K, "warmup": W,
           "gflop_per_task": fpt / 1e9, "alg_tflops": value * fpt / 1e12,
           "frac_of_3xtf32_peak": value * fpt / 1e12 / (roof["peak"] * world),
           "conv_class_tflops": roof["achieved"], "conv_class_frac": roof["frac"],
           "by_class_ms_per_step": roof["by_class_ms_per_step"], "workspace_mib": model._engine.workspace_bytes / 2 ** 20}
    del model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", type=str, default=DEFAULT_CONFIG)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short lines for the other BASELINE configurations")
    ap.add_argument("--batch-size", type=int, default=None, help="tasks per GPU (default: the config's batch_size)")
    ap.add_argument("--scaling", type=str, default="weak", choices=["weak", "strong"],
                    help="weak: every GPU holds the config's meta-batch; strong: the config's meta-batch is split over the GPUs")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic: do not flush L2 between timed steps")
    ap.add_argument("--sync-each-step", action="store_true", help="diagnostic: synchronize after every timed step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (same arguments, same inputs)")
    cli = ap.parse_args()

    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to fd 1 when
    # NCCL_DEBUG is set): from here on fd 1 points at stderr and the line goes to the saved original.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(line):
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    globals()["_emit"] = emit

    import torch
    from howtotrainyourmamlpytorch_b200 import make_args

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    over = {}
    if cli.batch_size:
        over["batch_size"] = cli.batch_size
    args = make_args(cli.config, **over)
    if cli.scaling == "strong" and world > 1:
        if int(args.batch_size) % world:
            raise SystemExit("strong scaling needs the meta-batch (%d) to be a multiple of the GPU count" % int(args.batch_size))
        args = make_args(cli.config, batch_size=int(args.batch_size) // world)
    SCALING[cli.config] = cli.scaling

    if cli.impl == "reference":
        run_reference_arm(cli, make_args(cli.config, **over), rank, world)
        return

    import torch.distributed as dist
    from howtotrainyourmamlpytorch_b200 import MAMLFewShotClassifier
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    W, K = max(3, cli.warmup), max(1, cli.steps)

    model = MAMLFewShotClassifier(im_shape=(2, args.image_channels, args.image_height, args.image_width), device=dev, args=args)
    B = int(args.batch_size)
    flush = None if cli.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    # ---------------- device-resident throughput (value); clocks sampled on rank 0 only (8 nvidia-smi pollers perturb)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    r = measure_device_loop(model, args, dev, rank, world, K, W, flush, sampler=sampler, sync_each_step=cli.sync_each_step)
    step_ms, device_step, barrier = r["step_ms"], r["device_step"], r["barrier"]
    if cli.dump_outputs:
        dump_outputs(model, r["last"], cli.dump_outputs, rank)
    host_batches = r["host_batches"]
    n_pool = len(host_batches)
    pinned_batches = [tuple(t.pin_memory() for t in hb) for hb in host_batches]
    launches_per_step = model._engine.last_launch_count() + 1 + (1 if args.per_step_bn_statistics else 0) + model.collective_launches()

    # ---------------- end to end through the public API with host buffers (e2e)
    for i in range(max(3, W)):
        model.run_train_iter(pinned_batches[i % n_pool], 0)
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        losses, preds = model.run_train_iter(pinned_batches[(W + i) % n_pool], 0)
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler is not None else None
    h2d = sum(t.numel() * (8 if j >= 2 else 4) for j, t in enumerate(host_batches[0]))   # images fp32, labels int64 on the device
    n_t = args.num_classes_per_set * args.num_target_samples
    d2h = 2 * 4 + B * n_t * args.num_classes_per_set * 4

    # ---------------- the collective alone (N > 1): CUDA events around the in-engine all-reduce of the result vector
    coll_us = 0.0
    if world > 1:
        coll_us = model.time_collective(iters=20)

    # ---------------- roofline leg: per-launch CUDA events by kernel class (separate, un-timed pass)
    prof_steps = 3
    prof = profile_classes(model, device_step, prof_steps)
    eng = model._engine

    # max over ranks
    t_dev = torch.tensor([r["sum_ms"], e2e_s * 1e3, r["loop_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, loop_ms = float(t_dev[0]), float(t_dev[1]), float(t_dev[2])
    per_rank = gather_rank_stats(step_ms, r["loop_ms"], coll_us, dev, world)

    peaks, peak_src = measured_peaks()
    extras = []
    if not cli.no_extras and cli.config == DEFAULT_CONFIG and not cli.batch_size:
        # the other BASELINE configurations, each sharded the way SURVEY.md section 8e prescribes for this GPU count
        plan = []
        if world == 1:
            plan = [("omniglot_maml_5w1s", 8, "single"), ("mini_imagenet_mamlpp_5w1s", 2, "single"),
                    ("mini_imagenet_mamlpp_5w5s", 2, "per-GPU shard of B=16 over 8 GPUs"),
                    ("omniglot_mamlpp_20w5s", 8, "per-GPU shard of B=64 over 8 GPUs")]
        else:
            if 8 % world == 0:
                plan.append(("omniglot_mamlpp_5w1s", 8 // world, "strong (B=8 split over %d GPUs)" % world))
            if world == 2:
                plan.append(("mini_imagenet_mamlpp_5w1s", 1, "strong (B=2 split over 2 GPUs)"))
            plan.append(("mini_imagenet_mamlpp_5w5s", 2, "B=%d, 2 tasks per GPU%s" % (2 * world, " (= BASELINE configs[3])" if world == 8 else "")))
            plan.append(("omniglot_mamlpp_20w5s", 8, "B=%d, 8 tasks per GPU%s" % (8 * world, " (= BASELINE configs[4])" if world == 8 else "")))
        for name, tpg, how in plan:
            try:
                extras.append(extra_config_line(name, tpg, how, dev, rank, world, local_rank, flush, peaks, peak_src))
            except Exception as exc:                   # an extra must never take the headline down
                extras.append({"config": name, "tasks_per_gpu": tpg, "error": repr(exc)[:300]})

    if rank == 0:
        tasks_total = B * world * K
        value = tasks_total / (total_ms * 1e-3)
        e2e_value = tasks_total / (e2e_ms * 1e-3)
        fpt = flops_per_task(args)
        traffic, traffic_note = None, None
        for cand in ("ncu_summary_r2.json", "ncu_summary_r1.json"):
            try:
                d = json.load(open(os.path.join(ROOT, "profiles", cand)))
                traffic = d["dominant_kernel_traffic_bytes_per_launch"]
                traffic_note = d.get("traffic_note", "dram__bytes_read+write of one dominant-kernel launch (ncu --set full, cold cache; profiles/%s)" % cand)
                break
            except Exception:
                continue
        roofline = roofline_from_profile(prof, prof_steps, peaks, peak_src, value, fpt, world, traffic)
        roofline["traffic_note"] = traffic_note
        line = {
            "metric": METRIC, "value": value, "unit": "tasks/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": cli.scaling, "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic", "config": workload_desc(cli.config, args, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "tasks/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / K},
            "gpu_launches": int(launches_per_step * K),
            "roofline": roofline,
            "gflop_per_task": fpt / 1e9,
            "wall_s_device_loop": r["wall_s"],
            "loop_ms_per_step_incl_flush": loop_ms / K,
            "step_ms": _stats(step_ms),
            "per_rank": {"columns": ["step_ms_min", "step_ms_median", "step_ms_max", "loop_ms", "collective_us"], "rows": per_rank},
            "collective": model.collective_desc(),
            "workspace_mib": eng.workspace_bytes / 2 ** 20,
            "last_loss": float(losses["loss"]),
            "other_configs": extras,
        }
        if not cli.no_cpu_baseline and world == 1:
            # the reference's own GPU path (it self-selects CUDA, few_shot_learning_system.py:73-81): the library-kernel
            # baseline on the same B200; then its CPU path on the host cores (bounded sample)
            g = run_unmodified_reference(cli.config, B, "cuda", steps=3, warmup=2, local_rank=local_rank)
            if "unavailable" in g:
                try:
                    line["torch_gpu_baseline"] = torch_gpu_port_tasks_per_sec(args, dev)
                    line["torch_gpu_baseline"]["fallback_reason"] = g["unavailable"]
                except Exception as exc:      # a baseline must never take the measurement down
                    line["torch_gpu_baseline"] = {"unavailable": repr(exc)[:200]}
            else:
                line["torch_gpu_baseline"] = {
                    "value": g["tasks_per_sec"], "unit": "tasks/s", "ms_per_step": g["ms_per_iter"],
                    "kind": "reference (unmodified, baseline/_ref) on its own GPU path: eager PyTorch cuDNN / ATen, fp32, TF32 off",
                    "sample": "%d timed iterations of %d tasks (median), %d warm-up" % (len(g["times_s"]), g["batch_size"], g["warmup"]),
                    "gpu": g.get("gpu")}
            line["cpu_baseline"], _ = reference_cpu_baseline(cli, args, steps=8, warmup=2)
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
