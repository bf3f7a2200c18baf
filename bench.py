#!/usr/bin/env python
"""Benchmark of the GenPercept one-step hot path (BASELINE.json metric: images/sec at 768x768 depth).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W

A "step" = one pass of ``GenPerceptPipeline.single_infer`` over one batch of 8 synthetic 768x768
images per GPU (BASELINE.json configs[1]; weak scaling: every rank runs its own batch, no data-path
collective, SURVEY.md 8e).  Rank 0 prints ONE JSON line:

  value        whole-job images/sec with the uint8 batch already resident in HBM (device timed).
  e2e          the same metric through the public API with pinned HOST buffers: H2D of the uint8
               batch and D2H of the fp32 maps inside the timed region.
  roofline     the dominant kernel (tcgen05 implicit GEMM): algorithmic FLOPs of all its launches in
               a step / their summed CUDA-event durations, vs the measured bf16 peak.
  cpu_baseline the CPU oracle (oracle/, a port of the diffusers path) on the host cores, bounded sample.

--impl reference times the reference's own CPU path.  diffusers is not installable here (no
network, absent from /opt/wheelhouse), so that arm runs the oracle port on the host cores; each
step is ONE image of the benched workload's size (768x768 by default: the same config, a bounded
sample of the batch), with the thread count chosen by a probe at the benched size.

--config N selects another BASELINE.json configuration (the default line is configs[1]):
  1  one 512x512 depth image (the reference's CPU plumbing case)      3  normal 768x768, 8 / rank, all-gather of the maps
  2  depth 768x768, batch 8 / GPU (default)                           4  DPT readout 768x768, 4 / rank
  5  depth, batch 1, resolution sweep 384 / 512 / 768 / 1024 (one line; `sweep` holds the four points)

--dump-outputs DIR writes what the last device-resident timed step returned (rank 0's fp32 maps, [B, C, H, W]) to
DIR/prediction.npy, so that two builds can be compared output for output: inputs and weights are seeded, so the same
arguments give the same inputs.  Maps larger than 64 MB are thinned to every k-th element of the flattened array.
"""
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

from genpercept_b200 import flops as FL  # noqa: E402
from genpercept_b200 import weights as W  # noqa: E402

METRIC = "images/sec at 768x768 depth"
UNIT = "images/s"
DUMP_LIMIT = 64 << 20


def text_embed():
    e = np.load(os.path.join(ROOT, "tests", "golden", "empty_text_embed_2x1024.npy")).astype(np.float32)
    return torch.from_numpy(e)[None]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": d.get("bf16_tflops_sustained", 1450.1), "tflops_burst": d.get("bf16_tflops", 1703.2),
                "hbm_gbs": d.get("hbm_gbs", 6486.5), "src": "MEASURED_PEAKS.json (sustained bf16 GEMM; kernel timed inside a long step)"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(d, arrays):
    """arrays: name -> float32 / float64 numpy array; each one thinned to a fixed stride to stay under DUMP_LIMIT in all."""
    os.makedirs(d, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    stride = -(-total // DUMP_LIMIT)
    for name, a in arrays.items():
        if stride > 1:
            a = np.ascontiguousarray(a.reshape(-1)[::stride])
            print(f"bench: {name} thinned to every {stride}th element ({a.size} values)", file=sys.stderr)
        np.save(os.path.join(d, f"{name}.npy"), a)


def best_thread_count(p, cores, res, mode="depth"):
    """The thread count is chosen AT THE BENCHED SIZE on the stage that dominates the CPU time there (the VAE encoder:
    the same convolutions at the same extents as the whole path, ~1/4 of its FLOPs): PyTorch's CPU conv path does
    not scale to all 128 host threads, and where it stops depends on the tensor extents."""
    x = torch.zeros((1, 3, res, res))
    best, best_t, log = None, None, []
    for t in sorted({min(cores, c) for c in (16, 32, 64, cores)}):
        torch.set_num_threads(t)
        t0 = time.perf_counter()
        p.encode_rgb(x)
        dt = time.perf_counter() - t0
        log.append((t, round(dt, 2)))
        if best is None or dt < best:
            best, best_t = dt, t
    return best_t, log


def cpu_baseline_sample(state, res, threads, steps=1, warmup=0, mode="depth", use_dpt=False):
    """Oracle (CPU port of the diffusers path) on ONE `res` x `res` image per step.  Returns
    (seconds per step, threads used, probe log)."""
    from oracle.pipeline import OraclePipeline
    p = OraclePipeline(state, text_embed(), use_dpt=use_dpt)
    fixed = os.environ.get("GP_BENCH_CPU_THREADS")            # skip the probe (tests)
    if fixed:
        threads, log = min(int(fixed), threads), "fixed by GP_BENCH_CPU_THREADS"
    else:
        threads, log = best_thread_count(p, threads, res)
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(1002)
    x = torch.randint(0, 256, (1, 3, res, res), generator=g, dtype=torch.uint8).float() / 255.0 * 2.0 - 1.0
    for _ in range(warmup):
        p.single_infer(x, mode=mode)
    t0 = time.perf_counter()
    for _ in range(steps):
        p.single_infer(x, mode=mode)
    return (time.perf_counter() - t0) / steps, threads, log


def run_reference(args, rank):
    """The reference's own CPU implementation of the path on the host cores (the oracle port: diffusers cannot be
    installed).  Each step = ONE image of the benched size (same metric, same config; a bounded sample of the batch:
    images are independent, so images/s does not depend on the batch size on the CPU)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    res = args.ref_res or args.res
    dpt = args.readout == "dpt"
    state = W.synth_state(1234, with_dpt=dpt)
    sec, used, log = cpu_baseline_sample(state, res, cores, steps=args.steps, warmup=min(args.warmup, 1),
                                         mode=args.mode, use_dpt=dpt)
    scale = FL.single_infer_flops(args.res, args.res, args.readout) / FL.single_infer_flops(res, res, args.readout)
    v = 1.0 / (sec * scale)
    sample = (f"each step = single_infer on 1 image {res}x{res} fp32, {args.readout} readout (oracle port of the diffusers "
              f"CPU path; {used} of {cores} host threads = fastest of a probe at this size: {log})"
              + ("" if res == args.res else f"; value = measured img/s / {scale:.2f} ({args.res}^2 : {res}^2 algorithmic FLOPs)"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1000.0, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args) + ", CPU reference arm (1 image per step)", "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": used, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


CONFIGS = {       # BASELINE.json configs[] -> bench arguments (index = position in the list + 1)
    1: dict(batch=1, res=512, mode="depth", readout="vae"),
    2: dict(batch=8, res=768, mode="depth", readout="vae"),
    3: dict(batch=8, res=768, mode="normal", readout="vae", gather=True),
    4: dict(batch=4, res=768, mode="depth", readout="dpt"),
    5: dict(batch=1, res=768, mode="depth", readout="vae", sweep=(384, 512, 768, 1024)),
}


def workload_name(args):
    return (f"{args.mode} {args.res}x{args.res} batch={args.batch}/GPU, {args.readout} readout "
            f"(BASELINE.json configs[{args.config - 1}])")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configuration (see the module docstring)")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default: the config's)")
    ap.add_argument("--res", type=int, default=None)
    ap.add_argument("--mode", default=None, choices=["depth", "normal"])
    ap.add_argument("--dtype", default="f16", choices=["f16", "bf16"])
    ap.add_argument("--precision", default="default", choices=["default", "high"])
    ap.add_argument("--readout", default=None, choices=["vae", "dpt"])
    ap.add_argument("--gather", action="store_true", default=None, help="all-gather the maps over NCCL inside the e2e step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-res", type=int, default=None, help="CPU arm: image size (default: the benched size)")
    ap.add_argument("--cuda-graph", action="store_true")
    ap.add_argument("--ops-json", default=None, help="write the per-op timing table here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the maps the last timed step computed to DIR/prediction.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    for k, v in CONFIGS[args.config].items():
        if k != "sweep" and getattr(args, k, None) is None:
            setattr(args, k, v)
    args.gather = bool(args.gather)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from genpercept_b200.pipeline import GenPerceptPipeline

    dt = torch.float16 if args.dtype == "f16" else torch.bfloat16
    dpt = args.readout == "dpt"
    state = W.synth_state(1234, with_dpt=dpt)
    small = args.batch * args.res * args.res <= 2 * 768 * 768
    pipe = GenPerceptPipeline(unet=state["unet"], vae=state["vae"], customized_head=state["dpt"] if dpt else None,
                              text_embed=text_embed(), torch_dtype=dt, device=local, precision=args.precision,
                              cuda_graph=True if args.cuda_graph else ("auto" if small else False))
    eng = pipe._engine
    C = 1 if (dpt or args.mode == "depth") else 3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(B, R, steps, warmup, sampler=None):
        """-> (ms device-resident, ms end to end, host copy of the last device-resident step's maps or None) for `steps`
        steps of B images R x R, max over ranks."""
        g = torch.Generator().manual_seed(1002 + rank)
        host_in = [torch.randint(0, 256, (B, 3, R, R), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
        dev_in = [h.cuda() for h in host_in]
        dev_out = torch.empty((B, C, R, R), dtype=torch.float32, device="cuda")
        host_out = torch.empty((B, C, R, R), dtype=torch.float32).pin_memory()
        gathered = torch.empty((world * B, C, R, R), dtype=torch.float32, device="cuda") if (args.gather and world > 1) else None
        for i in range(warmup):
            pipe.single_infer(dev_in[i % 2], mode=args.mode)
            eng.infer(host_in[i % 2], out_channels=C, out=host_out)
        if sampler is not None:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # ---- device-resident timing (value): the last kernel writes straight into dev_out
        barrier()
        e0.record()
        for i in range(steps):      # the last step always takes dev_in[0]: --dump-outputs does not depend on --steps
            eng.infer(dev_in[(steps - 1 - i) % 2], out_channels=C, out=dev_out)
        e1.record()
        barrier()
        ms_dev = max_over_ranks(e0.elapsed_time(e1))
        last = dev_out.cpu().numpy() if args.dump_outputs else None       # outside both timed regions
        # ---- end to end through the public API with host buffers (e2e)
        barrier()
        e0.record()
        for i in range(steps):
            if gathered is not None:
                # the final kernel writes this rank's maps into its slice of the gather buffer; NCCL gathers in place
                mine = gathered[rank * B:(rank + 1) * B]
                eng.infer(host_in[i % 2], out_channels=C, out=mine)               # H2D inside gp_infer
                dist.all_gather_into_tensor(gathered, mine)
                host_out.copy_(mine, non_blocking=True)
            else:
                pred = pipe.single_infer(host_in[i % 2], mode=args.mode)          # H2D inside gp_infer
                host_out.copy_(pred, non_blocking=True)                           # D2H of the step's result
            torch.cuda.current_stream().synchronize()
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        return ms_dev, ms_e2e, last

    sampler = ClockSampler(local) if rank == 0 else None
    B, R = args.batch, args.res
    ms_dev, ms_e2e, last = measure(B, R, args.steps, args.warmup, sampler)
    clocks = sampler.stop() if rank == 0 else None
    info = eng.plan_info()

    sweep = None
    if args.config == 5:            # resolution sweep, batch 1 (the headline stays the 768x768 point measured above)
        sweep = []
        for r in CONFIGS[5]["sweep"]:
            d, e = (ms_dev, ms_e2e) if r == R else measure(1, r, args.steps, args.warmup)[:2]
            fl = FL.single_infer_flops(r, r, args.readout)
            sweep.append({"res": r, "ms_per_image": d / args.steps, "images_per_s": world * args.steps / (d / 1000.0),
                          "e2e_images_per_s": world * args.steps / (e / 1000.0),
                          "algorithmic_tflops": world * args.steps * fl / (d / 1000.0) / 1e12})
        eng.plan(B, R, R)           # back to the headline plan for the per-op pass

    # ---- per-op pass: CUDA events around every op of one step (serialised, warm), rank 0 only
    roofline = None
    if rank == 0:
        eng.profile_ops(out_channels=C)                                  # warm
        passes = [eng.profile_ops(out_channels=C) for _ in range(3)]
        ops = passes[0]
        for o, *rest in zip(*passes):                                    # per-op MEDIAN of three passes
            o["usec"] = statistics.median([o["usec"]] + [r["usec"] for r in rest])
        ig = [o for o in ops if o["kind"] == 1 and o["usec"] > 0]
        t_ig = sum(o["usec"] for o in ig) * 1e-6
        f_ig = sum(o["flops"] for o in ig)
        x_ig = sum(o["flops_exec"] for o in ig)
        t_all = sum(o["usec"] for o in ops) * 1e-6
        pk = measured_peaks()
        ach = f_ig / t_ig / 1e12 if t_ig > 0 else 0.0
        ach_x = x_ig / t_ig / 1e12 if t_ig > 0 else 0.0
        step_tf = B * FL.single_infer_flops(R, R, args.readout) / (ms_dev / args.steps / 1000.0) / 1e12
        roofline = {"kernel": "gp::igemm_kernel + gp::igemm_patch_kernel (tcgen05 implicit GEMM)", "bound": "tensor",
                    "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"],
                    "achieved_executed": ach_x, "frac_executed": ach_x / pk["tflops"],
                    "whole_step": {"achieved": step_tf, "frac": step_tf / pk["tflops"],
                                   "what": "algorithmic FLOPs of the whole step / the timed step (every kernel, this GPU)"},
                    "traffic": None, "launches_per_step": len(ig), "share_of_step_time": t_ig / t_all if t_all > 0 else None,
                    "peak_source": pk["src"],
                    "how": "achieved = sum(ALGORITHMIC FLOPs of every implicit-GEMM launch of a step) / sum(CUDA-event duration "
                           "of those launches) (per-op median of 3 serialised warm passes, events on the launch stream); "
                           "achieved_executed counts the MMA work actually issued (the six upsample-fused convs run 4 of "
                           "their 9 algorithmic taps)"}
        # DRAM bytes moved by those launches: NOT measured in this run — one ncu pass over every launch of a warm step of
        # the default workload (scripts/prof_step.py), committed under profiles/.
        tf = os.path.join(ROOT, "profiles", "r2_step_dram.json")
        if os.path.exists(tf) and args.config == 2 and B == 8 and R == 768 and args.precision == "default" and len(ig) > 0:
            sd = json.load(open(tf))
            if sd.get("igemm_launches") == len(ig):
                roofline["traffic"] = sd["igemm_dram_bytes"] / len(ig)
                roofline["traffic_unit"] = "bytes per launch (mean over the step's implicit-GEMM launches; ncu dram__bytes_read+write)"
                roofline["traffic_source"] = "committed ncu capture profiles/r2_step_dram.json (not re-measured in this run)"
                roofline["algorithmic_bytes_per_launch"] = sum(o["bytes"] for o in ig) / len(ig)
        if args.ops_json:
            json.dump(ops, open(args.ops_json, "w"), indent=1)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        rr = args.ref_res or R
        sec, used, log = cpu_baseline_sample(state, rr, cores, steps=1, warmup=0, mode=args.mode, use_dpt=dpt)
        scale = FL.single_infer_flops(R, R, args.readout) / FL.single_infer_flops(rr, rr, args.readout)
        cpu = {"value": 1.0 / (sec * scale), "unit": UNIT, "cores": used, "kind": "port",
               "sample": f"oracle (CPU port of the diffusers path, fp32, {used} of {cores} host threads = fastest of a probe at this "
                         f"size {log}): 1 image {rr}x{rr} in {sec:.2f} s"
                         + ("" if rr == R else f", scaled by {scale:.2f} ({R}^2 : {rr}^2 algorithmic FLOPs)")}

    if rank == 0:
        n_img = world * B * args.steps
        per_img = FL.single_infer_flops(R, R, args.readout)
        out = {
            "metric": METRIC, "value": n_img / (ms_dev / 1000.0), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype if args.precision == "default" else "f16x2 (hi+lo pairs, fp32-class)",
            "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "weights": "seeded synthetic SD-2.1 topology (no checkpoints offline)",
                       "global_batch": world * B, "parallelism": f"dp{world} (independent replicas, batch sharded)"
                                                                 + (", one NCCL all-gather of the maps per step (e2e)" if args.gather and world > 1 else ""),
                       "l2": f"no flush needed: per-step working set {info['arena_bytes'] / 2**30:.1f} GiB arena + "
                             f"{info['weight_bytes'] / 2**30:.2f} GiB weights >> 126 MB L2; 2 alternating inputs",
                       "algorithmic_tflop_per_image": per_img / 1e12, "cuda_graph": bool(args.cuda_graph) or small,
                       "precision": args.precision},
            "model_tflops": n_img * per_img / (ms_dev / 1000.0) / 1e12,
            "e2e": {"value": n_img / (ms_e2e / 1000.0), "unit": UNIT, "h2d_bytes_per_step": B * 3 * R * R,
                    "d2h_bytes_per_step": B * C * R * R * 4, "ms_per_step": ms_e2e / args.steps,
                    "api": "GenPerceptPipeline.single_infer(pinned uint8 host batch) + D2H of the fp32 maps"
                           + (" + all_gather_into_tensor of every rank's maps" if args.gather and world > 1 else "")},
            "gpu_launches": int(info["launches"]) * args.steps * world,   # kernels launched in the device-timed region
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        }
        if sweep is not None:
            out["sweep"] = sweep
        print(json.dumps(out))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"prediction": last})
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
