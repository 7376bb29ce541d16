"""bench.py - headline benchmark of the B200 vocoder / synthesizer hot path (contract: see DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-secondary] [--no-cpu-baseline]
                    [--workload hifigan_cfg2|fregan_cfg2|wavernn_cfg1|wavernn_cfg3|tacotron_cfg4|e2e_cfg5] [--precision ...]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  The headline is BASELINE.json configs[1] (the config the metric is quoted on): HiFi-GAN
Generator forward, batch 32 random mels of 256 frames x 80 bins per GPU; a "step" is one forward over one batch; under
torchrun every rank runs its own batch (weak scaling: utterance batches shard across GPUs, no data-path collective).

  value      samples/s, inputs resident in HBM, CUDA events, max over ranks, measured AFTER a >= 2 s soak of the same
             step ("burst" = the same K steps timed right after warm-up, reported beside it)
  e2e        same metric through the drop-in module surface hifigan.inference.infer_waveforms() with HOST numpy mels:
             pinned H2D of the batch and D2H of the waveforms inside the timed region, host sync every step
  roofline   the tcgen05 conv kernel family: layer-granular algorithmic bytes / CUDA-event time of those launches
             (separate profiled pass) vs the measured HBM copy bandwidth; roofline_tensor: FLOPs vs the measured bf16 peak
             (burst peak for the burst figure, sustained peak for the soaked one)
  cpu_baseline  the oracle port of the reference forward on the host cores, bounded sample (rank 0, N = 1 only)
  secondary  every other BASELINE.json config, each with its own value / e2e / roofline / cpu_baseline:
             wavernn_cfg1 (configs[0]), wavernn_cfg3 (configs[2]; device noise AND the reference-identical torch stream),
             tacotron_cfg4 (configs[3]), e2e_cfg5 (configs[4], weak: 128 utterances per GPU; strong: 1024 utterances
             over N GPUs), hifigan_fp32_equivalent (3-term split everywhere), and at N > 1 the fold-sharded cfg 3
--impl reference: the CPU implementation (oracle port, all host threads) on the same config (rank 0 only).
--dump-outputs DIR: after the timed steps, rank 0 writes the waveforms its last timed step returned (the whole batch,
             float32 [32, 1, 51200], 6.6 MB) to DIR/wav.npy.  Inputs and weights are seeded, so two builds run with the same
             arguments can be compared output for output (GAN workloads: hifigan_cfg2, fregan_cfg2).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from bench_common import Ctx, cpu_child, host_threads, log, peaks  # noqa: E402

WORKLOADS = ["hifigan_cfg2", "fregan_cfg2", "wavernn_cfg1", "wavernn_cfg3", "tacotron_cfg4", "e2e_cfg5"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hifigan_cfg2", choices=WORKLOADS)
    ap.add_argument("--precision", default=os.environ.get("MOCKINGBIRD_B200_GAN_PRECISION", "auto"),
                    help="auto (drop-in default: load-time calibration picks f16tc or f16x3) | f16tc | f16x3 | fp32")
    ap.add_argument("--soak-seconds", type=float, default=2.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline workload only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the waveforms of the last timed step to DIR/wav.npy (hifigan_cfg2 / fregan_cfg2)")
    ap.add_argument("--cpu-child", nargs=3, default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.workload not in ("hifigan_cfg2", "fregan_cfg2")):
        ap.error("--dump-outputs needs --impl ours and --workload hifigan_cfg2 or fregan_cfg2")
    return args


# ------------------------------------------------------------------------------------------------
def cpu_hifigan(batch_rows: int, passes: int, threads: int, fregan: bool = False):
    """The CPU implementation (oracle port of the reference forward), batch-1 calls like
    hifigan/inference.py:66-70.  Returns (samples_per_s, seconds, samples)."""
    sys.path.insert(0, str(ROOT / "oracle"))
    sys.path.insert(0, str(ROOT / "synth_weights"))
    import torch
    import gan_oracle as go
    import ref_init as ri

    torch.set_num_threads(threads)
    cfg = ri.FREGAN_CONFIG if fregan else ri.HIFIGAN_CONFIG_16K
    sd = go.fold_weight_norm(ri.fregan_state_dict(cfg, 0)) if fregan else ri.hifigan_state_dict(cfg, 0)
    fwd = go.fregan_forward if fregan else go.hifigan_forward
    mel = torch.rand(32, 80, 256, generator=torch.Generator().manual_seed(2)) * 8 - 4
    with torch.no_grad():
        fwd(sd, cfg, mel[:1])  # warm-up
        t0 = time.perf_counter()
        n = 0
        for _ in range(passes):
            for i in range(batch_rows):
                y = fwd(sd, cfg, mel[i:i + 1])
                n += y.numel()
        dt = time.perf_counter() - t0
    return n / dt, dt, n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    if args.workload in ("wavernn_cfg1", "wavernn_cfg3"):
        import bench_wavernn

        return bench_wavernn.run_reference(args, threads)
    if args.workload == "tacotron_cfg4":
        import bench_tacotron

        return bench_tacotron.run_reference(args, threads)
    if args.workload == "e2e_cfg5":
        import bench_e2e

        return bench_e2e.run_reference(args, threads)
    per_step = []
    total = 0
    SAMPLE = 8  # utterances of the 32-utterance batch timed per step (bounded sample; the forward is per utterance)
    for s in range(args.warmup + args.steps):
        log(f"reference step {s}")
        v, dt, n = cpu_hifigan(SAMPLE, 1, threads, fregan=(args.workload == "fregan_cfg2"))
        if s >= args.warmup:
            per_step.append(dt)
            total += n
    secs = sum(per_step)
    value = total / secs
    ms_full_step = 1e3 * (32 * 51200) / value
    line = {
        "impl": "reference", "metric": "vocoder audio samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_full_step,
        "rtf": (ms_full_step * 1e-3) / (32 * 51200 / 16000.0), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: Generator fwd, batch 32 x 256 frames x 80 mels per GPU",
                   "per_gpu_batch": 32, "frames": 256, "precision": "fp32 (torch CPU)", "parallelism": "cpu"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps x {SAMPLE} of the 32 utterances x 256 frames (batch-1 calls like "
                                   "hifigan/inference.py:66-70), torch-CPU oracle (bit-identical to the reference forward); "
                                   "ms_per_step is scaled to the 32-utterance step"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# ------------------------------------------------------------------------------------------------
def measure_hifigan(ctx: Ctx, args, workload: str, precision: str, steps: int, warmup: int, soak_s: float, cpu: bool,
                    roofline: bool = True, dump_dir: str | None = None):
    """HiFi-GAN / Fre-GAN generator forward on the cfg-2 batch shape; returns the JSON dict (rank 0) or None.
    dump_dir: rank 0 writes the waveforms of the last timed resident step there as wav.npy."""
    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT / "synth_weights"))  # seeded random-init weights (no checkpoints exist)
    import ref_init as ri
    from mockingbird_b200 import _lib
    from mockingbird_b200.vocoder.fregan import inference as fre_vocoder
    from mockingbird_b200.vocoder.hifigan import inference as gan_vocoder

    torch, dist = ctx.torch, ctx.dist
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    fre = workload == "fregan_cfg2"  # SURVEY.md row C1 on the same batch shape (not a BASELINE.json config)
    cfg = ri.FREGAN_CONFIG if fre else ri.HIFIGAN_CONFIG_16K
    sd = ri.fregan_state_dict(cfg, 0) if fre else ri.hifigan_state_dict(cfg, 0)
    B, T = 32, 256
    mod = fre_vocoder if fre else gan_vocoder
    g = mod.load_state(sd, cfg, precision=precision)   # the module-level singleton the drop-in surface serves
    if world > 1:
        dist.broadcast(g.packed_arena(), src=0)         # rank 0's packed weights over NCCL (the only collective)
    hop = g.hop
    requested, precision = precision, g.precision  # "auto" resolves at load time (vocoder/_gan.py: _calibrate)
    mel = (torch.rand(B, 80, T, generator=torch.Generator().manual_seed(2 + rank)) * 8 - 4)
    mel_dev = mel.to(dev)
    mels_np = [mel[i].numpy() for i in range(B)]
    samples_per_step = B * T * hop
    lib = _lib.lib()
    produced = {"n": 0}
    last = {}

    def step_resident():
        last["wav"] = g(mel_dev)

    def step_e2e():
        wavs = mod.infer_waveforms(mels_np, batch_size=B)   # host numpy in, host numpy out, host sync inside
        produced["n"] = sum(len(w) for w in wavs)

    log(f"{workload}/{precision}: weights packed; resident pass")
    l0 = lib.mb_launch_count()
    r = ctx.timed(step_resident, steps, max(3, warmup), soak_s)
    launches_total = int(lib.mb_launch_count() - l0)
    launches = int(round(launches_total * steps / (max(3, warmup) + 2 * steps + r["soak_steps"])))
    if dump_dir is not None and rank == 0:
        out = Path(dump_dir)
        out.mkdir(parents=True, exist_ok=True)
        np.save(out / "wav.npy", last["wav"].float().cpu().numpy())
        log(f"dumped {out / 'wav.npy'}")
    log(f"resident: soaked {r['ms'] / steps:.3f} ms/step, burst {r['ms_burst'] / steps:.3f}; e2e pass")
    e = ctx.timed(step_e2e, steps, 2, min(soak_s, 1.0), host_clock=True)
    assert produced["n"] == samples_per_step
    ms_step = r["ms"] / steps
    ms_burst = r["ms_burst"] / steps
    value = world * samples_per_step / (ms_step * 1e-3)
    pk = peaks()
    roof = roof_tensor = roof_hbm = None
    step_tf = None
    if rank == 0 and roofline:
        acc = {}
        reps = 3
        for _ in range(reps):
            _, ms_layers = g.forward_profiled(mel_dev)
            for i, t in enumerate(ms_layers):
                info = g.layer_info(i)
                cls = "resblock_conv" if "resblocks" in info else ("ups" if " ups." in info else info.split()[1])
                macs, lbytes = g.layer_work(i, B, T)
                a = acc.setdefault(cls, [0.0, 0.0, 0.0, 0])
                a[0] += t
                a[1] += 2 * macs
                a[2] += lbytes
                a[3] += 1
        dom = max(acc, key=lambda k: acc[k][0])
        t_ms, flops, lbytes, cnt = acc[dom]
        tf = flops / (t_ms * 1e-3) / 1e12
        total_flops = sum(v[1] for v in acc.values()) / reps
        if precision != "fp32":
            mma_mult = 3.0 if precision == "f16x3" else 1.0
            roof_tensor = {"bound": "tensor", "kernel": f"tc_conv / tc_pair ({dom})", "unit": "TFLOP/s",
                           "achieved_soaked": total_flops / (ms_step * 1e-3) / 1e12, "peak_sustained": pk["tflops_sustained"],
                           "frac_soaked": mma_mult * total_flops / (ms_step * 1e-3) / 1e12 / pk["tflops_sustained"],
                           "achieved_burst": total_flops / (ms_burst * 1e-3) / 1e12, "peak_burst": pk["tflops_burst"],
                           "frac_burst": mma_mult * total_flops / (ms_burst * 1e-3) / 1e12 / pk["tflops_burst"],
                           "mma_flops_per_useful_flop": mma_mult, "peak_source": pk["source"] + ", bf16 (fp16 runs at the same rate)",
                           "note": "whole-step useful FLOPs / step time; frac counts the MMA passes really issued"}
            fam = [k for k in acc if k != "conv_post"]
            fam_ms = sum(acc[k][0] for k in fam) / reps
            fam_bytes = sum(acc[k][2] for k in fam) / reps
            fam_launches = sum(acc[k][3] for k in fam) / reps
            traffic = None
            tj = ROOT / "profiles" / "r02_hifigan_dram_traffic.json"
            if tj.exists() and not fre and precision == "f16tc":
                traffic = json.loads(tj.read_text())["tc_dram_bytes_per_launch"]
            gbs = fam_bytes / (fam_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "tc_conv_kernel + tc_pair_kernel (tcgen05 tap convs; all layers but conv_post)",
                    "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "traffic": traffic,
                    "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (profiles/)",
                    "plan_ops_per_step": fam_launches, "algorithmic_bytes_per_op": fam_bytes / max(fam_launches, 1),
                    "algorithmic_bytes_per_step": fam_bytes, "ms_per_step_in_kernel": fam_ms,
                    "share_of_step": fam_ms / ms_step, "peak_source": pk["source"] + ", HBM copy bandwidth",
                    "definition": "layer-granular fp32 bytes (inputs + outputs of every conv layer + weights once, SURVEY.md 8d) / "
                                  "event-timed duration of those launches (profiled pass, no PDL overlap)"}
        else:
            peak = 72.0  # 148 SM x 128 lanes x 2 x ~1.9 GHz FP32 FFMA, nominal
            roof = {"bound": "tensor", "kernel": f"tapconv_f32 ({dom})", "achieved": tf, "peak": peak, "unit": "TFLOP/s",
                    "frac": tf / peak, "traffic": None, "peak_source": "nominal fp32 FFMA (parity-anchor path)",
                    "launches_timed": cnt, "share_of_step": (t_ms / reps) / ms_step}
        step_bytes = sum(v[2] for v in acc.values()) / reps + (68_926_660 if fre else 51_902_980)  # + fp32 weights once
        gbs = step_bytes / (ms_step * 1e-3) / 1e9
        roof_hbm = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                    "achieved_burst": step_bytes / (ms_burst * 1e-3) / 1e9, "bytes_per_step": step_bytes,
                    "definition": "layer-granular fp32 bytes of the whole step (SURVEY.md 8d: 21.61 GB) / step time"}
        step_tf = total_flops / (ms_step * 1e-3) / 1e12
    cpu_d = None
    if rank == 0 and cpu:
        threads = host_threads()
        log(f"cpu baseline on {threads} threads")
        rc = cpu_child(workload, 2, threads, 240.0)
        if rc is not None:
            cpu_d = {"value": rc["value"], "unit": "samples/s", "cores": threads, "kind": "port",
                     "sample": f"2 passes x 32 utterances x 256 frames ({rc['seconds']:.1f} s), torch-CPU oracle "
                               "(bit-identical to the reference forward), batch-1 calls like hifigan/inference.py:66-70"}
    if rank != 0:
        return None
    dtype = {"f16tc": "f16 operands / f32 accumulate (3-term-split serial layers), f32 residual in the full-rate stage",
             "f16x3": "3-term f16 split on tensor cores (FP32-equivalent) / f32 accumulate", "fp32": "f32"}.get(precision, precision)
    return {
        "metric": "vocoder audio samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": steps, "warmup": max(3, warmup), "ms_per_step": ms_step,
        "rtf": (ms_step * 1e-3) / (samples_per_step / 16000.0), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": f"{workload}: Generator fwd, batch 32 x 256 frames x 80 mels per GPU",
                   "per_gpu_batch": B, "frames": T, "precision": precision, "precision_requested": requested,
                   "precision_calibration": g.calibration, "parallelism": f"dp{world}",
                   "l2": "per-step working set (2.9 GB of activations) >> 126 MB L2; no explicit flush",
                   "weights": "random init, torch.manual_seed(0) order of the reference constructor"},
        "burst": {"value": world * samples_per_step / (ms_burst * 1e-3), "ms_per_step": ms_burst, "clocks": r["clocks_burst"]},
        "soak": {"seconds": r["soak_s"], "steps": r["soak_steps"], "clocks": r["clocks_soak"]},
        "e2e": {"value": world * samples_per_step * steps / (e["ms"] * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": B * 80 * T * 4 + B * 4, "d2h_bytes_per_step": samples_per_step * 4,
                "ms_per_step": e["ms"] / steps, "burst_value": world * samples_per_step * steps / (e["ms_burst"] * 1e-3),
                "surface": "vocoder.hifigan.inference.infer_waveforms(list of host numpy mels) -> list of host numpy waveforms"},
        "gpu_launches": launches, "clocks": r["clocks"], "roofline": roof, "roofline_tensor": roof_tensor,
        "roofline_hbm_step": roof_hbm, "step_tflops": step_tf, "cpu_baseline": cpu_d,
    }


def _short(d, keys=("value", "unit", "ms_per_step", "burst", "e2e", "roofline", "cpu_baseline", "config", "dtype", "gpu_launches",
                    "steps", "scaling", "n_gpus")):
    """secondary entries keep the contract's keys, drop the bulk"""
    return None if d is None else {k: d[k] for k in d if k in keys or k.startswith(("value_", "e2e_", "raw_", "mel_", "utter", "stage", "rtf", "us_", "note"))}


def run_ours(args):
    ctx = Ctx()
    try:
        cpu = (not args.no_cpu_baseline) and ctx.world == 1
        if args.workload in ("hifigan_cfg2", "fregan_cfg2"):
            line = measure_hifigan(ctx, args, args.workload, args.precision, args.steps, args.warmup, args.soak_seconds, cpu,
                                   dump_dir=args.dump_outputs)
            secondary = {}
            if args.workload == "hifigan_cfg2" and not args.no_secondary:
                import bench_e2e
                import bench_tacotron
                import bench_wavernn

                def sec(name, fn):
                    try:
                        t0 = time.perf_counter()
                        d = fn()
                        if ctx.rank == 0:
                            secondary[name] = _short(d)
                            log(f"secondary {name}: {time.perf_counter() - t0:.1f} s")
                    except Exception as ex:  # a secondary must never cost the headline line
                        log(f"secondary {name} failed: {ex!r}")
                        if ctx.rank == 0:
                            secondary[name] = {"error": repr(ex)[:300]}

                if ctx.world == 1:
                    sec("hifigan_fp32_equivalent", lambda: measure_hifigan(ctx, args, "hifigan_cfg2", "f16x3", max(3, args.steps // 4),
                                                                         2, 0.5, False, roofline=True))
                    sec("wavernn_cfg1", lambda: bench_wavernn.measure_cfg1(ctx, args, cpu))
                sec("wavernn_cfg3", lambda: bench_wavernn.measure_cfg3(ctx, args, cpu))
                if ctx.world > 1:
                    sec("wavernn_cfg3_fold_sharded", lambda: bench_wavernn.measure_cfg3_sharded(ctx, args))
                sec("tacotron_cfg4", lambda: bench_tacotron.measure(ctx, args, cpu, steps=3))
                sec("e2e_cfg5", lambda: bench_e2e.measure(ctx, args, cpu, steps=2))
                sec("e2e_cfg5_strong_1024", lambda: bench_e2e.measure(ctx, args, False, steps=1, strong_total=1024))
            if ctx.rank == 0:
                if secondary:
                    line["secondary"] = secondary
                print(json.dumps(line), flush=True)
        else:
            import bench_e2e
            import bench_tacotron
            import bench_wavernn

            fn = {"wavernn_cfg1": lambda: bench_wavernn.measure_cfg1(ctx, args, cpu, steps=args.steps),
                  "wavernn_cfg3": lambda: bench_wavernn.measure_cfg3(ctx, args, cpu, steps=args.steps),
                  "tacotron_cfg4": lambda: bench_tacotron.measure(ctx, args, cpu, steps=args.steps),
                  "e2e_cfg5": lambda: bench_e2e.measure(ctx, args, cpu, steps=args.steps)}[args.workload]
            line = fn()
            if ctx.rank == 0:
                print(json.dumps(line), flush=True)
    finally:
        ctx.close()


def main():
    args = parse()
    if args.cpu_child is not None:
        workload, amount, threads = args.cpu_child[0], int(args.cpu_child[1]), int(args.cpu_child[2])
        if workload in ("hifigan_cfg2", "fregan_cfg2"):
            v, dt, n = cpu_hifigan(32, amount, threads, fregan=(workload == "fregan_cfg2"))
        elif workload == "tacotron_cfg4":
            import bench_tacotron

            v, dt = bench_tacotron.cpu_oracle(amount, threads)
        elif workload == "e2e_cfg5":
            import bench_e2e

            v, dt = bench_e2e.cpu_oracle(amount, threads)
        else:
            import bench_wavernn

            v, dt = bench_wavernn.cpu_torch_oracle(workload, amount, threads)
        print(json.dumps({"value": v, "seconds": dt}))
        return
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    main()
