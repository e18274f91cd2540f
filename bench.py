#!/usr/bin/env python
"""bench.py — novel views/sec of the ViewFormer hot path on B200 (BASELINE.json metric, config 2).

One "step" = one pass of generate() over a batch of synthetic scenes:
    uint8 images [B, 10, 128, 128, 3] + cameras [B, 10, 7]
      -> VQ-encode the 9 context views -> MIGT forward (mask tokens in view 10) -> argmax -> VQ-decode
      -> uint8 novel view [B, 128, 128, 3]                     (evaluate/evaluate_transformer.py:97-146)
B = 32 scenes per GPU (BASELINE.json configs[1]); N GPUs run N independent shards (weak scaling, no collective on
the data path — scenes are independent).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...     # the reference algorithm on the host CPU cores (torch-CPU oracle)

Prints ONE JSON line (rank 0).  `value` = views/s with inputs resident in HBM; `e2e` = same metric through the public
generate() call with pinned-host inputs, H2D/D2H inside the timed region; `roofline` = the dominant kernel
(tcgen05 implicit-GEMM 3x3 conv 128->128 @128x128) timed alone with CUDA events against the measured bf16 peak;
`cpu_baseline` = the oracle timed on a bounded sample on this box's host cores.
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

import torch  # noqa: E402

N_CTX = 9
T_VIEWS = N_CTX + 1
IMG = 128
WORKLOAD = ("interiornet-transformer generate(), 9 context views, batch 32 scenes per GPU (BASELINE configs[1]): "
            "uint8 images -> VQ-encode 9 ctx -> MIGT -> argmax -> VQ-decode -> uint8 view")     # identical in both arms


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scenes", type=int, default=32, help="scenes per GPU per step")
    ap.add_argument("--precision", default="mixed", choices=["mixed", "bf16", "tf32", "fp32"],
                    help="mixed (headline) = fp32-faithful encoder (bit-exact codebook indices) + bf16 tensor-core transformer / decoder; "
                         "bf16 / tf32 = everything on the tensor-core path in that operand type; fp32 = exact CUDA-core path")
    ap.add_argument("--also", default=None, help="comma list of further precisions timed for the side-by-side `value_by_precision` "
                                                 "(default at N=1: the other three; at N>1: none)")
    ap.add_argument("--cpu-scenes", type=int, default=2, help="scenes in the bounded CPU-baseline sample")
    ap.add_argument("--cpu-budget-s", type=float, default=75.0, help="wall-time budget of the --impl reference arm (warm-up + steps)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity block")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying the captured CUDA graph")
    ap.add_argument("--workload", default="generate", choices=["generate", "kvcache", "train"],
                    help="generate = BASELINE configs[1] (default, the judged line); kvcache = configs[4]: 19-context KV-cached query decode; "
                         "train = configs[3]: codebook training step (--scenes = images per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (generate workload, rank 0) as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "generate" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the generate workload of --impl b200")
    return args


# ------------------------------------------------------------------------------------------------- helpers
def synth_inputs(n_scenes, seed):
    g = torch.Generator().manual_seed(seed)
    lo = torch.rand((n_scenes * T_VIEWS, 3, IMG // 8, IMG // 8), generator=g)
    x = torch.nn.functional.interpolate(lo, size=(IMG, IMG), mode="bilinear", align_corners=False)
    x = x + 0.08 * torch.randn(x.shape, generator=g)
    images = (x.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).reshape(n_scenes, T_VIEWS, IMG, IMG, 3).contiguous()
    xyz = torch.randn((n_scenes, T_VIEWS, 3), generator=g)
    q = torch.randn((n_scenes, T_VIEWS, 4), generator=g)
    q = q / q.norm(dim=-1, keepdim=True)
    q = q * torch.where(q[..., :1] >= 0, 1.0, -1.0)
    return images, torch.cat([xyz, q], -1).contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def count_in(self, t0, t1):
        return sum(1 for t, _ in self.rows if t0 <= t <= t1)

    def stop(self, windows):
        """windows: [(t0, t1)] monotonic intervals during which the GPU ran the measured step; only samples read inside
        them count (nvidia-smi is started before the warm-up so that it is already streaming when the timed region begins)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for t, r in self.rows:
            if not any(t0 <= t <= t1 for t0, t1 in windows):
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, outputs):
    """Every tensor of ``outputs`` (all indexed by scene first) as <path>/<name>.npy in float32: uint8 pixels, codebook indices and
    cameras are exact in float32.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the scenes is written, the same for every name."""
    import numpy as np
    arrays = {k: v.detach().float().cpu() for k, v in outputs.items() if torch.is_tensor(v)}
    n = next(iter(arrays.values())).shape[0]
    per_scene = sum(a[0].numel() * 4 for a in arrays.values())
    keep = min(n, DUMP_LIMIT_BYTES // per_scene)
    rows = torch.arange(n) if keep == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a[rows].numpy())


def ncu_traffic(rel_path, scale, what="288 images/launch"):
    """dram__bytes_read.sum + dram__bytes_write.sum of the roofline kernel from the committed `ncu --set full` capture (metric dump
    under profiles/), scaled by the launch's image count.  Read from the file, not a literal; None when the capture is absent."""
    path = os.path.join(ROOT, rel_path)
    if not os.path.exists(path):
        return None, "no capture committed"
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for line in open(path):
        f = [c.strip().strip('"') for c in line.rstrip("\n").split(",")]
        if f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and len(f) >= 3 and f[1] in unit:
            tot += float(f[2]) * unit[f[1]]
    return (tot * scale if tot else None), f"{rel_path} (ncu --set full of this kernel, {what}) x {scale:.3f}"


# ------------------------------------------------------------------------------------------------- reference arm (CPU)
def cpu_threads():
    """All 100+ logical CPUs of the GPU box oversubscribe oneDNN/MKL (measured in round 1: 16-32 threads are fastest)."""
    return max(1, min(32, os.cpu_count() or 1))


class CpuReference:
    """The reference's algorithm on the host cores (oracle restatement; the real torch/TF reference cannot travel to the GPU box):
    generate_batch_predictions with 10 encodes + dense masked attention + full-sequence LM head, as the reference executes them
    (evaluate_transformer.py:97-146).  Every call is ONE scene-batch; callers bound the number of calls by wall time."""

    def __init__(self, vq_sd, migt_sd, vcfg, tcfg):
        from oracle import vqgan_oracle as vo, migt_oracle as mo
        self.mo = mo
        self.tcfg = tcfg
        self.cores = cpu_threads()
        torch.set_num_threads(self.cores)
        self.fwd = lambda d: mo.forward(migt_sd, tcfg, d, use_localization=False)
        self.enc = lambda x: vo.encode(vq_sd, vcfg, x)[2]
        self.dec = lambda c: vo.decode_code(vq_sd, vcfg, c)

    def __call__(self, images, cams):
        with torch.no_grad():
            t0 = time.perf_counter()
            out = self.mo.generate_batch_predictions(self.fwd, self.enc, self.dec, self.tcfg, images, cams, use_localization=False)
            return out, time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from viewformer_b200.config import VQGANConfig, MIGTConfig
    from oracle import synth
    vcfg, tcfg = VQGANConfig(), MIGTConfig(localization_weight="0")
    vq_sd, migt_sd = synth.make_vqgan_state_dict(vcfg, 0), synth.make_migt_state_dict(tcfg, 0)
    ref = CpuReference(vq_sd, migt_sd, vcfg, tcfg)
    n = 1                                            # scenes per step: a bounded sample of the 32-scene workload
    images, cams = synth_inputs(max(n, 2), 777)
    t_start = time.perf_counter()
    warm = min(args.warmup, 1)
    for _ in range(warm):
        ref(images[:n], cams[:n])
    times = []
    for i in range(args.steps):
        _, dt = ref(images[:n], cams[:n])
        times.append(dt)
        if time.perf_counter() - t_start + dt > args.cpu_budget_s:      # the next step would not fit the wall-time budget
            break
    total = sum(times)
    vps, sec = n * len(times) / total, total / len(times)
    sample = (f"{n} scene x {T_VIEWS} views per step (bounded sample of the {args.scenes}-scene workload), {len(times)} of {args.steps} requested steps "
              f"inside the {args.cpu_budget_s:.0f} s wall budget, torch-CPU fp32 oracle of the reference algorithm")
    print(json.dumps({
        "impl": "reference", "metric": "novel views/sec (128x128, 9-ctx)", "value": vps, "unit": "views/s", "n_gpus": args.gpus,
        "steps": len(times), "steps_requested": args.steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "precision": "fp32", "scenes_per_step": n, "views": T_VIEWS, "image": IMG, "localization": False,
                   "encodes_per_scene": "10 (the reference encodes the target view too, evaluate_transformer.py:109-116)",
                   "sample": f"bounded sample: {n} of the workload's {args.scenes} scenes per step"},
        "cpu_baseline": {"value": vps, "unit": "views/s", "cores": ref.cores, "kind": "port", "sample": sample},
        "e2e": {"value": vps, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------- B200 arm
def model_pair(precision, vcfg, tcfg, dev, seed=0):
    """(codebook, transformer) of one precision mode.  ``mixed`` pairs the exact-encoder VQGAN with the bf16 transformer."""
    from viewformer_b200 import VQGAN, MIGT
    codebook = VQGAN(vcfg, precision=precision, device=dev).init_weights(seed)
    transformer = MIGT(tcfg, precision="bf16" if precision == "mixed" else precision, device=dev).init_weights(seed)
    return codebook, transformer


def parity_block(codebook, transformer, out_timed, images_d, cams_d, vcfg, tcfg, dev):
    """Outside the timed region, on the bench's own inputs: the timed mode against the exact fp32 CUDA-core path.
    (a) encoder codes of all scenes (bit-exact bar), (b) transformer argmax on identical context codes, (c) decoded uint8 pixels
    on identical codes, (d) the whole timed pipeline's generated codes against the exact pipeline's."""
    from viewformer_b200 import VQGAN, MIGT, _lib
    B = images_d.shape[0]
    xvq = VQGAN(vcfg, precision="fp32", device=dev).load_state_dict(codebook.state_dict())
    xtr = MIGT(tcfg, precision="fp32", device=dev).load_state_dict(transformer.state_dict())
    codes_t = codebook.encode_u8(images_d, first_views=N_CTX)
    codes_x = xvq.encode_u8(images_d, first_views=N_CTX)
    cams, _ = _lib.cameras_prepare(cams_d.contiguous(), tcfg.augment_poses == "relative")
    ctx = codes_x.reshape(B, N_CTX, 8, 8)
    gen_t = transformer.generate_codes(ctx, cams)
    gen_x = xtr.generate_codes(ctx, cams)
    px_t = codebook.decode_code_u8(gen_x).int()
    px_x = xvq.decode_code_u8(gen_x).int()
    torch.cuda.synchronize()
    pd = (px_t - px_x).abs()
    blk = {
        "reference_path": "fp32 CUDA-core path (vf_simt_gemm / exact kernels; bit-exact against the CPU oracle in tests/)",
        "code_mismatches": int((codes_t != codes_x).sum()), "codes_compared": int(codes_x.numel()),
        "generated_code_mismatches_same_context": int((gen_t != gen_x).sum()), "generated_codes_compared": int(gen_x.numel()),
        "pixel_max_abs_diff_u8_same_codes": int(pd.max()), "pixel_mean_abs_diff_u8_same_codes": float(pd.float().mean()),
        "pipeline_generated_code_mismatches": int((out_timed["generated_codes"] != gen_x).sum()),
    }
    del xvq, xtr
    return blk, codes_x


def run_b200(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    from viewformer_b200 import generate_batch_predictions, _lib
    from viewformer_b200.config import VQGANConfig, MIGTConfig
    vcfg, tcfg = VQGANConfig(), MIGTConfig(localization_weight="0")
    codebook, transformer = model_pair(args.precision, vcfg, tcfg, dev)

    B = args.scenes
    images_h, cams_h = synth_inputs(B, 1234 + rank)
    images_pin, cams_pin = images_h.pin_memory(), cams_h.pin_memory()
    images_d, cams_d = images_h.to(dev), cams_h.to(dev)
    out_pin = torch.empty((B, IMG, IMG, 3), dtype=torch.uint8).pin_memory()

    def make_steps(cb, tr):
        graphed, note = None, "eager"
        if not args.no_graph and not tr.use_localization:
            from viewformer_b200 import GraphedPredictions
            try:
                graphed = GraphedPredictions(tr, cb, B, T_VIEWS)          # capture once; every step is one graph replay
                note = "cuda graph replay (GraphedPredictions)"
            except Exception as e:                                        # same kernels either way: only the launch mode changes
                print(f"[bench] CUDA graph capture failed ({e!r}); launching eagerly", file=sys.stderr)
                torch.cuda.synchronize()
                note = "eager (graph capture failed)"

        def resident():
            if graphed is not None:
                return graphed(images_d, cams_d)              # device -> static device buffers (15.7 MB d2d) + replay
            return generate_batch_predictions(tr, cb, images_d, cams_d)

        def e2e():
            if graphed is not None:
                r = graphed(images_pin, cams_pin)             # pinned host -> static device buffers + replay
            else:
                r = generate_batch_predictions(tr, cb, images_pin.to(dev, non_blocking=True), cams_pin.to(dev, non_blocking=True))
            out_pin.copy_(r["generated_images"], non_blocking=True)
            return r
        return resident, e2e, graphed, note

    step_resident, step_e2e, graphed, graph_note = make_steps(codebook, transformer)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(ms of `steps` calls of fn, what the last call returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step_resident()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step_resident()                      # host-side enqueue time of one step (launch-bound check), not part of the timed region
    host_ms = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    w0 = time.monotonic()
    ms_total, last = timed(step_resident, args.steps)
    # the graph's outputs are static buffers that the next replay overwrites: keep the last timed step's
    out_timed = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in last.items()}
    windows = [(w0, time.monotonic())]
    launches = _lib.launch_count() if graphed is None else graphed.launches_per_replay * args.steps
    clock_note = "timed region"
    if rank == 0 and sampler.proc is not None and sampler.count_in(*windows[0]) < 3:
        # a short timed region (K steps of ~30 ms) can end between two 100 ms nvidia-smi samples: keep the GPU on the
        # identical step for ~1.5 s more (untimed) so that the clocks / throttle reasons under this load are observed
        w1 = time.monotonic()
        while time.monotonic() - w1 < 1.5:
            step_resident()
            torch.cuda.synchronize()
        windows.append((w1, time.monotonic()))
        clock_note = "timed region + 1.5 s of the identical step right after it (region shorter than the sampling period)"
    clocks = sampler.stop(windows) if rank == 0 else None
    if clocks is not None:
        clocks["sampled"] = clock_note
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    torch.cuda.synchronize()

    views = world * B * args.steps
    value = views / (ms_total / 1e3)
    e2e_value = views / (ms_e2e / 1e3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out_timed)

    # ---- in-run parity of the timed mode (rank 0, outside the timed region)
    parity, codes_exact = None, None
    if not args.no_parity:
        parity, codes_exact = parity_block(codebook, transformer, out_timed, images_d, cams_d, vcfg, tcfg, dev)

    # ---- the other precisions, side by side (same inputs, same step, `steps` timed replays each)
    also = args.also if args.also is not None else (",".join(p for p in ("bf16", "tf32", "fp32") if p != args.precision) if world == 1 else "")
    by_prec = {args.precision: {"value": value / world, "ms_per_step": ms_total / args.steps,
                                "code_mismatches_vs_fp32": None if parity is None else parity["code_mismatches"]}}
    if world == 1:
        for pname in [x for x in also.split(",") if x]:
            cb2, tr2 = model_pair(pname, vcfg, tcfg, dev)
            res2, _, g2, _ = make_steps(cb2, tr2)
            for _ in range(3):
                res2()
            ms2, _ = timed(res2, args.steps)
            entry = {"value": B * args.steps / (ms2 / 1e3), "ms_per_step": ms2 / args.steps, "steps": args.steps}
            if codes_exact is not None:
                entry["code_mismatches_vs_fp32"] = int((cb2.encode_u8(images_d, first_views=N_CTX) != codes_exact).sum())
            by_prec[pname] = entry
            del cb2, tr2, res2, g2
            torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel: the 3x3 conv 128->128 @128x128 of the encoder (288 images per launch).
    # mixed / x3: the exact split-fp16 kernel — three fp16 MMA passes per product, so the tensor pipe executes 3x the convolution's
    # algorithmic FLOPs; `achieved` is the ALGORITHMIC rate (contract), `achieved_executed_mma` what the pipe actually does.
    peak_tf, peak_hbm, peak_src = measured_peaks()
    n_img = B * N_CTX
    exact = args.precision in ("mixed", "x3")

    def time_launch(fn, reps=5):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps

    xf = torch.randn((n_img, IMG, IMG, 128), device=dev)
    wf = torch.randn((128 * 9, 128), device=dev) / 34.0
    b = torch.zeros(128, device=dev)
    o = torch.empty((n_img, IMG, IMG, 128), device=dev)
    if exact:
        x = _lib.groupnorm(xf, None, None, swish=False, out_dtype=torch.float16, normalize=False)
        w = _lib.split_f16x2(wf).reshape(128, 18 * 128)
    else:
        x, w = xf.to(torch.bfloat16), wf.reshape(128, 9 * 128).to(torch.bfloat16)
    del xf
    sec = time_launch(lambda: _lib.tc_conv(x, w, b, out=o))
    flops = 2.0 * n_img * IMG * IMG * 128 * 9 * 128          # SURVEY §8(d): 2*M*N*K of the implicit GEMM
    passes = 3 if exact else 1
    ach = passes * flops / sec / 1e12
    cap = "profiles/r02_exact_conv_wide_ncu_metrics.csv" if exact else "profiles/r01_conv_wide_ncu_nores_metrics.csv"
    traffic, traffic_src = ncu_traffic(cap, n_img / 288.0)
    roof = {"kernel": ("tc_conv3x3_wide_kernel<exact>: persistent tcgen05 implicit GEMM on split-fp16 operands (3 MMA passes, chunked accumulation), "
                       if exact else "tc_conv3x3_wide_kernel: persistent tcgen05 implicit GEMM, ") +
                      "128 channels x 256 pixels per tile (3x3 conv 128->128 @128x128, %d images/launch)" % n_img,
            # `achieved` / `frac`: ALGORITHMIC flops of the convolution (2*M*N*K) over the launch time, as the contract defines them.  The
            # exact mode spends three fp16 MMA passes per algorithmic flop to return fp32-faithful results: `achieved_executed_mma` /
            # `frac_executed_mma` say how busy the tensor pipe actually is (the number to compare with ncu's sm__pipe_tc_cycles_active).
            "bound": "tensor", "achieved": flops / sec / 1e12, "peak": peak_tf, "unit": "TFLOP/s", "frac": flops / sec / 1e12 / peak_tf,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "launch_ms": sec * 1e3, "mma_passes": passes,
            "achieved_executed_mma": ach, "frac_executed_mma": ach / peak_tf,
            "algorithmic_flops_per_launch": flops,
            "algorithmic_bytes_per_launch": n_img * IMG * IMG * 128 * ((4 if exact else 2) + 4)}
    del x, w, o

    # ---- second roofline entry: the codebook lookup (HBM-bound by the north_star: 1032 algorithmic bytes per token)
    Mvq = 1 << 20
    q = codebook._w["q"]
    zq = torch.randn((Mvq, q["et"].shape[1]), device=dev)
    roof_vq = None
    if q.get("eh") is not None:
        sec_vq = time_launch(lambda: _lib.vq_lookup_fused(zq, q["et"], q["esq"], q["eh"], emb_dk=q["emb"], want_quant=False, want_diff=False), reps=3)
        ach_vq = Mvq * (q["et"].shape[1] * 4 + 8) / sec_vq / 1e9
        tr_vq, tr_vq_src = ncu_traffic("profiles/r02_vq_fused_ncu_metrics.csv", 1.0, "vq_lookup_fused_kernel at M = 2^20; the exact pass adds 0.03 GB")
        roof_vq = {"kernel": "vq_lookup_fused_kernel + vq_rescue_kernel: fp16 distance GEMM on CTA pairs, top-2 from TMEM, fp64 settlement of near-ties "
                             "(z ~ N(0,1) [2^20, 256] fp32 -> int64 indices, K = 1024)",
                   "bound": "hbm", "achieved": ach_vq, "peak": peak_hbm, "unit": "GB/s", "frac": ach_vq / peak_hbm, "traffic": tr_vq,
                   "traffic_source": tr_vq_src, "peak_source": peak_src, "launch_ms": sec_vq * 1e3,
                   "algorithmic_bytes_per_launch": Mvq * (q["et"].shape[1] * 4 + 8)}
    del zq

    # ---- CPU baseline: the oracle on the first scenes of THIS run's inputs; its outputs double as a parity check of the timed pipeline
    cpu = None
    if not args.no_cpu_baseline and world == 1:      # reported on rank 0 at N = 1 only
        ref = CpuReference(codebook.state_dict(), transformer.state_dict(), vcfg, tcfg)
        n = max(1, min(args.cpu_scenes, B))
        ref(images_h[:1], cams_h[:1])                                 # warm-up: one scene
        want, dt = ref(images_h[:n], cams_h[:n])
        cpu = {"value": n / dt, "unit": "views/s", "cores": ref.cores, "kind": "port",
               "sample": f"the first {n} of the {B} bench scenes x {T_VIEWS} views, 1 timed pass after a 1-scene warm-up, {ref.cores} threads, torch-CPU fp32 "
                         f"oracle of the reference algorithm (10 encodes, dense masked attention, full LM head)"}
        if parity is not None:
            got_codes = codebook.encode_u8(images_d[:n].contiguous(), first_views=N_CTX).reshape(n, N_CTX, 8, 8).cpu()
            parity["oracle_scenes"] = n
            parity["oracle_code_mismatches"] = int((got_codes != want["codes"][:, :N_CTX]).sum())
            parity["oracle_codes_compared"] = int(got_codes.numel())
            parity["oracle_generated_code_mismatches"] = int((out_timed["generated_codes"][:n].cpu() != want["generated_codes"]).sum())
            # decoder against the oracle on IDENTICAL codes (the oracle's own generated codes), so that a flipped argmax of two
            # near-tied logits in the bf16 transformer does not show up as a pixel difference
            pdiff = (codebook.decode_code_u8(want["generated_codes"].to(dev)).cpu().int() - want["generated_images"].int()).abs()
            parity["oracle_pixel_max_abs_diff_u8_same_codes"] = int(pdiff.max())
            parity["oracle_pixel_mean_abs_diff_u8_same_codes"] = float(pdiff.float().mean())

    in_bytes = images_pin.numel() + cams_pin.numel() * 4
    print(json.dumps({
        "metric": "novel views/sec (128x128, 9-ctx)", "value": value, "unit": "views/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {"mixed": "f32 encoder (bit-exact codes) + bf16 transformer/decoder"}.get(args.precision, args.precision),
        "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "precision": args.precision, "scenes_per_gpu": B, "views": T_VIEWS, "image": IMG, "localization": False,
                   "parallelism": f"dp{world} (independent shards)",
                   "encodes_per_scene": "9 (the reference also encodes the target view and discards it; cpu_baseline runs the reference's 10)",
                   "l2": "inputs larger than L2 (15.7 MB images + >2 GB activations per step); no flush needed"},
        "e2e": {"value": e2e_value, "unit": "views/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": int(in_bytes),
                "d2h_bytes_per_step": int(out_pin.numel())},
        "gpu_launches": launches // max(1, args.steps), "launch_mode": graph_note,
        "host_enqueue_ms_per_step": host_ms,
        "clocks": clocks,
        "parity": parity,
        "value_by_precision": by_prec,
        "roofline": roof,
        "roofline_vq_lookup": roof_vq,
        "cpu_baseline": cpu,
    }))
    if world > 1:
        dist.destroy_process_group()


def run_kvcache(args):
    """BASELINE configs[4]: transformer decode with a context KV cache — 19 context views prefilled once per scene,
    every step answers one query view per scene (64 mask tokens against the cached K/V^T).  Transformer only."""
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    from viewformer_b200 import MIGT, _lib
    from viewformer_b200.config import MIGTConfig
    tr = MIGT(MIGTConfig(localization_weight="0"), precision=args.precision, device=dev).init_weights(0)
    B, Tc = args.scenes, 19
    g = torch.Generator().manual_seed(99 + rank)
    codes = torch.randint(0, 1024, (B, Tc, 8, 8), generator=g).to(dev)
    _, cams = synth_inputs(B, 5 + rank)
    cams = torch.cat([cams, cams], 1)[:, :Tc + 1].contiguous().to(dev)
    cams, _ = _lib.cameras_prepare(cams, True)
    ctx_p, qry_p = cams[:, :Tc].contiguous(), cams[:, Tc].contiguous()

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cache = tr.prefill_context(codes, ctx_p)
    sync(); e0.record(); cache = tr.prefill_context(codes, ctx_p); e1.record(); sync()
    prefill_ms = e0.elapsed_time(e1)
    for _ in range(max(3, args.warmup)):
        tr.query(cache, qry_p)
    sync(); e0.record()
    for _ in range(args.steps):
        tr.query(cache, qry_p)
    e1.record(); sync()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(json.dumps({"metric": "novel views/sec (KV-cached transformer decode, 19-ctx)", "value": world * B * args.steps / (float(ms) / 1e3),
                          "unit": "views/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                          "ms_per_step": float(ms) / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": args.precision, "data": "synthetic",
                          "config": {"workload": "co3d-all transformer decode w/ KV-cache, 19 ctx views (BASELINE configs[4])",
                                     "scenes_per_gpu": B, "prefill_ms": prefill_ms}}))
    if world > 1:
        dist.destroy_process_group()


def run_train(args):
    """BASELINE configs[3]: codebook training step — forward, backward, bucketed NCCL gradient all-reduce under backward, packed
    EMA-statistics all-reduce, Adam — on `--scenes` images per GPU (32 = 256 images over 8 GPUs).  fp32 results as the reference requires
    (vqgan_th.py:326); the 3x3 convs run on the exact split-fp16 tensor-core kernels.  One step = one optimisation step; the batch is
    copied from pinned host memory inside the timed region."""
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    from viewformer_b200 import VQGAN
    from viewformer_b200.config import VQGANConfig
    from viewformer_b200.train import VQGANTrainer
    tr = VQGANTrainer(VQGAN(VQGANConfig(perceptual_weight=0.0), precision="fp32", device=dev).init_weights(0))
    n = args.scenes
    x = (torch.rand((n, 3, IMG, IMG), generator=torch.Generator().manual_seed(7 + rank)) * 2 - 1).pin_memory()

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        loss = tr.training_step(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync(); e0.record()
    for _ in range(args.steps):
        loss = tr.training_step(x)
    e1.record(); sync()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(json.dumps({"metric": "codebook training images/sec", "value": world * n * args.steps / (float(ms) / 1e3), "unit": "images/s",
                          "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": float(ms) / args.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (exact split-fp16 tensor-core convs)",
                          "data": "synthetic", "loss": float(loss),
                          "config": {"workload": "shapenet-srn codebook training step (BASELINE configs[3])", "images_per_gpu": n,
                                     "gradient_buckets": len(tr.buckets), "h2d_bytes_per_step": x.numel() * 4}}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.workload == "train" and a.impl == "b200":
        run_train(a)
    elif a.workload == "kvcache" and a.impl == "b200":
        run_kvcache(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
