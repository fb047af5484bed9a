#!/usr/bin/env python
"""bench.py — the video->text prefill path of VideoLLaMA2-7B (16 frames @336, 256-token prompt) on B200.

  python bench.py --gpus N --steps K --warmup W            our arm (libvl2 sm_100a kernels)
  python bench.py --impl reference ...                      the reference's own PyTorch-CPU path (oracle port), rank 0 only

A "step" is one pass of the hot path over one video: pixels + prompt ids -> ViT -> STC connector -> splice -> decoder
prefill -> last-position logits.  `value` = prefill tokens/s of the WHOLE job with inputs resident in HBM
(S tokens x N videos / step time; N ranks run N independent videos: weak scaling, no data-path collective);
`e2e` = the same through the public API (model.generate(..., max_new_tokens=1)) from pinned HOST buffers with the
H2D copy of the frames and the D2H read of the result inside the timed region.  `frame_parallel` reports the
frame-sharded ViT + NCCL all-gather stage (strong scaling of one video's vision stage) when N > 1.
One JSON line on stdout (rank 0).  Nothing here reads /root/reference.
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
sys.dont_write_bytecode = True      # a run leaves the tree as it found it (it may be read-only)

METRIC = "video-frames/sec + prefill tokens/sec (VideoLLaMA2-7B, 16f@336) at 1/2/4/8 B200"
FRAMES, PROMPT = 16, 256
WORKLOAD = ("VideoLLaMA2-7B ({model}) 16 frames@{img} + 256-token prompt -> S={S} prefill, last-position logits; "
            "one video per GPU")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"], "hbm_gbs": d["hbm_gbs"],
                "src": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for n, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle's port of the reference path (bf16, SDPA like the reference's HF modules on
# CPU), the WHOLE config-2 step measured piece by piece - nothing is extrapolated
# ------------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU baseline may use: min(scheduler affinity, cgroup CPU quota, physical cores).  os.cpu_count() alone
    oversubscribes a container whose cgroup quota is smaller than the host (round 1: one ViT frame took 46 s on '128'
    threads of a quota-limited box) and hyper-thread siblings only slow oneDNN GEMMs down."""
    info = {"os_cpu_count": os.cpu_count() or 1}
    n = info["os_cpu_count"]
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
        n = min(n, info["affinity"])
    except Exception:
        pass
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        info["cgroup_quota_cpus"] = quota
        n = min(n, max(1, int(quota)))
    try:
        cores = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    cores.add((phys, core))
                phys = core = None
        if cores:
            info["physical_cores"] = len(cores)
            n = min(n, len(cores))
    except Exception:
        pass
    info["threads"] = max(1, n)
    return info


def cpu_reference_step(n_steps: int = 1, budget_s: float = 150.0):
    """One WHOLE config-2 step (16 frames through the 23 consumed ViT layers, the STC connector, the splice, 32 decoder
    layers at S=1776, the last-position head) of the oracle's restatement of the reference path on the host cores:
    bf16 like the reference's HF modules, F.scaled_dot_product_attention like HF's CPU attention backend.  The 7B
    synthetic checkpoint is generated stage by stage OUTSIDE the timed windows (so 16 GB never sit in host memory) and
    every piece of the step is executed and timed; the step time is the sum of the measured pieces.  Repeats while the
    wall-clock budget allows and reports the spread."""
    import torch
    import torch.nn.functional as F
    from oracle import synth, torch_ref
    th = host_threads()
    torch.set_num_threads(th["threads"])
    cfg = synth.CONFIGS["cfg2"]
    dt = torch.bfloat16
    px, ids = synth.inputs(cfg)
    v, l = cfg.vision, cfg.llm
    steps = []
    t_start = time.perf_counter()

    def timed(fn):
        t = time.perf_counter()
        out = fn()
        return out, time.perf_counter() - t

    with torch.no_grad():
        while len(steps) < max(1, n_steps):
            sd = dict(synth.iter_state(synth.vision_specs(v)))
            feats, t_vit = timed(lambda: torch_ref.vit_features(sd, v, px, cfg.select_layer, dt, sdpa=True))
            sd = dict(synth.iter_state(synth.stc_specs(v.hidden, l.hidden)))
            mm, t_stc = timed(lambda: torch_ref.stc_forward(sd, feats[None], cfg.stc_pad, cfg.stc_depth, dt))
            table = synth.make_tensor("model.embed_tokens.weight", (l.vocab, l.hidden), "emb")
            h, t_splice = timed(lambda: torch_ref.splice_embeddings(ids[0], table, mm[0]))
            del table, sd
            cos, sin = torch_ref.rope_cos_sin(cfg.seq, l.head_dim, l.theta, dt)
            t_layers = []
            for i in range(l.layers):
                sd = dict(synth.iter_state(synth.llm_layer_specs(l, i)))
                h, t = timed(lambda: torch_ref.decoder_layer(sd, l, i, h, cos, sin, dt, sdpa=True))
                t_layers.append(t)
            del sd
            norm = synth.make_tensor("model.norm.weight", (l.hidden,), "gain")
            head = synth.make_tensor("lm_head.weight", (l.vocab, l.hidden), "w")
            _, t_head = timed(lambda: F.linear(torch_ref.rmsnorm(h[-1:], norm, l.eps), head))
            del head
            t_vis = t_vit + t_stc
            t_llm = sum(t_layers) + t_head
            steps.append({"t_all_s": t_vis + t_splice + t_llm, "t_vit_s": t_vit, "t_stc_s": t_stc, "t_llm_s": t_llm,
                          "t_layer_min_s": min(t_layers), "t_layer_max_s": max(t_layers)})
            elapsed = time.perf_counter() - t_start
            if elapsed + elapsed / len(steps) > budget_s:
                break
    alls = sorted(x["t_all_s"] for x in steps)
    med = steps[[x["t_all_s"] for x in steps].index(alls[len(alls) // 2])]
    t_all = med["t_all_s"]
    t_vis = med["t_vit_s"] + med["t_stc_s"]
    return {"t_all_s": t_all, "t_vis_s": t_vis, "t_llm_s": med["t_llm_s"], "tok_per_s": cfg.seq / t_all,
            "frames_per_s": cfg.frames / t_vis, "llm_tok_per_s": cfg.seq / med["t_llm_s"], "cores": th["threads"],
            "steps_run": len(steps), "t_all_min_s": alls[0], "t_all_max_s": alls[-1], "host": th,
            "wall_s": time.perf_counter() - t_start,
            "sample": f"{len(steps)} whole config-2 step(s), every stage executed and timed (16 frames x 23 ViT layers "
                      f"{med['t_vit_s']:.1f}s, STC {med['t_stc_s']:.1f}s, 32 decoder layers at S={cfg.seq} + last-row head "
                      f"{med['t_llm_s']:.1f}s; per-layer {med['t_layer_min_s']:.2f}-{med['t_layer_max_s']:.2f}s); bf16, SDPA, "
                      f"{th['threads']} threads (os.cpu_count {th['os_cpu_count']}); weights generated outside the timed windows; "
                      f"spread over steps {alls[0]:.1f}-{alls[-1]:.1f}s"}


def run_reference(args, rank: int):
    if rank != 0:
        return
    # every step is a whole config-2 step of the port (tens of seconds of CPU work): run as many of the requested steps as
    # fit a few minutes and report how many were run - `steps` and `ms_per_step` describe what was actually measured
    r = cpu_reference_step(n_steps=max(1, args.steps), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["tok_per_s"], "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": r["steps_run"], "warmup": 0, "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": r["t_all_s"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(model="mistral7b", img=336, S=1776), "frames": FRAMES, "prompt": PROMPT,
                   "seq": 1776, "note": "reference algorithm (oracle port: bf16, SDPA) on the host CPU, whole steps, no extrapolation"},
        "frames_per_s": r["frames_per_s"], "llm_prefill_tok_per_s": r["llm_tok_per_s"],
        "cpu_baseline": {"value": r["tok_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                         "spread_s": [r["t_all_min_s"], r["t_all_max_s"]], "host": r["host"]},
        "e2e": {"value": r["tok_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[4]: VideoLLaMA2-72B (Qwen2-72B) decoder, tensor-parallel over the ranks of one box
# ------------------------------------------------------------------------------------------------------------------
def bench_tp72b(args, rank, world, dev):
    """Decoder prefill of the 72B geometry (80 layers, H 8192, I 29568, 64q/8kv heads) sharded tensor-parallel over `world`
    GPUs (model/tp_decoder.py), S = 1776 synthetic input embeddings -> last-position logits: whole-job prefill tokens/s, the
    tensor roofline fraction per GPU and the all-reduce share of the step (the same step timed with the collectives skipped).
    `e2e`: the whole BASELINE configuration - pixels + ids -> token through generate(): CLIP tower and the connector's first
    RegStage sharded by frame over the ranks, one all-gather, the 8192-wide connector tail, then the tensor-parallel decoder."""
    import torch
    import torch.distributed as dist
    from videollama2_b200 import presets
    from videollama2_b200.model.tp_decoder import TPDecoderEngine
    layers = int(os.environ.get("VL2_TP_LAYERS", "80"))
    cfg = presets.make_config(dict(presets.QWEN2_72B, num_hidden_layers=layers), FRAMES)
    fl = presets.flops(cfg, FRAMES, PROMPT)
    S = fl["S"]
    from videollama2_b200.model import VLLMs
    from videollama2_b200 import parallel
    with_vision = os.environ.get("VL2_TP_VISION", "1") == "1"
    if not with_vision:
        cfg.mm_vision_tower = None
    model = VLLMs[cfg.model_type](cfg, tp_group=True)
    sd = presets.random_tp_shard(cfg, rank, world, dev)
    if with_vision:
        sd.update(presets.random_vision_state(cfg, dev))
    model.load_state_dict(sd, dev, presharded=True)
    del sd
    eng = model.get_model().decoder
    assert isinstance(eng, TPDecoderEngine)
    torch.cuda.empty_cache()
    emb = (0.5 * torch.randn((S, cfg.hidden_size), generator=torch.Generator(device=dev).manual_seed(7), device=dev)).to(torch.bfloat16)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / k

    step = lambda: eng.prefill(emb, all_logits=False)[0]
    # (1) collectives through NCCL (all-reduce + a separate row-statistics kernel)
    for _ in range(max(3, args.warmup)):
        step()
    ms_nccl = timed(step, args.steps)
    logits_nccl = step().float()
    # (2) the library's own kernel: in-switch reduction + RMSNorm statistics + broadcast in one launch (the default)
    nvls = None
    ms = ms_nccl
    clocks = None
    try:
        eng.enable_nvls_all_reduce(S, use_multicast=os.environ.get("VL2_TP_MULTICAST", "1") == "1",
                                   inswitch_reduce=os.environ.get("VL2_TP_INSWITCH", "0") == "1")
        for _ in range(max(3, args.warmup)):
            step()
        sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
        if rank == 0:
            sampler.start()
        t0 = time.time()
        ms_nvls = timed(step, args.steps)
        clocks = sampler.stop(t0, time.time()) if rank == 0 else None
        lg = step().float()
        nvls = {"ms_per_step": ms_nvls, "multicast_broadcast": bool(eng._nvls.multicast),
                "inswitch_reduce": bool(eng._nvls.inswitch_reduce),
                "rel_l2_vs_nccl_path": float((lg - logits_nccl).norm() / logits_nccl.norm()),
                "same_argmax_as_nccl_path": bool(int(lg.argmax()) == int(logits_nccl.argmax()))}
        ms = ms_nvls
    except Exception as e:      # symmetric memory / multicast unavailable on this box: the NCCL path is the measurement
        nvls = {"error": repr(e)[:300]}
        eng._nvls = None
    # (3) the same step without the collectives: what the all-reduces cost on the critical path
    from videollama2_b200 import ops as _ops
    real = eng._reduce_stats

    def no_collective(gemm_into):
        x = gemm_into(None)
        return x, _ops.row_sumsq(x)
    eng._reduce_stats = no_collective
    for _ in range(2):
        step()
    ms_noar = timed(step, max(3, args.steps // 2))
    eng._reduce_stats = real
    # the collective alone: [S, H] bf16 sum over the group, back to back
    buf = torch.randn((S, cfg.hidden_size), device=dev).to(torch.bfloat16)
    n_ar = 2 * layers
    ms_ar = timed(lambda: [dist.all_reduce(buf) for _ in range(n_ar)], 3)
    # ---- the whole configuration: frame-sharded ViT + first RegStage -> all-gather -> connector tail -> TP decoder,
    # through generate(max_new_tokens=1) from pinned host frames on every rank (SPMD: identical inputs everywhere)
    e2e = None
    if with_vision:
        try:
            model.get_vision_tower().enable_cuda_graphs(True)
            model.get_model().mm_projector.enable_cuda_graphs(True)
            model.enable_frame_parallel(None, shard_s1=True, llm_rank=None)       # every rank goes on to its decoder shard
            px0, ids_host = presets.synthetic_inputs(cfg, FRAMES, PROMPT)
            px_host = px0.pin_memory()
            mask = torch.ones_like(ids_host, dtype=torch.bool)

            def step_e2e():
                return model.generate(ids_host, images=[(px_host.to(dev, non_blocking=True), "video")], attention_mask=mask,
                                      max_new_tokens=1, do_sample=False).cpu()

            def vision_only():
                return model.encode_images_or_videos([(px_host.to(dev, non_blocking=True), "video")])
            for _ in range(3):
                tok = step_e2e()
            ms_e2e = timed(step_e2e, args.steps)
            for _ in range(2):
                vision_only()
            ms_vis = timed(vision_only, args.steps)
            t_dev = tok.to(dev)
            lo_t, hi_t = t_dev.clone(), t_dev.clone()
            dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
            fl_all = presets.flops(cfg, FRAMES, PROMPT)
            e2e = {"value": S / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": int(px_host.numel() * 2 + ids_host.numel() * 8), "d2h_bytes_per_step": 8,
                   "vision_stage_ms": ms_vis, "frames_per_s": FRAMES / (ms_vis * 1e-3), "same_token_on_all_ranks": bool(torch.equal(lo_t, hi_t)),
                   "flops_per_step": fl_all["total"], "tflops_per_gpu": fl_all["total"] / world / (ms_e2e * 1e-3) / 1e12,
                   "api": "Videollama2Qwen2ForCausalLM(tp_group).generate(ids, images=[(frames,'video')], max_new_tokens=1) with "
                          "enable_frame_parallel(llm_rank=None): ViT + first RegStage sharded by frame, one all-gather, "
                          "connector tail on every rank, tensor-parallel decoder"}
        except Exception as exc:      # the decoder line stands on its own
            e2e = {"error": repr(exc)[:400]}
    logits = step()
    same = torch.tensor([float(logits.float().abs().sum())], device=dev)
    lo, hi = same.clone(), same.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    if rank == 0:
        pk = peaks()
        dec_fl = fl["llm"]
        per_gpu = dec_fl / world / (ms * 1e-3) / 1e12
        ar_bytes = S * cfg.hidden_size * 2
        line = {
            "metric": METRIC, "value": S / (ms * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"VideoLLaMA2-72B (Qwen2-72B geometry, {layers} layers) decoder prefill S={S} (16 frames@336 + "
                                   f"256-token prompt), last-position logits, tensor-parallel x{world}; `e2e` = the whole configuration incl. the "
                                   f"frame-sharded vision stage",
                       "frames": FRAMES, "prompt": PROMPT, "seq": S, "parallelism": f"tp{world}", "weights": "device RNG, sharded",
                       "flops_per_step": dec_fl, "cuda_graphs": False},
            "llm_prefill_tok_per_s": S / (ms * 1e-3),
            "roofline": {"bound": "tensor", "achieved": per_gpu, "peak": pk["bf16_sustained"], "unit": "TFLOP/s per GPU",
                         "frac": per_gpu / pk["bf16_sustained"], "peak_src": pk["src"] + " sustained", "traffic": None},
            "tensor_parallel": {"ranks": world, "ms_per_step": ms, "ms_without_all_reduce": ms_noar,
                                "all_reduce_share_of_step": 1.0 - ms_noar / ms, "all_reduces_per_step": n_ar,
                                "all_reduce_bytes": ar_bytes, "all_reduce_alone_ms_per_step": ms_ar,
                                "all_reduce_alone_us_each": ms_ar / n_ar * 1e3,
                                "all_reduce_busbw_gbs": ar_bytes * 2 * (world - 1) / world / (ms_ar / n_ar * 1e-3) / 1e9,
                                "logits_identical_on_all_ranks": bool(float(lo) == float(hi)),
                                "ms_per_step_nccl_path": ms_nccl, "own_kernel_path": nvls,
                                "collective": "vl2_tp_allreduce_stats (peer-load reduce in rank order + multimem.st broadcast, barriers in-kernel) when "
                                              "available, else NCCL all-reduce + vl2_row_sumsq; `ms_per_step` is the faster path "
                                              "that ran" if nvls and "error" not in nvls else "NCCL all-reduce (torch.distributed), bf16"},
            "clocks": clocks, "gpu_launches": None, "e2e": e2e, "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vl2", choices=["vl2", "reference"])
    ap.add_argument("--model", default="mistral7b", choices=["mistral7b", "qwen2_7b", "qwen2_7b_v21", "qwen2_72b"],
                    help="qwen2_7b_v21 = the released VideoLLaMA2.1 geometry: SigLIP-so400m@384 tower + stc_connector_v35")
    ap.add_argument("--dtype", default="bfloat16", choices=["bfloat16", "float16"],
                    help="16-bit storage type: bfloat16 (headline) or float16 (the reference's inference dtype; libvl2_f16.so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true",
                    help="skip the untimed full-depth parity pass against tests/golden/full_cfg*.pt (on by default)")
    ap.add_argument("--gpu-rng-weights", action="store_true",
                    help="random weights from the device RNG (fast start-up; the output can then not be parity-checked)")
    ap.add_argument("--no-kernel-profile", action="store_true")
    ap.add_argument("--decode-tokens", type=int, default=16, help="extra (untimed-region) KV-cache decode measurement; 0 = skip")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly instead of replaying CUDA graphs")
    ap.add_argument("--profile-one-step", action="store_true",
                    help="warm up, then run ONE step between cudaProfilerStart/Stop and exit (for `ncu --profile-from-start off`)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (last-position logits, float32) as DIR/<name>.npy, so two "
                         "builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.model == "qwen2_72b" or args.profile_one_step):
        ap.error("--dump-outputs applies to the timed prefill step of the --impl vl2 single-model workloads")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    # host threads: a container whose cgroup CPU quota is smaller than os.cpu_count() must not run 128 OpenMP threads (they
    # spin after every parallel region, burn the quota and get the whole process - including the launching thread - throttled)
    # ... and the GPU arm has next to no CPU work: a small pool leaves the quota to the launching thread and the CUDA driver
    torch.set_num_threads(max(1, min(4, host_threads()["threads"] // max(1, int(os.environ.get("WORLD_SIZE", "1"))))))
    import torch.distributed as dist
    from videollama2_b200 import ops, presets
    from videollama2_b200.model import VLLMs
    from videollama2_b200 import parallel

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: keep fd 1 clean (rank 0 prints
        # ONE JSON line) by pointing it at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    if args.model == "qwen2_72b":       # config 5: tensor-parallel decoder (needs the process group; 8 GPUs for all 80 layers)
        if world < 2:
            raise SystemExit("--model qwen2_72b is the tensor-parallel configuration: launch with torchrun, --gpus 2/4/8")
        bench_tp72b(args, rank, world, dev)
        dist.destroy_process_group()
        return
    llm = presets.MISTRAL_7B if args.model == "mistral7b" else presets.QWEN2_7B
    if args.model == "qwen2_7b_v21":
        cfg = presets.make_config(llm, FRAMES, "stc_connector_v35", presets.SIGLIP_SO400M_384)
    else:
        cfg = presets.make_config(llm, FRAMES)
    cfg.torch_dtype = args.dtype
    IMG = cfg.vision_config.image_size
    fl = presets.flops(cfg, FRAMES, PROMPT)
    S = fl["S"]
    # the deterministic synthetic checkpoint (host RNG): the SAME bytes the committed full-depth goldens were computed
    # with by the real reference classes, so the benchmarked model's own output can be parity-checked (--check)
    t_w = time.time()
    if args.gpu_rng_weights:
        sd = presets.random_state_dict(cfg, dev)
    else:
        sd = presets.synthetic_state_dict(cfg, dev, threads=max(1, min(16, (os.cpu_count() or 8) // max(1, world))))
    model = VLLMs[cfg.model_type].from_state_dict(cfg, sd, device=dev)
    del sd
    torch.cuda.empty_cache()
    weights_s = time.time() - t_w
    if not args.no_graphs and not args.profile_one_step:
        model.enable_cuda_graphs(True)

    # SURVEY.md §8d inputs (rank 0 = the goldens' video; other replicas get their own frames)
    px0, ids_host = presets.synthetic_inputs(cfg, FRAMES, PROMPT)
    if rank > 0:
        g = torch.Generator(device="cpu").manual_seed(1234 + rank)
        px0 = torch.randn((FRAMES, 3, IMG, IMG), generator=g).to(torch.bfloat16)
    px_host = px0.to(cfg.storage_dtype).pin_memory()
    px_dev = px_host.to(dev)
    mask = torch.ones_like(ids_host, dtype=torch.bool)

    last = {}

    def step_resident():
        _, _, _, emb, _ = model.prepare_inputs_labels_for_multimodal(ids_host, mask, None, None, [(px_dev, "video")])
        logits, _ = model.get_model().decoder.prefill(emb[0], all_logits=False)
        last["logits"] = logits
        return logits

    def step_e2e():
        px = px_host.to(dev, non_blocking=True)
        return model.generate(ids_host, images=[(px, "video")], attention_mask=mask, max_new_tokens=1, do_sample=False).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / k, t0, time.time()

    check = None
    fixture = {"mistral7b": "cfg2", "qwen2_7b": "cfg3"}.get(args.model)
    if rank == 0 and not args.no_check and not args.gpu_rng_weights and not args.profile_one_step and fixture is not None:
        from videollama2_b200 import selfcheck
        if os.path.exists(selfcheck.fixture_path(fixture)):
            model.enable_cuda_graphs(False)
            check = selfcheck.fulldepth_check(model, fixture, px_host, ids_host)
            check["golden"] = "real reference classes on CPU, fp32 on bf16-rounded weights (oracle/make_golden_full.py)"
            if not args.no_graphs:
                model.enable_cuda_graphs(True)
            if not check["ok"]:
                print(f"bench.py: FULL-DEPTH PARITY CHECK FAILED: {json.dumps(check)}", file=sys.stderr, flush=True)
    for _ in range(args.warmup):
        step_resident()
    if args.profile_one_step:
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step, t0, t1 = timed(step_resident, args.steps)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # copied before anything else runs: with CUDA graphs the logits live in the graph's static output buffer
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "logits.npy"), last["logits"].float().cpu().numpy())

    for _ in range(2):
        step_e2e()
    ms_e2e, _, _ = timed(step_e2e, args.steps)

    # KV-cache decode (SURVEY.md §8f row 1): greedy tokens after the prefill through the public generate() API
    decode = None
    if args.decode_tokens > 0 and rank == 0:
        n_new = args.decode_tokens + 2

        def gen(n):
            torch.cuda.synchronize()
            t_a = time.perf_counter()
            out = model.generate(ids_host, images=[(px_dev, "video")], attention_mask=mask, max_new_tokens=n,
                                 do_sample=False, use_cache=True, eos_token_id=None)
            torch.cuda.synchronize()
            return (time.perf_counter() - t_a) * 1e3, int(out.shape[1])

        gen(n_new + 8)                          # sizes the KV cache for the longest run and captures the single-token decode graph
        t_short, got_s = gen(8)                 # two runs that differ only in the number of decode steps
        t_long, got = gen(n_new + 8)
        # the same graph replayed back to back, timed on the device (what one token costs without the host's share)
        dec = model.get_model().decoder
        dec.kv_len = S
        dec.decode_graph_begin(3)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dec.decode_graph_run(args.decode_tokens)
        e1.record()
        torch.cuda.synchronize()
        ms_tok_dev = e0.elapsed_time(e1) / args.decode_tokens
        if got > got_s:
            ms_wall = (t_long - t_short) / (got - got_s)        # through generate(): includes the host's share; noisy on a
            ms_tok = ms_tok_dev                                  # quota-throttled host, so the device-timed figure is the headline
            w_bytes = sum(t.numel() * t.element_size() for L in model.get_model().decoder.layers for t in L.values())
            w_bytes += model.get_model().decoder.w["lm_head"].numel() * 2
            hbm = float(peaks().get("hbm_gbs") or 6500.0)
            decode = {"new_tokens": got, "ms_per_token": ms_tok, "ms_per_token_device_timed": ms_tok_dev,
                      "ms_per_token_generate_wall": ms_wall if ms_wall > 0 else None,
                      "tok_per_s": 1e3 / ms_tok if ms_tok > 0 else None,
                      "weight_bytes_per_token": int(w_bytes), "achieved_gbps": w_bytes / ms_tok / 1e6,
                      "hbm_peak_gbps": hbm, "frac_of_hbm": w_bytes / ms_tok / 1e6 / hbm,
                      "note": "greedy, batch 1, weight-streaming GEMV + single-token attention kernels; one CUDA-graph replay per "
                              "token (position and token live in device memory); ms_per_token = the graph generate() uses, replayed "
                              "back to back between CUDA events; ms_per_token_generate_wall = wall-clock difference of two "
                              "generate() calls that differ only in max_new_tokens (null when host noise exceeds it)"}

    # frame preprocessing on the device (SURVEY.md §8f row 3): 16 decoded 1080p uint8 frames -> pixel_values
    prep = None
    if rank == 0 and world == 1 and not args.profile_one_step:
        from videollama2_b200 import mm_utils as vl2_mm
        proc = model.get_vision_tower().image_processor
        gp = torch.Generator(device="cpu").manual_seed(77)
        raw = torch.randint(0, 256, (FRAMES, 1080, 1920, 3), generator=gp, dtype=torch.uint8).pin_memory()
        raw_dev = raw.to(dev)
        for _ in range(2):
            vl2_mm.process_video(raw_dev, proc, num_frames=FRAMES, device=dev)
        ms_prep_dev, _, _ = timed(lambda: vl2_mm.process_video(raw_dev, proc, num_frames=FRAMES, device=dev), 5)
        ms_prep_e2e, _, _ = timed(lambda: vl2_mm.process_video(raw.to(dev, non_blocking=True), proc, num_frames=FRAMES,
                                                              device=dev), 5)
        in_bytes = raw.numel()
        tmp_bytes = FRAMES * 1920 * IMG * 3
        algo = in_bytes + 2 * tmp_bytes + FRAMES * 3 * IMG * IMG * 2
        prep = {"input": f"{FRAMES} x 1080x1920x3 uint8 (pad to square, Pillow-exact bicubic to {IMG}, normalise, bf16)",
                "ms_resident": ms_prep_dev, "ms_from_pinned_host": ms_prep_e2e, "frames_per_s": FRAMES / (ms_prep_dev * 1e-3),
                "algorithmic_bytes": int(algo), "achieved_gbps": algo / ms_prep_dev / 1e6,
                "frac_of_hbm": algo / ms_prep_dev / 1e6 / float(peaks().get("hbm_gbs") or 6500.0),
                "h2d_bytes": int(in_bytes)}
        del raw_dev

    # stage split (device events, same stream; graph replays when graphs are on, like the timed step)
    def stage_times():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        torch.cuda.synchronize()
        ev[0].record()
        feats = model.get_vision_tower()(px_dev)
        ev[1].record()
        _, _, _, emb, _ = model.prepare_inputs_labels_for_multimodal(ids_host, mask, None, None, [(px_dev, "video")])
        ev[2].record()
        model.get_model().decoder.prefill(emb[0], all_logits=False)
        ev[3].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])

    st = [stage_times() for _ in range(5)]
    t_vit = statistics.median(s[0] for s in st)
    t_vis = statistics.median(s[1] for s in st)      # ViT + STC + splice (encode_images_or_videos inside)
    t_llm = statistics.median(s[2] for s in st)

    # dominant-kernel roofline: every tcgen05 GEMM launch of one step bracketed by CUDA events on the launch stream
    roof = None
    model.enable_cuda_graphs(False)      # per-kernel event timing needs eager launches
    l0 = ops.launch_count()
    step_resident()                      # the same step launched eagerly: how many libvl2 kernels one step runs
    torch.cuda.synchronize()
    launches = ops.launch_count() - l0

    if not args.no_kernel_profile and rank == 0:
        recs = []
        orig = ops.gemm

        def gemm_timed(a, w, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = orig(a, w, **kw)
            e1.record()
            recs.append((e0, e1, 2.0 * a.shape[0] * w.shape[0] * a.shape[1]))
            return out

        for mod in (sys.modules["videollama2_b200.model.encoder"], sys.modules["videollama2_b200.model.projector"],
                    sys.modules["videollama2_b200.model.decoder"]):
            mod.ops = type("OpsProxy", (), {"__getattr__": lambda self, n, _o=ops: gemm_timed if n == "gemm" else getattr(_o, n)})()
        try:
            step_resident()
            torch.cuda.synchronize()
        finally:
            for mod in (sys.modules["videollama2_b200.model.encoder"], sys.modules["videollama2_b200.model.projector"],
                        sys.modules["videollama2_b200.model.decoder"]):
                mod.ops = ops
        g_ms = sum(a.elapsed_time(b) for a, b, _ in recs)
        g_fl = sum(f for _, _, f in recs)
        pk = peaks()
        # dram__bytes_read + dram__bytes_write per GEMM launch come from an ncu capture, which cannot run inside a timed
        # bench: the committed extract is used ONLY if it was taken from this very build (source digest match)
        traffic, traffic_src = None, "no ncu capture of this build committed under profiles/"
        tp = os.path.join(ROOT, "profiles", "r02_gemm_dram_traffic.json")
        if os.path.exists(tp):
            from videollama2_b200 import build as vl2_build
            tj = json.load(open(tp))
            if tj.get("source_digest") == vl2_build._digest():
                traffic, traffic_src = tj.get("traffic_bytes_per_launch"), tj.get("source")
            else:
                traffic_src = "profiles/r02_gemm_dram_traffic.json is from another build (digest mismatch): not reported"
        ach = g_fl / (g_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "gemm_bf16_tcgen05_kernel", "achieved": ach, "peak": pk["bf16_sustained"],
                "unit": "TFLOP/s", "frac": ach / pk["bf16_sustained"], "traffic": traffic, "traffic_src": traffic_src, "launches": len(recs),
                "avg_launch_ms": g_ms / max(1, len(recs)), "flops_per_launch": g_fl / max(1, len(recs)),
                "gemm_ms_per_step": g_ms, "gemm_share_of_step": g_ms / ms_step, "peak_src": pk["src"] + " sustained",
                "whole_step": {"achieved": fl["total"] / (ms_step * 1e-3) / 1e12,
                               "frac": fl["total"] / (ms_step * 1e-3) / 1e12 / pk["bf16_sustained"]}}

    # ONE video on all N GPUs through the product API (north_star's split): model.enable_frame_parallel() shards the
    # per-frame part of encode_images_or_videos (ViT + first RegStage) over the ranks, ONE all-gather in front of the
    # connector's Conv3d, the decoder on rank 0.  Every rank passes the same frames.  Device-timed, max over ranks.
    fp = None
    if world > 1:
        if not args.no_graphs:
            model.enable_cuda_graphs(True)
        px_same_host, _ = presets.synthetic_inputs(cfg, FRAMES, PROMPT)
        px_same_host = px_same_host.pin_memory()
        px_same = px_same_host.to(dev)
        vid = [(px_same, "video")]
        tower, proj = model.get_vision_tower(), model.get_model().mm_projector
        hw = tower.num_patches_per_side

        def t_of(fn, k=max(5, args.steps)):
            for _ in range(2):
                fn()
            return timed(fn, k)[0]

        # single-GPU references on this rank (graph replays): whole vision stage, and the part that shards
        ms_vis_1 = t_of(lambda: model.encode_images_or_videos(vid))
        ms_part_1 = t_of(lambda: proj.forward_s1(tower(px_same).view(FRAMES, hw, hw, -1)))
        ms_one_1 = t_of(lambda: model.generate(ids_host, images=[(px_same_host.to(dev, non_blocking=True), "video")],
                                               attention_mask=mask, max_new_tokens=1, do_sample=False).cpu())
        ref_feats = model.encode_images_or_videos(vid).clone()
        model.enable_frame_parallel(None, shard_s1=True, llm_rank=0)
        fpo = model._frame_parallel
        a_, b_ = parallel.frame_shard(FRAMES, rank, world)
        got_feats = model.encode_images_or_videos(vid)
        exact = torch.tensor([1 if torch.equal(got_feats, ref_feats) else 0], device=dev)
        dist.all_reduce(exact, op=dist.ReduceOp.MIN)
        ms_vis_n = t_of(lambda: model.encode_images_or_videos(vid))

        def sharded_part():          # ViT + s1 on this rank's frames + the all-gather
            s1 = proj.forward_s1(tower(px_same[a_:b_]).view(b_ - a_, hw, hw, -1))
            return parallel.all_gather_frames(s1.reshape(b_ - a_, hw * hw, -1), FRAMES)
        ms_part_n = t_of(sharded_part)
        s1_loc = proj.forward_s1(tower(px_same[a_:b_]).view(b_ - a_, hw, hw, -1)).reshape(b_ - a_, hw * hw, -1)
        ms_gather = t_of(lambda: parallel.all_gather_frames(s1_loc, FRAMES))

        def one_video_e2e():
            out = model.generate(ids_host, images=[(px_same_host.to(dev, non_blocking=True), "video")], attention_mask=mask,
                                 max_new_tokens=1, do_sample=False)
            return out.cpu() if out is not None else None
        ms_one_n = t_of(one_video_e2e)
        model.enable_frame_parallel(False)
        fp = {"ranks": world, "frames_per_rank": parallel.shard_sizes(FRAMES, world), "api": "model.enable_frame_parallel(); "
              "encode_images_or_videos / generate (ViT + first RegStage sharded by frame, one NCCL all-gather of [F,576,4096] "
              "bf16, decoder on rank 0)", "bit_exact_vs_1gpu": bool(int(exact.item()) == 1),
              "gather_bytes": int(FRAMES * tower.num_patches * proj.hidden_size * 2), "all_gather_ms": ms_gather,
              "sharded_part": {"what": "ViT + STC s1 (+ all-gather): everything in front of the first time-mixing op",
                               "ms_1gpu": ms_part_1, "ms": ms_part_n, "speedup_vs_1gpu": ms_part_1 / ms_part_n,
                               "frames_per_s": FRAMES / (ms_part_n * 1e-3)},
              "vision_stage": {"what": "encode_images_or_videos (pixels -> connector output)", "ms_1gpu": ms_vis_1, "ms": ms_vis_n,
                               "speedup_vs_1gpu": ms_vis_1 / ms_vis_n, "frames_per_s": FRAMES / (ms_vis_n * 1e-3)},
              "one_video_e2e": {"what": "generate(max_new_tokens=1) from pinned host frames, one video on all ranks",
                                "ms_1gpu": ms_one_1, "ms": ms_one_n, "speedup_vs_1gpu": ms_one_1 / ms_one_n,
                                "tok_per_s": S / (ms_one_n * 1e-3)}}
        fp["speedup_vs_1gpu"] = fp["sharded_part"]["speedup_vs_1gpu"]

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # the CPU leg belongs to the N = 1 line only
        try:
            r = cpu_reference_step(n_steps=1)
            cpu = {"value": r["tok_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                   "frames_per_s": r["frames_per_s"], "llm_prefill_tok_per_s": r["llm_tok_per_s"], "ms_per_step": r["t_all_s"] * 1e3,
                   "host": r["host"]}
        except Exception as e:  # the baseline must never take the bench line down
            cpu = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e!r}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": world * S / (ms_step * 1e-3), "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.dtype == "bfloat16" else "fp16", "data": "synthetic",
            "config": {"workload": WORKLOAD.format(model=args.model, img=IMG, S=S), "frames": FRAMES, "prompt": PROMPT, "seq": S,
                       "global_batch": world, "weights": "device RNG" if args.gpu_rng_weights else
                       f"deterministic synthetic checkpoint (host RNG, seed {presets.SYNTH_SEED}; {weights_s:.0f}s to generate + load)",
                       "parallelism": f"replicas x{world} (+ frame-sharded ViT reported separately)",
                       "cuda_graphs": not args.no_graphs,
                       "l2": "weights (16 GB) >> L2 (126 MB): every step streams them from HBM; no explicit flush",
                       "flops_per_step": fl["total"]},
            "frames_per_s": world * FRAMES / (t_vis * 1e-3), "vit_frames_per_s": world * FRAMES / (t_vit * 1e-3),
            "llm_prefill_tok_per_s": world * S / (t_llm * 1e-3),
            "stage_ms": {"vit": t_vit, "vision_total": t_vis, "llm_prefill": t_llm},
            "e2e": {"value": world * S / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": px_host.numel() * 2 + ids_host.numel() * 8, "d2h_bytes_per_step": 8,
                    "api": "Videollama2MistralForCausalLM.generate(ids, images=[(frames,'video')], max_new_tokens=1)"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "check": check, "decode": decode,
            "preprocess": prep,
        }
        if fp is not None:
            line["frame_parallel"] = fp
            # first-class copies of the one-video-on-N-GPUs numbers (the split north_star names)
            line["frame_parallel_frames_per_s"] = fp["sharded_part"]["frames_per_s"]
            line["frame_parallel_speedup"] = fp["sharded_part"]["speedup_vs_1gpu"]
            line["one_video_e2e_tok_per_s"] = fp["one_video_e2e"]["tok_per_s"]
            line["one_video_e2e_speedup"] = fp["one_video_e2e"]["speedup_vs_1gpu"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
