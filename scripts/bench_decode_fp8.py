"""KV-cache decode with fp8 (E4M3) decoder weights against bf16, Mistral-7B synthetic checkpoint, config-2 prefill length.

One process builds the same checkpoint twice (decode_weights="bf16" and "fp8") and reports:
  * per-shape GEMV time and achieved GB/s for both weight types (weights rotate through a pool larger than the 126 MB L2,
    the calls are captured in one CUDA graph, as scripts/microbench_decode.py does);
  * decode ms/token, device-timed (the generate() decode graph replayed back to back between CUDA events, as bench.py
    does) and through generate() (wall-clock difference of two calls that differ only in max_new_tokens: it carries the
    host's noise), bf16 and fp8 runs alternating, one discarded warm-up round and then `--repeats` each; SM clocks are
    sampled by nvidia-smi during these rounds;
  * per-kernel device time of one token for both (torch.profiler over graph replays, a separate pass);
  * teacher-forced fp8-vs-bf16 last-position logits relL2 per step, and greedy agreement over `--tokens` tokens.
Prints one JSON line (with the GPU name, power limit and the SM clocks under load) and writes it to --out if given.
Usage: python scripts/bench_decode_fp8.py [--repeats 3] [--tokens 64] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from videollama2_b200 import ops, presets
from videollama2_b200.model import VLLMs

FRAMES, PROMPT = 16, 256          # bench.py's config 2: S = 1776 after the splice


def gpu_info(index=0):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, sm, sm_max = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit_w": float(pl), "sm_mhz": int(sm), "sm_max_mhz": int(sm_max)}
    except Exception as exc:         # nvidia-smi missing: the device name still comes from torch
        return {"gpu": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_mhz": None, "sm_max_mhz": None,
                "nvidia_smi": str(exc)}


class ClockSampler:
    """SM clock (MHz) sampled every 200 ms by nvidia-smi while the timed rounds run."""

    def __init__(self, index=0):
        self.index, self.proc = index, None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        self.mhz = []
        if self.proc is not None:
            self.proc.terminate()
            out, _ = self.proc.communicate(timeout=30)
            self.mhz = [int(v) for v in out.split() if v.strip().isdigit()]

    def summary(self):
        if not self.mhz:
            return None
        return {"samples": len(self.mhz), "median": int(statistics.median(self.mhz)), "min": min(self.mhz),
                "max": max(self.mhz)}


def kernel_breakdown(dec, S, tokens=8):
    """Device time per token by kernel (torch.profiler, CUDA activity) over `tokens` back-to-back graph replays."""
    from torch.profiler import ProfilerActivity, profile
    dec.kv_len = S
    dec.decode_graph_begin(3)
    dec.decode_graph_run(2)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dec.decode_graph_run(tokens)
        torch.cuda.synchronize()
    groups = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if not t or ev.key.startswith("cuda") or "Memcpy" in ev.key or "Memset" in ev.key:
            continue
        name = ev.key.split("(")[0].replace("void ", "").strip()
        groups[name] = groups.get(name, 0.0) + t / tokens / 1e3           # us -> ms per token
    total = sum(groups.values())
    return {"kernel_ms_per_token": round(total, 4),
            "by_kernel_ms_per_token": {k: round(v, 4) for k, v in sorted(groups.items(), key=lambda kv: -kv[1])}}


def graph_time_us(fn, n):
    """Mean time of fn(i), i = 0..n-1, captured in one CUDA graph, replayed 3 times between events."""
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / (3 * n) * 1e3


def gemv_shapes(dev):
    res = {}
    for name, N, K, act, rms in [("qkv", 6144, 4096, 0, 1e-5), ("o", 4096, 4096, 0, 0.0),
                                 ("gate_up", 28672, 4096, ops.ACT_SWIGLU, 1e-5), ("down", 4096, 14336, 0, 0.0),
                                 ("lm_head", 32000, 4096, 0, 1e-5)]:
        x = torch.randn((1, K), device=dev, dtype=torch.bfloat16)
        out = torch.empty((1, N // 2 if act == ops.ACT_SWIGLU else N), device=dev, dtype=torch.bfloat16)
        row = {"N": N, "K": K}
        for kind in ("bf16", "fp8"):
            nbytes = N * K * (2 if kind == "bf16" else 1) + (N * 4 if kind == "fp8" else 0)
            pool = max(2, int(400e6 // nbytes) + 1)
            ws = []
            for _ in range(pool):
                w = torch.randn((N, K), device=dev, dtype=torch.float32) * 0.02
                ws.append((w.to(torch.bfloat16), None) if kind == "bf16" else ops.quantize_fp8_rows(w))
                del w
            us = graph_time_us(lambda i: ops.gemv(x, ws[i % pool][0], w_scale=ws[i % pool][1], act=act, rms_eps=rms,
                                                  out=out), 40)
            row[kind] = {"us": round(us, 2), "GBps": round(nbytes / us / 1e3, 1)}
            del ws
        row["fp8_over_bf16"] = round(row["fp8"]["us"] / row["bf16"]["us"], 3)
        res[name] = row
    return res


def rel(a, b):
    return float((a.float() - b.float()).norm() / (b.float().norm() + 1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--tokens", type=int, default=64)
    ap.add_argument("--decode-steps", type=int, default=64, help="graph replays per device-timed window")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode_fp8.py needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    shapes = gemv_shapes(dev)
    torch.cuda.empty_cache()

    cfg = presets.make_config(presets.MISTRAL_7B, FRAMES)
    sd = presets.synthetic_state_dict(cfg, dev, threads=max(1, min(16, os.cpu_count() or 8)))
    models = {"bf16": VLLMs[cfg.model_type].from_state_dict(cfg, sd, device=dev),
              "fp8": VLLMs[cfg.model_type].from_state_dict(cfg, sd, device=dev, decode_weights="fp8")}
    del sd
    torch.cuda.empty_cache()
    px, ids = presets.synthetic_inputs(cfg, FRAMES, PROMPT)
    px = px.to(dev)
    mask = torch.ones_like(ids, dtype=torch.bool)
    imgs = [(px, "video")]
    emb = models["bf16"].prepare_inputs_labels_for_multimodal(ids, mask, None, None, imgs)[3][0]
    S = emb.shape[0]
    for m in models.values():
        m.enable_cuda_graphs(True)

    def gen(m, n):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = m.generate(ids, images=imgs, attention_mask=mask, max_new_tokens=n, do_sample=False, eos_token_id=None)
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, out

    n_long = args.decode_steps + 8
    greedy = {k: gen(m, max(n_long, args.tokens))[1] for k, m in models.items()}   # sizes caches, captures graphs
    runs = {k: {"device_ms": [], "generate_ms": []} for k in models}
    with ClockSampler(0) as clocks:
        for rnd in range(args.repeats + 1):                           # round 0 is a warm-up and is not reported
            for k, m in models.items():                               # bf16 and fp8 alternate
                t_short, _ = gen(m, 8)
                t_long, _ = gen(m, n_long)
                dec = m.get_model().decoder
                dec.kv_len = S
                dec.decode_graph_begin(3)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                dec.decode_graph_run(args.decode_steps)
                e1.record()
                torch.cuda.synchronize()
                if rnd > 0:
                    runs[k]["generate_ms"].append((t_long - t_short) / (n_long - 8))
                    runs[k]["device_ms"].append(e0.elapsed_time(e1) / args.decode_steps)
    decode = {}
    for k in models:
        dec = models[k].get_model().decoder
        layers, head = dec._decode_set()
        w_bytes = sum(t.numel() * t.element_size() for L in layers for n, t in L.items())
        w_bytes += sum(t.numel() * t.element_size() for n, t in head.items() if n.startswith("lm_head"))
        med = statistics.median(runs[k]["device_ms"])
        decode[k] = {"ms_per_token_device_timed": [round(v, 4) for v in runs[k]["device_ms"]],
                     "ms_per_token_generate_wall": [round(v, 4) for v in runs[k]["generate_ms"]],
                     "median_device_ms": round(med, 4),
                     "median_generate_wall_ms": round(statistics.median(runs[k]["generate_ms"]), 4),
                     "weight_bytes_per_token": int(w_bytes), "weight_GBps_at_median": round(w_bytes / med / 1e6, 1)}
        try:
            decode[k]["profile"] = kernel_breakdown(dec, S)
        except Exception as exc:        # the timing above stands on its own
            decode[k]["profile"] = {"error": repr(exc)}
    ratio = decode["fp8"]["median_device_ms"] / decode["bf16"]["median_device_ms"]

    # teacher-forced: both engines fed the bf16 model's greedy tokens from the same prefill
    for m in models.values():
        m.enable_cuda_graphs(False)
    decs = {k: m.get_model().decoder for k, m in models.items()}
    for d in decs.values():
        d.prefill(emb, all_logits=False, keep_cache=True, max_len=S + args.tokens + 1)
    dist = []
    for tok in greedy["bf16"][0, : args.tokens].tolist():
        e = models["bf16"].get_model().embed_tokens(torch.tensor([tok]))
        a, b = decs["bf16"].decode_step(e), decs["fp8"].decode_step(e)
        dist.append(rel(b, a))
    g16, g8 = greedy["bf16"][0, : args.tokens].tolist(), greedy["fp8"][0, : args.tokens].tolist()
    first_diff = next((i for i, (a, b) in enumerate(zip(g16, g8)) if a != b), len(g16))
    info["sm_mhz_idle_before_run"] = info.pop("sm_mhz")
    res = {"bench": "decode_fp8", **info, "sm_mhz_during_decode_rounds": clocks.summary(), "model": "Mistral-7B synthetic (presets.synthetic_state_dict), config-2 prefill",
           "S": S, "gemv": shapes, "decode": decode, "fp8_over_bf16_device_ms": round(ratio, 3),
           "teacher_forced_logits_relL2": {"per_step": [round(d, 4) for d in dist], "mean": round(sum(dist) / len(dist), 4),
                                           "max": round(max(dist), 4)},
           "greedy_agreement": {"tokens": len(g16), "equal_positions": sum(int(a == b) for a, b in zip(g16, g8)),
                                "first_divergence": first_diff},
           "note": "synthetic untrained weights: the fp8-vs-bf16 distance says nothing about a real checkpoint's quality; "
                   "ms_per_token_generate_wall = (generate(n_long) - generate(8)) / (n_long - 8) wall clock, host noise "
                   "included - the device-timed figure is the headline"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
