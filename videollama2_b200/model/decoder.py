"""Mistral-7B / Qwen2 decoder prefill (+ greedy decode) on libvl2 kernels.

Arithmetic of HF MistralModel / Qwen2Model (HF:mistral/modeling_mistral.py:35-48,51-82,122-239,262-470;
HF:qwen2/modeling_qwen2.py:187-246): RMSNorm -> fused QKV GEMM (+bias for Qwen2) -> RoPE -> causal GQA flash attention
-> o_proj(+residual) -> RMSNorm -> gate/up GEMM with SwiGLU epilogue -> down_proj(+residual) -> norm -> lm_head.
Weights are repacked once: q/k/v concatenated, gate/up rows interleaved so SwiGLU happens inside the GEMM tile, and the
RMSNorm gains multiplied into the weight columns: the per-layer norms cost no kernel (row statistics are produced by
the residual GEMM epilogues, the 1/rms factor is applied in the consuming GEMM's epilogue).
With decode_weights="fp8" the single-token decode streams fp8 E4M3 copies of every linear weight (one fp32 scale per
output row, vl2_gemv_fp8): half the bytes per token.  Prefill always runs on the 16-bit weights."""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch

from .. import ops


DECODE_WEIGHTS = ("bf16", "fp8")


def check_decode_weights(decode_weights: str) -> str:
    if decode_weights not in DECODE_WEIGHTS:
        raise ValueError(f"decode_weights must be one of {DECODE_WEIGHTS}, not {decode_weights!r}")
    return decode_weights


class DecoderEngine:
    def __init__(self, config, decode_weights: str = "bf16"):
        self.config = config
        # "bf16": decode streams the prefill's 16-bit weights; "fp8": E4M3 copies with per-row scales (load_state_dict)
        self.decode_weights = check_decode_weights(decode_weights)
        self.layers8: List[Dict[str, torch.Tensor]] = []
        self.w8: Dict[str, torch.Tensor] = {}
        self.H = config.hidden_size
        self.Hq = config.num_attention_heads
        self.Hkv = config.num_key_value_heads
        self.D = config.hidden_size // config.num_attention_heads
        self.I = config.intermediate_size
        self.eps = config.rms_norm_eps
        self.dtype = getattr(config, "storage_dtype", torch.bfloat16)      # bf16 or fp16 (selects the library build)
        self.layers: List[Dict[str, torch.Tensor]] = []
        self.w: Dict[str, torch.Tensor] = {}
        self.is_loaded = False
        self.kv: List[torch.Tensor] = []   # per layer [S_max, (Hq+2Hkv)*D] fused qkv rows (K,V columns = cache)
        self.kv_len = 0
        self._graphed = None
        self._decode_graph = None   # (graph, tok_dev, pos_dev, logits) of the captured single-token step
        self._decode_log = None     # (device id buffer, device step counter) the graph appends its arg-max tokens to
        self._decode_read = 0
        self.graph_decode = False
        self.decode_pdl = os.environ.get("VL2_DECODE_PDL", "0") == "1"   # PDL edges inside the decode graph
        # MB of o_proj + gate/up weights pulled into L2 on a forked graph branch while the attention phase runs
        # (HBM is idle there); 0 disables the fork
        self.decode_prefetch_mb = float(os.environ.get("VL2_DECODE_PREFETCH_MB", "0"))
        self._side_stream = None

    def enable_cuda_graphs(self, on: bool = True):
        """Graph the cache-less last-position prefill (the bench / first-token path)."""
        from ..graphs import GraphedStage
        self._graphed = GraphedStage(lambda e: self._prefill_last(e)) if on else None
        self.graph_decode = on
        self._decode_graph = None
        return self

    def _prefill_last(self, embeds: torch.Tensor) -> torch.Tensor:
        return self.prefill(embeds, all_logits=False, keep_cache=False, _no_graph=True)[0]

    def load_state_dict(self, sd: Dict[str, torch.Tensor], device) -> "DecoderEngine":
        dev = torch.device(device)
        bf = lambda t: t.to(device=dev, dtype=self.dtype).contiguous()
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
        self.layers = []
        self.layers8, self.w8 = [], {}
        fp8 = self.decode_weights == "fp8"
        # RoPE runs in the epilogue of the fused QKV GEMM on ADJACENT column pairs: permute the q / k weight rows (and
        # biases) so that the partners (i, i + D/2) of a head come out as columns (2i, 2i+1).  q.k is invariant under the
        # permutation (same one for q and k), v is untouched, so attention and the KV cache consume the rows as they are.
        nqk = (self.Hq + self.Hkv) * self.D
        qk_perm = torch.cat([ops.rope_interleave_rows(self.Hq + self.Hkv, self.D),
                             torch.arange(nqk, nqk + self.Hkv * self.D)]).to(dev)
        for i in range(self.config.num_hidden_layers):
            p = f"model.layers.{i}."
            names = ("q_proj", "k_proj", "v_proj")
            # RMSNorm gains are folded into the columns of the weight that consumes the normalised activations:
            # rmsnorm(x; g) W^T = rstd(x) * (x (W * g)^T); rstd is applied per row in the GEMM epilogue.
            g1 = sd[p + "input_layernorm.weight"].to(device=dev, dtype=torch.float32)
            g2 = sd[p + "post_attention_layernorm.weight"].to(device=dev, dtype=torch.float32)
            wqkv = torch.cat([sd[p + f"self_attn.{n}.weight"] for n in names], 0).to(device=dev, dtype=torch.float32)
            wqkv = wqkv[qk_perm]          # RoPE partners of every q / k head become adjacent output columns
            wgu = torch.stack([sd[p + "mlp.gate_proj.weight"], sd[p + "mlp.up_proj.weight"]], 1).reshape(
                2 * self.I, self.H).to(device=dev, dtype=torch.float32)
            wqkv, wgu = wqkv * g1[None, :], wgu * g2[None, :]
            L = {
                "wqkv": wqkv.to(self.dtype).contiguous(),
                "wo": bf(sd[p + "self_attn.o_proj.weight"]),
                "wgu": wgu.to(self.dtype).contiguous(),
                "wd": bf(sd[p + "mlp.down_proj.weight"]),
            }
            if p + "self_attn.q_proj.bias" in sd:
                L["bqkv"] = f32(torch.cat([sd[p + f"self_attn.{n}.bias"] for n in names], 0).to(dev)[qk_perm])
            self.layers.append(L)
            if fp8:     # quantised from the same fp32 (folded, permuted, interleaved) tensors: one rounding, not two
                src = {"wqkv": wqkv, "wo": f32(sd[p + "self_attn.o_proj.weight"]), "wgu": wgu,
                       "wd": f32(sd[p + "mlp.down_proj.weight"])}
                L8 = {k: v for k, v in L.items() if k.startswith("b")}
                for k, wf in src.items():
                    L8[k], L8[k + "_s"] = ops.quantize_fp8_rows(wf)
                self.layers8.append(L8)
                del src
            del wqkv, wgu
        # final-norm gain folded into the lm_head columns (the GEMV / GEMM epilogue applies 1/rms itself)
        lm_head = (sd["lm_head.weight"].to(device=dev, dtype=torch.float32)
                   * sd["model.norm.weight"].to(device=dev, dtype=torch.float32)[None, :])
        self.w = {"embed": bf(sd["model.embed_tokens.weight"]), "norm": bf(sd["model.norm.weight"]),
                  "lm_head": lm_head.to(self.dtype).contiguous(),
                  "ones": torch.ones((self.H,), device=dev, dtype=self.dtype)}
        if fp8:
            self.w8["lm_head"], self.w8["lm_head_s"] = ops.quantize_fp8_rows(lm_head)
        del lm_head
        inv = 1.0 / (self.config.rope_theta ** (torch.arange(0, self.D, 2, dtype=torch.int64).float() / self.D))
        self.w["inv_freq"] = inv.to(dev)
        # one table for every position the model can see (8 MB at 32768 x 64): captured graphs keep its address
        self._rope_tab = ops.rope_table(int(getattr(self.config, "max_position_embeddings", 32768) or 32768), self.D,
                                        self.config.rope_theta, dev, self.dtype)
        self.device = dev
        self.is_loaded = True
        return self

    @property
    def embed_tokens(self) -> torch.Tensor:
        return self.w["embed"]

    def rope_table(self, n_pos: int) -> torch.Tensor:
        """Packed bf16 (cos, sin) of every (position, frequency), built once at load."""
        if self._rope_tab.shape[0] < n_pos:
            raise ValueError(f"sequence of {n_pos} positions exceeds max_position_embeddings ({self._rope_tab.shape[0]})")
        return self._rope_tab

    # ---- prefill ---------------------------------------------------------------------------------------------
    def _layer(self, L, x: torch.Tensor, S: int, pos0: int, qkv_out: Optional[torch.Tensor], ss_x: torch.Tensor):
        """One decoder layer.  ss_x [S, parts]: partial sums of squares of the incoming residual stream's rows.
        Returns (outgoing stream, its partial sums of squares [S, H/32] written by the down_proj epilogue)."""
        Hq, Hkv, D = self.Hq, self.Hkv, self.D
        # RMSNorm scale, bias and RoPE all happen in this GEMM's epilogue; K / V land in the cache layout directly
        qkv = ops.gemm(x, L["wqkv"], bias=L.get("bqkv"), out=qkv_out, rms_in=ss_x, rms_eps=self.eps,
                       rope=(self.rope_table(pos0 + S), pos0, D, (Hq + Hkv) * D))
        o = ops.attention(qkv[:, : Hq * D], qkv[:, Hq * D: (Hq + Hkv) * D], qkv[:, (Hq + Hkv) * D:], B=1, S=S, Hq=Hq,
                          Hkv=Hkv, D=D, causal=True, scale=D ** -0.5)
        ss_mid = torch.empty((S, self.H // 32), device=x.device, dtype=torch.float32)
        x = ops.gemm(o, L["wo"], residual=x, sumsq_out=ss_mid)                      # stats of the mid-layer stream
        h = ops.gemm(x, L["wgu"], act=ops.ACT_SWIGLU, rms_in=ss_mid, rms_eps=self.eps)
        ss_out = torch.empty((S, self.H // 32), device=x.device, dtype=torch.float32)
        x = ops.gemm(h, L["wd"], residual=x, sumsq_out=ss_out)                      # stats for the next layer
        return x, ss_out

    def prefill(self, embeds: torch.Tensor, all_logits: bool = False, keep_cache: bool = False,
                max_len: Optional[int] = None, _no_graph: bool = False, tap=None):
        """embeds [S,H] bf16 -> (logits fp32 [S,V] or [1,V], final hidden [S,H] or None when graph-replayed).
        `tap(layer_index, stream)` (parity checks only) sees the residual stream after every layer; it forces the
        eager path."""
        if not self.is_loaded:
            raise RuntimeError("DecoderEngine: weights not loaded")
        if self._graphed is not None and not _no_graph and not all_logits and not keep_cache and tap is None:
            return self._graphed(embeds.contiguous()), None
        S = embeds.shape[0]
        x = embeds
        if keep_cache:
            self._ensure_cache(max_len or S, x.device)
            self.kv_len = S
        ss_x = ops.row_sumsq(x)
        for i, L in enumerate(self.layers):
            x, ss_x = self._layer(L, x, S, 0, self.kv[i][:S] if keep_cache else None, ss_x)
            if tap is not None:
                tap(i, x)
        if all_logits:
            logits = ops.gemm(x, self.w["lm_head"], out_dtype=torch.float32, rms_in=ss_x, rms_eps=self.eps)
        else:
            logits = ops.gemv(x[S - 1:].contiguous(), self.w["lm_head"], rms_eps=self.eps, out_dtype=torch.float32)
        return logits, x

    def _ensure_cache(self, cap: int, device) -> None:
        """The per-layer fused-row cache is allocated once and reused (a captured decode graph holds its addresses)."""
        if self.kv and self.kv[0].shape[0] >= cap and self.kv[0].device == torch.device(device):
            return
        cap = (cap + 255) // 256 * 256
        width = (self.Hq + 2 * self.Hkv) * self.D
        self.kv = [torch.empty((cap, width), device=device, dtype=self.dtype) for _ in self.layers]
        self._decode_graph = None

    # ---- KV-cache decode (one token) -----------------------------------------------------------------------
    def _decode_set(self):
        """(per-layer weight dicts, dict holding lm_head) that decode streams.  The fp8 dicts hold every weight `k` as
        float8_e4m3fn with its per-row scale under `k + "_s"`; the 16-bit dicts have no scales (w_scale=None)."""
        return (self.layers8, self.w8) if self.decode_weights == "fp8" else (self.layers, self.w)

    def decode_step(self, x: torch.Tensor) -> torch.Tensor:
        """x [1,H] bf16 (embedding of the newest token) -> logits fp32 [1,V]; appends K/V at position kv_len.
        Every linear layer is a weight-streaming GEMV with the RMSNorm in front of it fused (vl2_gemv_bf16, or
        vl2_gemv_fp8 with decode_weights="fp8"), attention is the split-KV vl2_attention_decode."""
        if not self.kv:
            raise RuntimeError("decode_step needs prefill(keep_cache=True) first")
        pos = self.kv_len
        if pos >= self.kv[0].shape[0]:
            raise RuntimeError(f"KV cache full ({pos} positions)")
        Hq, Hkv, D = self.Hq, self.Hkv, self.D
        layers, head = self._decode_set()
        for i, L in enumerate(layers):
            cache = self.kv[i]
            row = cache[pos:pos + 1]
            ops.gemv(x, L["wqkv"], w_scale=L.get("wqkv_s"), bias=L.get("bqkv"), out=row, rms_eps=self.eps)
            ops.rope_inplace(row, 1, Hq, Hkv, D, 0, Hq * D, pos, self.w["inv_freq"], interleaved=True)
            o = ops.attention_decode(row[0, : Hq * D], cache[:, Hq * D: (Hq + Hkv) * D], cache[:, (Hq + Hkv) * D:],
                                     n_pos=pos + 1, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5)
            x = ops.gemv(o, L["wo"], w_scale=L.get("wo_s"), residual=x)
            h = ops.gemv(x, L["wgu"], w_scale=L.get("wgu_s"), act=ops.ACT_SWIGLU, rms_eps=self.eps)
            x = ops.gemv(h, L["wd"], w_scale=L.get("wd_s"), residual=x)
        self.kv_len = pos + 1
        return ops.gemv(x, head["lm_head"], w_scale=head.get("lm_head_s"), rms_eps=self.eps, out_dtype=torch.float32)

    # ---- the same step as ONE CUDA graph ---------------------------------------------------------------------
    def _decode_body(self, tok_dev: torch.Tensor, pos_dev: torch.Tensor, stage: torch.Tensor, log=None) -> torch.Tensor:
        """Single-token step whose position and token live in device memory: embeds *tok_dev, appends K/V at *pos_dev,
        writes argmax(logits) back to tok_dev and increments pos_dev, so one captured graph serves every token."""
        Hq, Hkv, D = self.Hq, self.Hkv, self.D
        x = torch.index_select(self.w["embed"], 0, tok_dev)
        o = torch.empty((1, Hq * D), device=x.device, dtype=self.dtype)
        layers, head = self._decode_set()
        for i, L in enumerate(layers):
            cache = self.kv[i]
            ops.gemv(x, L["wqkv"], w_scale=L.get("wqkv_s"), bias=L.get("bqkv"), out=stage, rms_eps=self.eps)
            joined = None
            if self.decode_prefetch_mb > 0:       # fork: weight prefetch into L2 next to the attention phase
                main = torch.cuda.current_stream()
                if self._side_stream is None:
                    self._side_stream = torch.cuda.Stream(device=x.device)
                fork = torch.cuda.Event()
                fork.record(main)
                self._side_stream.wait_event(fork)
                with torch.cuda.stream(self._side_stream):
                    budget = int(self.decode_prefetch_mb * 1e6)
                    n_wo = L["wo"].numel() * L["wo"].element_size()
                    ops.l2_prefetch(L["wo"], min(budget, n_wo))
                    if budget > n_wo:
                        ops.l2_prefetch(L["wgu"], budget - n_wo)
                    joined = torch.cuda.Event()
                    joined.record(self._side_stream)
            ops.decode_rope_append(stage, cache, pos_dev, Hq, Hkv, D, self.w["inv_freq"], interleaved=True)
            ops.attention_decode_dyn(stage[0, : Hq * D], cache[:, Hq * D: (Hq + Hkv) * D], cache[:, (Hq + Hkv) * D:],
                                     pos_dev, Hq=Hq, Hkv=Hkv, D=D, scale=D ** -0.5, out=o)
            if joined is not None:
                torch.cuda.current_stream().wait_event(joined)
            x = ops.gemv(o, L["wo"], w_scale=L.get("wo_s"), residual=x)
            h = ops.gemv(x, L["wgu"], w_scale=L.get("wgu_s"), act=ops.ACT_SWIGLU, rms_eps=self.eps)
            x = ops.gemv(h, L["wd"], w_scale=L.get("wd_s"), residual=x)
        logits = ops.gemv(x, head["lm_head"], w_scale=head.get("lm_head_s"), rms_eps=self.eps, out_dtype=torch.float32)
        tok_dev.copy_(torch.argmax(logits, dim=1))
        pos_dev.add_(1)
        if log is not None:          # device-side log of the generated ids: the host reads it in chunks, not per token
            gen_buf, step_dev = log
            gen_buf.scatter_(0, step_dev, tok_dev)
            step_dev.add_(1)
        return logits

    def decode_graph_begin(self, first_token: int) -> None:
        """Arm the graph-replayed decode loop after prefill(keep_cache=True): token := first_token, pos := kv_len."""
        if not self.kv:
            raise RuntimeError("decode_graph_begin needs prefill(keep_cache=True) first")
        dev = self.kv[0].device
        if self._decode_graph is None:
            tok_dev = torch.zeros((1,), device=dev, dtype=torch.int64)
            pos_dev = torch.zeros((1,), device=dev, dtype=torch.int32)
            stage = torch.empty((1, (self.Hq + 2 * self.Hkv) * self.D), device=dev, dtype=self.dtype)
            gen_buf = torch.zeros((self.kv[0].shape[0] + 1,), device=dev, dtype=torch.int64)
            step_dev = torch.zeros((1,), device=dev, dtype=torch.int64)
            log = (gen_buf, step_dev)
            scratch_pos = self.kv[0].shape[0] - 1     # warm-up writes land in the last cache row (rewritten when reached)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    pos_dev.fill_(scratch_pos)
                    step_dev.zero_()
                    with ops.pdl(self.decode_pdl):
                        self._decode_body(tok_dev, pos_dev, stage, log)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph), ops.pdl(self.decode_pdl):
                logits = self._decode_body(tok_dev, pos_dev, stage, log)
            self._decode_graph = (graph, tok_dev, pos_dev, logits, stage)
            self._decode_log = log
        _, tok_dev, pos_dev, _, _ = self._decode_graph
        tok_dev.fill_(int(first_token))
        pos_dev.fill_(self.kv_len)
        self._decode_log[1].zero_()
        self._decode_read = 0

    def decode_graph_run(self, k: int) -> None:
        """Enqueue k token steps back to back (no host round trip in between: each replay embeds the token the previous one
        left in device memory and logs its own arg-max into the device-side id buffer)."""
        graph = self._decode_graph[0]
        if self.kv_len + k > self.kv[0].shape[0]:
            raise RuntimeError(f"KV cache full ({self.kv_len} + {k} positions)")
        for _ in range(k):
            graph.replay()
        self.kv_len += k

    def decode_graph_tokens(self, k: int) -> list:
        """The next k logged token ids (one device->host copy, one synchronisation for the whole chunk)."""
        a = self._decode_read
        self._decode_read = a + k
        return self._decode_log[0][a:a + k].tolist()

    def decode_graph_step(self) -> torch.Tensor:
        """Replay one token; returns the device int64[1] holding the NEW token (argmax), logits stay in the graph's
        static buffer (`decode_graph_logits`)."""
        graph, tok_dev, _, _, _ = self._decode_graph
        if self.kv_len >= self.kv[0].shape[0]:
            raise RuntimeError(f"KV cache full ({self.kv_len} positions)")
        graph.replay()
        self.kv_len += 1
        return tok_dev

    @property
    def decode_graph_logits(self) -> torch.Tensor:
        return self._decode_graph[3]
