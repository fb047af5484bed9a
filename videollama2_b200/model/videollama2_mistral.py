"""Videollama2MistralForCausalLM with the reference's call surface (videollama2/model/videollama2_mistral.py:47-153),
backed by the B200 engine instead of HF MistralForCausalLM."""
from __future__ import annotations

from types import SimpleNamespace
from typing import Dict, List, Optional

import torch

from .. import ops
from .config import Videollama2Config
from .decoder import check_decode_weights
from .videollama2_arch import Videollama2MetaForCausalLM, Videollama2MetaModel


class Videollama2MistralConfig(Videollama2Config):
    model_type = "videollama2_mistral"


class CausalLMOutput(SimpleNamespace):
    """Field-compatible with transformers' CausalLMOutputWithPast for what callers read (.logits, .loss, .labels)."""

    def __getitem__(self, i):
        return (self.loss, self.logits)[i] if self.loss is not None else (self.logits,)[i]


class EngineKVCache:
    """What `forward(use_cache=True)` returns as `past_key_values`: a handle to the K/V rows the decoder engine holds for
    the ONE sequence it is decoding (the engine owns a single per-layer cache; a handle is valid until the next prefill).
    Passing it back with one new token runs a single-token decode step - the call pattern of HF's generation loop
    (videollama2_mistral.py:63-108 forwards `past_key_values` to the HF decoder)."""

    def __init__(self, engine, serial):
        self.engine, self.serial = engine, serial

    def get_seq_length(self, layer_idx: int = 0) -> int:
        return self.engine.kv_len


class Videollama2MistralForCausalLM(Videollama2MetaForCausalLM):
    config_class = Videollama2MistralConfig

    def __init__(self, config, tp_group=None, decode_weights: str = "bf16", **kwargs):
        self.config = config
        self.model = Videollama2MetaModel(config, tp_group=tp_group, decode_weights=decode_weights)
        self.vocab_size = config.vocab_size
        self._device = torch.device("cpu")

    # ---- construction -----------------------------------------------------------------------------------------
    @classmethod
    def from_state_dict(cls, config, state_dict: Dict[str, torch.Tensor], device="cuda", tp_group=None, dtype=None,
                        decode_weights: str = "bf16"):
        """Build from HF-named weights (the reference's checkpoint format, SURVEY.md §8b) and repack for the kernels.
        `tp_group` (a process group, or True for the default one): shard the decoder tensor-parallel over its ranks
        (model/tp_decoder.py); every rank passes the same full state dict and keeps its slices.
        `dtype`: torch.bfloat16 (default) or torch.float16 - the storage type of weights and activations; float16 runs the
        fp16 build of the kernel library (libvl2_f16.so), matching the reference's `torch_dtype=float16` loading.
        `decode_weights`: "bf16" (default) - KV-cache decode streams the same 16-bit weights as prefill; "fp8" - decode
        streams fp8 E4M3 copies of every decoder linear weight and lm_head (one fp32 scale per output row, ~1 byte per
        parameter of extra device memory): about half the bytes per generated token.  Prefill, and so the first new token,
        is unchanged; later tokens follow the fp8-quantised model.  Not available with `tp_group`."""
        check_decode_weights(decode_weights)
        if dtype is not None:          # torch.float16 (the reference's inference dtype) or torch.bfloat16
            config.torch_dtype = str(dtype).replace("torch.", "")
        self = cls(config, tp_group=tp_group, decode_weights=decode_weights)
        self.load_state_dict(state_dict, device)
        return self

    def load_state_dict(self, sd: Dict[str, torch.Tensor], device="cuda", presharded: bool = False):
        """`presharded` (tensor-parallel decoder only): the decoder tensors in `sd` are already this rank's slices
        (tp_decoder.shard_state_dict layout) - how a 72B checkpoint is loaded without any rank holding all of it."""
        dev = torch.device(device)
        m = self.model
        if presharded:
            m.decoder.load_state_dict(sd, dev, presharded=True)
        else:
            m.decoder.load_state_dict(sd, dev)
        if m.vision_tower is not None:
            m.vision_tower.load_state_dict(sd, dev, prefix="model.vision_tower.vision_tower.vision_model.")
            m.mm_projector.load_state_dict(sd, dev, prefix="model.mm_projector.")
        self._device = dev
        return self

    def get_model(self):
        return self.model

    @property
    def device(self):
        return self._device

    @property
    def dtype(self):
        return self.config.storage_dtype

    def eval(self):
        return self

    def enable_cuda_graphs(self, on: bool = True):
        """Replay tower / connector / prefill as CUDA graphs (one per input shape)."""
        m = self.model
        if m.vision_tower is not None:
            m.vision_tower.enable_cuda_graphs(on)
            m.mm_projector.enable_cuda_graphs(on)
        m.decoder.enable_cuda_graphs(on)
        return self

    # ---- forward (videollama2_mistral.py:63-108) -----------------------------------------------------------------
    @torch.no_grad()
    def forward(self, input_ids=None, attention_mask=None, position_ids=None, past_key_values=None, inputs_embeds=None,
                labels=None, use_cache=None, output_attentions=None, output_hidden_states=None, images=None,
                return_dict=None, **kwargs):
        if output_attentions:
            raise NotImplementedError("output_attentions is not supported by the fused attention kernel")
        dec = self.get_model().decoder
        if past_key_values is not None:
            # single-token continuation on the engine's cache (HF generation-loop call pattern)
            if not isinstance(past_key_values, EngineKVCache) or past_key_values.engine is not dec or \
                    past_key_values.serial != getattr(self, "_cache_serial", None):
                raise ValueError("past_key_values must be the handle returned by this model's last forward(use_cache=True)")
            x = inputs_embeds if inputs_embeds is not None else self.get_model().embed_tokens(input_ids)
            if x.dim() == 3:
                x = x[0]
            if x.shape[0] != 1:
                raise NotImplementedError("forward(past_key_values=...) takes exactly one new token")
            logits = dec.decode_step(x.to(dec.dtype).contiguous())
            return CausalLMOutput(loss=None, logits=logits.view(1, 1, -1), past_key_values=past_key_values,
                                  hidden_states=None, attentions=None)
        if inputs_embeds is None and input_ids is not None and input_ids.shape[1] != 1 and self._vision_only_rank(images):
            return None
        new_len = None
        if inputs_embeds is None:
            input_ids, attention_mask, past_key_values, inputs_embeds, labels = \
                self.prepare_inputs_labels_for_multimodal(input_ids, attention_mask, past_key_values, labels, images)
            if inputs_embeds is None:   # text-only early-out (arch.py:166-169)
                inputs_embeds = self.get_model().embed_tokens(input_ids)
            else:
                new_len = self._last_new_len
        if inputs_embeds.dim() == 2:
            inputs_embeds = inputs_embeds.unsqueeze(0)
        B, S, _ = inputs_embeds.shape
        logits = torch.zeros((B, S, self.vocab_size), device=inputs_embeds.device, dtype=torch.float32)
        hidden = [] if output_hidden_states else None
        keep = bool(use_cache) and B == 1                           # the engine caches one sequence
        for b in range(B):
            n = S if new_len is None else new_len[b]
            if attention_mask is not None and new_len is None:
                n = int(attention_mask[b].sum().item())            # right padding only (reference convention)
            lg, hx = dec.prefill(inputs_embeds[b, :n].to(dec.dtype).contiguous(), all_logits=True, keep_cache=keep,
                                 max_len=n + int(kwargs.get("cache_extra_positions", 1024)) if keep else None)
            logits[b, :n] = lg
            if hidden is not None:
                hidden.append(hx)
        loss = None
        if labels is not None:
            shift_logits = logits[:, :-1].reshape(-1, self.vocab_size)
            shift_labels = labels[:, 1:].reshape(-1).to(shift_logits.device)
            loss = torch.nn.functional.cross_entropy(shift_logits, shift_labels, ignore_index=-100)
        pkv = None
        if keep:
            self._cache_serial = getattr(self, "_cache_serial", 0) + 1
            pkv = EngineKVCache(dec, self._cache_serial)
        out = CausalLMOutput(loss=loss, logits=logits, past_key_values=pkv, hidden_states=hidden, attentions=None)
        out.labels = labels
        return out

    __call__ = forward

    # ---- generate (videollama2_mistral.py:110-144) -----------------------------------------------------------------
    @torch.no_grad()
    def generate(self, inputs=None, images=None, **kwargs):
        """Greedy decoding, or sampling with HF's temperature / top-k(50) / top-p warpers when do_sample=True (optional
        `generator=` for reproducibility); returns only the NEW token ids (as HF generate does with inputs_embeds)."""
        kwargs.pop("position_ids", None)
        attention_mask = kwargs.pop("attention_mask", None)
        if "inputs_embeds" in kwargs:
            raise NotImplementedError("`inputs_embeds` is not supported")
        sample = bool(kwargs.get("do_sample", False)) and kwargs.get("temperature", 1.0) not in (0, 0.0, None)
        temperature = float(kwargs.get("temperature", 1.0) or 1.0)
        top_p, top_k = float(kwargs.get("top_p", 1.0) or 1.0), int(kwargs.get("top_k", 50) or 0)
        rng = kwargs.get("generator")
        if inputs.shape[0] != 1:
            return self._generate_batch(inputs, images, attention_mask, kwargs)
        max_new = int(kwargs.get("max_new_tokens", 20))
        eos = kwargs.get("eos_token_id", getattr(self.config, "eos_token_id", None))
        eos_ids = set(eos if isinstance(eos, (list, tuple)) else [eos]) if eos is not None else set()
        stopping = kwargs.get("stopping_criteria") or []
        if self._vision_only_rank(images):
            return None
        if images is not None:
            _, attention_mask, _, inputs_embeds, _ = self.prepare_inputs_labels_for_multimodal(
                input_ids=inputs, attention_mask=attention_mask, past_key_values=None, labels=None, images=images)
            if inputs_embeds is None:
                inputs_embeds = self.get_model().embed_tokens(inputs)
        else:
            inputs_embeds = self.get_model().embed_tokens(inputs)
        dec = self.get_model().decoder
        x = inputs_embeds[0].to(dec.dtype).contiguous()
        new_ids: List[int] = []
        # prefill once (keeps per-layer K/V), then one weight-streaming decode step per new token
        use_cache = kwargs.get("use_cache", True)
        S = x.shape[0]
        self._cache_serial = getattr(self, "_cache_serial", 0) + 1        # handles of earlier forward(use_cache=True) calls die here
        logits, _ = dec.prefill(x, all_logits=False, keep_cache=use_cache and max_new > 1, max_len=S + max_new)
        graphed = use_cache and max_new > 1 and dec.graph_decode
        from ..sampling import sample_token
        if graphed and not sample:
            return self._generate_greedy_graphed(dec, logits, max_new, eos_ids, stopping, int(kwargs.get("decode_chunk", 8)))
        for step in range(max_new):
            if sample:      # the graph's own argmax token is overridden below; its logits buffer is what we sample from
                row = logits[0] if not (graphed and step > 0) else dec.decode_graph_logits[0]
                tok = sample_token(row, temperature, top_p, top_k, rng)
            else:
                tok = int(torch.argmax(logits[0]).item()) if not (graphed and step > 0) else int(tok_dev.item())
            new_ids.append(tok)
            out_ids = torch.tensor([new_ids], dtype=torch.long)
            if tok in eos_ids or any(sc(out_ids, None) for sc in stopping) or step == max_new - 1:
                break
            if graphed:   # one graph launch per token: embed, 32 layers, lm_head, argmax all on the device
                if step == 0:
                    dec.decode_graph_begin(tok)
                elif sample:
                    tok_dev.fill_(tok)           # the replay embeds *tok_dev: the sampled token, not the argmax
                tok_dev = dec.decode_graph_step()
                continue
            e = self.get_model().embed_tokens(torch.tensor([tok]))
            if use_cache:
                logits = dec.decode_step(e)
            else:   # exact but O(n^2): re-run the prefill kernels on the grown sequence
                x = torch.cat([x, e], 0)
                logits, _ = dec.prefill(x, all_logits=False)
        return torch.tensor([new_ids], dtype=torch.long, device=self.device)

    def _generate_batch(self, inputs, images, attention_mask, kwargs):
        """Batch > 1 (HF `generate` semantics of videollama2_mistral.py:110-144 for a padded batch): the rows are decoded
        one after the other through the batch-1 path - each row keeps its own real tokens (`attention_mask`), takes the
        images its placeholders consume in order (a row without a placeholder consumes one slot, videollama2_arch.py:181-191)
        - and the new ids are right-padded with `pad_token_id` to the longest row, as HF pads finished sequences."""
        from ..mm_utils import splice_plan
        if kwargs.get("stopping_criteria"):
            raise NotImplementedError("stopping_criteria with batch > 1 (the criteria objects are built for one prompt)")
        B = inputs.shape[0]
        pad = kwargs.get("pad_token_id", getattr(self.config, "pad_token_id", None))
        if pad is None:
            eos = kwargs.get("eos_token_id", getattr(self.config, "eos_token_id", None))
            pad = (eos[0] if isinstance(eos, (list, tuple)) else eos) if eos is not None else 0
        rows, mm = [], 0
        for b in range(B):
            ids = inputs[b]
            if attention_mask is not None:
                ids = ids[attention_mask[b].to(torch.bool).to(ids.device)]
            used = splice_plan(ids.tolist(), [0] * (len(images) if images is not None else 0) + [0], 0)[2] if images is not None else 0
            imgs = images[mm:mm + used] if images is not None else None
            mm += used
            out = self.generate(ids.unsqueeze(0), images=imgs, attention_mask=torch.ones((1, ids.numel()), dtype=torch.bool),
                                **kwargs)
            rows.append(None if out is None else out[0])
        if any(r is None for r in rows):       # a frame-parallel rank that does not decode
            return None
        n = max(int(r.numel()) for r in rows)
        res = torch.full((B, n), int(pad), dtype=torch.long, device=self.device)
        for b, r in enumerate(rows):
            res[b, : r.numel()] = r
        return res

    def _generate_greedy_graphed(self, dec, logits, max_new: int, eos_ids, stopping, chunk: int):
        """Greedy decoding with the host off the critical path: the captured single-token graph feeds itself (token and
        position live in device memory) and appends every arg-max to a device-side id log, so the host enqueues `chunk`
        replays at a time and reads the log once per chunk.  EOS / stopping criteria are evaluated on the host in token
        order; tokens the device produced past the stopping point are discarded (at most chunk - 1 wasted steps), so the
        returned ids equal the token-by-token loop's (tests/test_e2e_gpu.py)."""
        ids_buf = torch.empty((1, max_new), dtype=torch.long)

        def stops(n):          # n = number of ids so far
            tok = int(ids_buf[0, n - 1])
            return tok in eos_ids or any(sc(ids_buf[:, :n], None) for sc in stopping) or n == max_new

        ids_buf[0, 0] = int(torch.argmax(logits[0]).item())
        n = 1
        if not stops(n):
            dec.decode_graph_begin(int(ids_buf[0, 0]))
            done = False
            first = True
            while not done:
                k = min(max_new - n, 2 if first else max(1, chunk))     # a short first chunk: early EOS costs little
                first = False
                dec.decode_graph_run(k)
                for tok in dec.decode_graph_tokens(k):
                    ids_buf[0, n] = tok
                    n += 1
                    if stops(n):
                        done = True
                        break
        return ids_buf[:, :n].to(self.device)

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, inputs_embeds=None, **kwargs):
        images = kwargs.pop("images", None)
        _inputs = {"input_ids": input_ids, "past_key_values": past_key_values, "inputs_embeds": inputs_embeds}
        _inputs.update(kwargs)
        if images is not None:
            _inputs["images"] = images
        return _inputs
