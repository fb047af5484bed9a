"""Vision mixins + embedding splice with the reference's method names and semantics
(videollama2/model/videollama2_arch.py:28-263), running on libvl2 kernels."""
from __future__ import annotations

import collections

from typing import Dict, List, Optional

import torch

from .. import mm_utils, ops
from ..constants import IGNORE_INDEX, MODAL_INDEX_MAP, NUM_FRAMES
from .decoder import DecoderEngine, check_decode_weights
from .encoder import build_vision_tower
from .projector import build_vision_projector


class Videollama2MetaModel:
    """Holds the tower, the projector and the decoder (reference: Videollama2MetaModel + the HF *Model it is mixed into)."""

    def __init__(self, config, tp_group=None, decode_weights: str = "bf16"):
        self.config = config
        check_decode_weights(decode_weights)
        if tp_group is not None and decode_weights != "bf16":
            raise NotImplementedError("decode_weights='fp8' is not supported with a tensor-parallel decoder")
        self.vision_tower = None
        self.mm_projector = None
        if getattr(config, "mm_vision_tower", None) is not None:
            self.vision_tower = build_vision_tower(config)
            self.mm_projector = build_vision_projector(config)
        if tp_group is not None:        # tensor-parallel decoder over the ranks of `tp_group` (True = the default group)
            from .tp_decoder import TPDecoderEngine
            self.decoder = TPDecoderEngine(config, None if tp_group is True else tp_group)
        else:
            self.decoder = DecoderEngine(config, decode_weights=decode_weights)

    def get_vision_tower(self):
        vision_tower = getattr(self, "vision_tower", None)
        if type(vision_tower) is list:
            vision_tower = vision_tower[0]
        return vision_tower

    def embed_tokens(self, ids: torch.Tensor) -> torch.Tensor:
        """Embedding lookup through the gather kernel (ids >= 0)."""
        bad = (ids < 0) | (ids >= self.config.vocab_size)
        if bool(bad.any()):     # the reference's nn.Embedding raises on these (e.g. a modal placeholder left without images)
            raise IndexError(f"embed_tokens: id {int(ids[bad].reshape(-1)[0])} outside [0, {self.config.vocab_size})")
        flat = ids.reshape(-1).to(device=self.decoder.device, dtype=torch.int64).contiguous()
        out = torch.empty((flat.numel(), self.config.hidden_size), device=self.decoder.device, dtype=self.decoder.dtype)
        if flat.numel():
            dst = torch.arange(flat.numel(), device=self.decoder.device, dtype=torch.int32)
            ops.embed_splice(flat, dst, self.decoder.embed_tokens, out)
        return out.view(*ids.shape, self.config.hidden_size)


class Videollama2MetaForCausalLM:
    """Mixin of the *ForCausalLM wrappers (reference: videollama2_arch.py:98-263)."""

    def get_model(self) -> Videollama2MetaModel:
        raise NotImplementedError

    def num_frames(self):
        return getattr(self.config, "num_frames", NUM_FRAMES)

    def get_vision_tower(self):
        return self.get_model().get_vision_tower()

    # ---- vision-feature cache (SURVEY.md §8f row 1) -----------------------------------------------------------
    def enable_vision_cache(self, entries: int = 2):
        """The reference's eval runners call mm_infer twice per video (eval/inference_video_mcqa_videomme.py:275,279,
        inference_video_oqa_vcgpt_consistency.py:106,115) and re-encode the same frames each time.  With the cache on,
        `encode_images_or_videos` keys its result on a 128-bit content checksum of the frame tensor (computed on the
        device, one pass over the pixels) plus shape / modality, and returns the stored visual tokens on a hit.
        Off by default: identical semantics to the reference either way, the cache only skips recomputation."""
        self._vision_cache = collections.OrderedDict() if entries > 0 else None
        self._vision_cache_entries = entries
        self.vision_cache_hits = 0
        return self

    @staticmethod
    def _content_key(images):
        keys = []
        for data, modal in images:
            w = data.contiguous().view(torch.uint8).view(-1)
            pad = (-w.numel()) % 8
            if pad:
                w = torch.cat([w, w.new_zeros(pad)])
            w = w.view(torch.int64)
            idx = torch.arange(1, w.numel() + 1, device=w.device, dtype=torch.int64)
            h = torch.stack([w.sum(), (w * (2 * idx + 1)).sum()])        # wrap-around int64 arithmetic: two checksums
            keys.append((modal, tuple(data.shape), str(data.dtype), tuple(int(v) for v in h.tolist())))
        return tuple(keys)

    def encode_images_or_videos(self, images):
        cache = getattr(self, "_vision_cache", None)
        if cache is not None:
            key = self._content_key(images)
            hit = cache.get(key)
            if hit is not None:
                cache.move_to_end(key)
                self.vision_cache_hits += 1
                return hit
            out = self._encode_images_or_videos(images).clone()   # the stages' graph buffers are reused: keep a copy
            cache[key] = out
            while len(cache) > self._vision_cache_entries:
                cache.popitem(last=False)
            return out
        return self._encode_images_or_videos(images)

    # ---- frame-parallel vision stage (videollama2_b200/parallel.py) ---------------------------------------------
    def enable_frame_parallel(self, group=None, shard_s1: bool = True, llm_rank: int = 0):
        """Shard the per-frame part of `encode_images_or_videos` (ViT + first RegStage) over the ranks of `group` and
        all-gather before the connector's Conv3d.  Every rank must then call encode / forward / generate with identical
        inputs; ranks other than `llm_rank` return None from forward / generate once the collective is done
        (`llm_rank=None`: every rank goes on to the decoder - the tensor-parallel configuration).
        `group=None` with an initialised default process group uses WORLD; call with `group=False` to switch it off."""
        from .. import parallel
        if group is False:
            self._frame_parallel = None
        else:
            self._frame_parallel = parallel.FrameParallel(group, shard_s1=shard_s1, llm_rank=llm_rank)
        return self

    def _vision_only_rank(self, images) -> bool:
        """True on a frame-parallel rank that does not run the decoder: it takes part in the vision collective and stops."""
        fp = getattr(self, "_frame_parallel", None)
        if fp is None or fp.world == 1 or fp.llm_rank is None or fp.rank == fp.llm_rank or images is None \
                or self.get_vision_tower() is None:
            return False
        self.encode_images_or_videos(images)
        return True

    # arch.py:114-134
    def _encode_images_or_videos(self, images):
        num_frames = getattr(self.config, "num_frames", NUM_FRAMES)
        data_batch = []
        for data, modal in images:
            if modal == "image":
                data = data.expand(num_frames, -1, -1, -1)   # an image is a T-frame still
            data_batch.append(data)
        data_batch = torch.stack(data_batch, dim=0)
        assert len(data_batch.size()) == 5
        b, t = data_batch.size(0), data_batch.size(1)
        frames = data_batch.reshape(b * t, *data_batch.shape[2:])
        fp = getattr(self, "_frame_parallel", None)
        if fp is not None and fp.world > 1 and "tc_connector" in self.config.mm_projector_type:
            return fp.encode(self, frames, b, t)
        frames_features = self.get_model().get_vision_tower()(frames)
        frames_features = frames_features.view(b, t, *frames_features.shape[1:])
        return self.temporal_aggregator(frames_features)

    # aliases named in BASELINE.json
    encode_images = encode_images_or_videos
    encode_videos = encode_images_or_videos

    # arch.py:136-159
    def temporal_aggregator(self, frames_features):
        ptype = self.config.mm_projector_type
        if "tc_connector" in ptype or "tp_connector" in ptype or ptype in ("spatial_conv", "spatial_pool"):
            return self.get_model().mm_projector(frames_features)
        if ptype in ("mlp2x_gelu", "linear"):
            raise NotImplementedError(f"projector type {ptype} is not implemented in the B200 engine")
        raise Exception(f"Unsupported projector type {ptype}!!!")

    # arch.py:161-263
    def prepare_inputs_labels_for_multimodal(self, input_ids, attention_mask, past_key_values, labels, images):
        vision_tower = self.get_vision_tower()
        if vision_tower is None or images is None or input_ids.shape[1] == 1:
            return input_ids, attention_mask, past_key_values, None, labels
        model = self.get_model()
        dev = model.decoder.device
        mm_features = self.encode_images_or_videos(images)            # [n_mm, L, H]
        n_mm, L, H = mm_features.shape
        plan = mm_utils.build_splice(input_ids.cpu(), [L] * n_mm)
        B, max_len = input_ids.shape[0], plan["max_len"]
        ragged = any(n != max_len for n in plan["new_len"])
        alloc = torch.zeros if ragged else torch.empty                # right padding is zeros (arch.py:229-231)
        embeds = alloc((B * max_len, H), device=dev, dtype=model.decoder.dtype)
        if plan["text_dst"]:
            ids_dev = input_ids.to(dev)[torch.tensor(plan["text_b"], device=dev), torch.tensor(plan["text_src"], device=dev)]
            dst = torch.tensor(plan["text_dst"], device=dev, dtype=torch.int32)
            ops.embed_splice(ids_dev.contiguous(), dst, model.decoder.embed_tokens, embeds)
        for mm_idx, b, pos, n in plan["mm_dst"]:
            embeds[b * max_len + pos: b * max_len + pos + n].copy_(mm_features[mm_idx].to(model.decoder.dtype))
        embeds = embeds.view(B, max_len, H)
        new_labels = labels
        if labels is not None:
            new_labels = mm_utils.spliced_labels(labels, input_ids.cpu(), [L] * n_mm, max_len)
        if attention_mask is not None:
            attention_mask = mm_utils.spliced_attention_mask(attention_mask, input_ids.shape[1], plan["new_len"], max_len)
        self._last_new_len = plan["new_len"]
        return None, attention_mask, past_key_values, embeds, new_labels
