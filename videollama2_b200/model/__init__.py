"""Model registry + loader with the reference's names (videollama2/model/__init__.py:31-193)."""
from __future__ import annotations

import json
import os

import torch

from .config import Videollama2Config, VisionConfig
from .decoder import check_decode_weights
from .encoder import CLIPVisionTower, SiglipVisionTower, build_vision_tower
from .projector import STCConnector, STCConnectorV35, build_vision_projector, load_mm_projector
from .videollama2_mistral import Videollama2MistralConfig, Videollama2MistralForCausalLM
from .videollama2_qwen2 import Videollama2Qwen2Config, Videollama2Qwen2ForCausalLM

VLLMs = {
    "videollama2": Videollama2MistralForCausalLM,
    "videollama2_mistral": Videollama2MistralForCausalLM,
    "videollama2_qwen2": Videollama2Qwen2ForCausalLM,
}

VLLMConfigs = {
    "videollama2": Videollama2MistralConfig,
    "videollama2_mistral": Videollama2MistralConfig,
    "videollama2_qwen2": Videollama2Qwen2Config,
}


def _read_checkpoint(model_path: str):
    """HF checkpoint directory -> state dict (sharded safetensors or pytorch_model.bin)."""
    idx = os.path.join(model_path, "model.safetensors.index.json")
    files = []
    if os.path.exists(idx):
        with open(idx) as fh:
            files = sorted(set(json.load(fh)["weight_map"].values()))
    elif os.path.exists(os.path.join(model_path, "model.safetensors")):
        files = ["model.safetensors"]
    sd = {}
    if files:
        from safetensors.torch import load_file
        for f in files:
            sd.update(load_file(os.path.join(model_path, f)))
        return sd
    binf = os.path.join(model_path, "pytorch_model.bin")
    if os.path.exists(binf):
        return torch.load(binf, map_location="cpu")
    raise FileNotFoundError(f"no model.safetensors[.index.json] / pytorch_model.bin under {model_path}")


_TOWER_PFX = "model.vision_tower.vision_tower."


def _read_tower_checkpoint(tower_dir: str):
    """A local HF CLIPVisionModel / SiglipVisionModel (or full CLIPModel / SiglipModel) checkpoint -> the reference's
    names (`model.vision_tower.vision_tower.vision_model.*`, encoder.py:26-29: the tower wraps the HF model as
    `self.vision_tower`)."""
    raw = _read_checkpoint(tower_dir)
    out = {}
    for k, v in raw.items():
        if k.startswith("vision_model."):
            out[_TOWER_PFX + k] = v
    if not out:
        raise ValueError(f"{tower_dir}: no `vision_model.*` tensors in the tower checkpoint")
    return out


def assemble_state_dict(model_path: str, model_base=None, config=None):
    """The reference's two full-weight loading branches (model/__init__.py:138-180) for LOCAL directories:
      * SFT checkpoint (model_base None): every tensor comes from `model_path`;
      * base + projector (model/__init__.py:138-164): the LLM from `model_base`, `mm_projector.bin` from `model_path`
        (projector.py:49-63, same `model.mm_projector.*` names), and the vision tower from the local directory named by
        `config.mm_vision_tower` (the reference constructs the tower un-initialised in this branch and relies on the
        training script's `load_pretrained=True`; an inference engine has to read it from somewhere).
    Returns an HF-named state dict ready for `from_state_dict`."""
    if model_base is None:
        return _read_checkpoint(model_path)
    sd = dict(_read_checkpoint(model_base))
    proj = load_mm_projector(model_path)
    sd.update({k: v for k, v in proj.items()})
    tower = getattr(config, "mm_vision_tower", None) if config is not None else None
    if tower is not None and not any(k.startswith(_TOWER_PFX) for k in sd):
        if not os.path.isdir(tower):
            raise FileNotFoundError(f"base+projector loading needs the vision tower weights in a local directory; "
                                    f"mm_vision_tower='{tower}' is not one")
        sd.update(_read_tower_checkpoint(tower))
    return sd


def load_pretrained_model(model_path, model_base=None, model_name=None, load_8bit=False, load_4bit=False,
                          device_map="auto", device="cuda", use_flash_attn=False, decode_weights="bf16", **kwargs):
    """The reference loader (model/__init__.py:48-193) for LOCAL directories: the SFT-checkpoint branch (:165-180) and the
    base + `mm_projector.bin` branch (:138-164); returns (tokenizer, model, image_processor, context_len).  LoRA / 4-bit /
    8-bit branches are training artefacts outside the accelerated path.  `decode_weights="fp8"`: fp8 E4M3 weights for the
    KV-cache decode steps only (see Videollama2MistralForCausalLM.from_state_dict)."""
    check_decode_weights(decode_weights)
    if load_8bit or load_4bit:
        raise NotImplementedError("bitsandbytes loading is not supported by the B200 engine")
    if model_name and "lora" in model_name.lower():
        raise NotImplementedError("LoRA-adapter loading is not supported by the B200 engine (merge the adapter first)")
    with open(os.path.join(model_path, "config.json")) as fh:
        raw = json.load(fh)
    model_type = raw.get("model_type", "videollama2_mistral")
    if model_type not in VLLMs:
        raise ValueError(f"unsupported model_type {model_type} (supported: {sorted(VLLMs)})")
    config = VLLMConfigs[model_type].from_dict(raw)
    config.model_type = model_type
    tower = config.mm_vision_tower
    if "vision_config" in raw:
        config.vision_config = VisionConfig.from_dict(raw["vision_config"], hint=tower or "")
    elif tower is not None:
        config.vision_config = VisionConfig.from_dir(tower)     # local directory, or a known hub id (built-in dims)
    sd = assemble_state_dict(model_path, model_base, config)
    model = VLLMs[model_type].from_state_dict(config, sd, device=device, decode_weights=decode_weights)
    from transformers import AutoTokenizer
    # the reference loads the SLOW tokenizer for every videollama2 branch (model/__init__.py:146,167): fast and slow
    # Llama / Mistral tokenizers can split differently around special tokens, and tokenizer_multimodal_token tokenizes
    # the prompt chunk by chunk
    tok_dir = model_base if model_base is not None else model_path
    try:
        tokenizer = AutoTokenizer.from_pretrained(tok_dir, use_fast=False)
    except (ValueError, ImportError, OSError):                  # checkpoint ships tokenizer.json only
        tokenizer = AutoTokenizer.from_pretrained(tok_dir, use_fast=True)
    processor = None
    if config.mm_vision_tower is not None:
        processor = model.get_vision_tower().image_processor
    context_len = raw.get("max_sequence_length", 2048)
    return tokenizer, model, processor, context_len
