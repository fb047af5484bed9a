"""Regenerate tests/golden/reference_calls.pt: what the REAL reference returned for the calls that tests/test_oracle.py and
tests/test_host_logic.py compare against (the tiny model's fp32 logits and STC connector output, its state-dict
names / shapes, tokenizer_multimodal_token, mm_infer, KeywordsStoppingCriteria), so those comparisons run everywhere.
TEST INFRASTRUCTURE.  Needs the reference tree (oracle/ref_loader.py):  python -m oracle.make_golden_calls"""
from __future__ import annotations

import importlib
import os

import torch

from . import mm_infer_ref, ref_loader, synth
from .make_golden import OUT, PROMPTS, ToyTokenizer

PATH = os.path.join(OUT, "reference_calls.pt")
TOKENIZER_PROMPTS = PROMPTS + [("a <video> b <video> c", "<video>"), ("", "<video>")]
STC_SEED = 11


def stc_input(cfg) -> torch.Tensor:
    """A batch of two 4-frame videos of vision features for the connector alone."""
    return torch.randn((2, 4, 16, cfg.vision.hidden), generator=torch.Generator().manual_seed(STC_SEED))


class DecodingToyTokenizer:
    """Word-piece toy with a decoder: id 3 + i <-> _VOCAB[i]; pieces are concatenated without spaces, so a keyword can
    straddle several ids (what the decoded-text branch of KeywordsStoppingCriteria exists for)."""
    bos_token_id = 1
    _VOCAB = ["he", "llo", " wor", "ld", "hello!", " stop", "x", "y"]

    class _Enc:
        def __init__(self, ids):
            self.input_ids = ids

    def __call__(self, text, add_special_tokens=True):
        ids, rest = [], text
        while rest:
            for i, p in sorted(enumerate(self._VOCAB), key=lambda t: -len(t[1])):
                if rest.startswith(p):
                    ids.append(3 + i)
                    rest = rest[len(p):]
                    break
            else:
                raise ValueError(rest)
        return self._Enc(([self.bos_token_id] if add_special_tokens else []) + ids)

    def batch_decode(self, ids, skip_special_tokens=True):
        return ["".join(self._VOCAB[int(t) - 3] for t in row if int(t) >= 3) for row in ids]


def keyword_cases(tok):
    """Output-id sequences for KeywordsStoppingCriteria(["hello"]): the keyword spelled by its own ids, by one id for
    "hello!", absent, at the start, not at the tail, and batches of two."""
    kw = tok("hello", add_special_tokens=False).input_ids             # ["he", "llo"]
    bang = tok("hello!", add_special_tokens=False).input_ids          # one id spelling "hello!"
    x, y = tok("x", add_special_tokens=False).input_ids[0], tok("y", add_special_tokens=False).input_ids[0]
    return [torch.tensor([[x, y] + kw]), torch.tensor([[x, y, x] + bang]), torch.tensor([[x, y, x, y]]),
            torch.tensor([bang]), torch.tensor([[x] + bang + [y, y, y, y]]), torch.tensor([[x, y, y] + bang + [y]]),
            torch.tensor([[x, y] + kw, [x, y, y, y]]), torch.tensor([[x] + kw, [y] + kw])]


def main():
    ref_loader.load()
    ref_mm = importlib.import_module("videollama2.mm_utils")
    cfg = synth.CONFIGS["tiny"]
    sd = synth.state_dict(cfg)
    px, ids = synth.inputs(cfg)
    m = ref_loader.build_reference_model(cfg, torch.float32, sd)
    stc_in = stc_input(cfg)
    with torch.no_grad():
        logits = m(input_ids=ids, attention_mask=torch.ones_like(ids), images=[(px.float(), "video")]).logits[0]
        stc_out = m.get_model().mm_projector(stc_in)
    tok = ToyTokenizer()
    instruct, modal, mtype, kw = mm_infer_ref.CASES[0]
    text, call = mm_infer_ref.run_reference(instruct, modal, mtype, torch.zeros((2, 3, 4, 4)), **kw)
    dtok = DecodingToyTokenizer()
    stop = ref_mm.KeywordsStoppingCriteria(["hello"], dtok, torch.zeros(1, 2, dtype=torch.long))
    out = {
        "tiny_logits": logits.float(),
        "stc_seed": STC_SEED,
        "stc_out": stc_out.float(),
        "state_dict_shapes": {k: tuple(v.shape) for k, v in m.state_dict().items()},
        "tokenizer": [(p, t, ref_mm.tokenizer_multimodal_token(p, tok, t)) for p, t in TOKENIZER_PROMPTS],
        "mm_infer": {"case": 0, "text": text, "input_ids": mm_infer_ref.summarise(call)["input_ids"]},
        "keywords_hello": [bool(stop(c, None)) for c in keyword_cases(dtok)],
    }
    torch.save(out, PATH)
    print("wrote", PATH, {k: tuple(v.shape) for k, v in out.items() if isinstance(v, torch.Tensor)}, out["keywords_hello"])


if __name__ == "__main__":
    main()
