"""Exact (integer) parity of the host-side token / splice logic with the reference
(videollama2/mm_utils.py:277-302, videollama2/model/videollama2_arch.py:161-263) via the committed fixtures, which
record what the reference functions returned."""
import os

import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_tokenizer_multimodal_token_exact():
    from oracle.make_golden import ToyTokenizer
    from oracle import torch_ref
    from videollama2_b200 import mm_utils
    fx = torch.load(os.path.join(GOLD, "tokenizer_multimodal_token.pt"))["tokenizer"]
    tok = ToyTokenizer()
    assert len(fx) >= 6
    for prompt, tag, ref_ids in fx:
        assert mm_utils.tokenizer_multimodal_token(prompt, tok, tag) == ref_ids
        assert torch_ref.tokenizer_multimodal_token(prompt, tok, tag) == ref_ids
        t = mm_utils.tokenizer_multimodal_token(prompt, tok, tag, return_tensors="pt")
        assert t.dtype == torch.long and t.tolist() == ref_ids
    with pytest.raises(ValueError):
        mm_utils.tokenizer_multimodal_token("x", tok, "<video>", return_tensors="np")


@pytest.mark.parametrize("name", ["tiny", "tiny_v35"])
def test_batch_splice_plan_exact(name):
    """Ragged batch of two (placeholder at different positions): new lengths, mask, labels, text-row placement."""
    from oracle import synth
    from videollama2_b200 import mm_utils
    g = torch.load(os.path.join(GOLD, f"{name}.pt"))["splice_batch"]
    cfg = synth.CONFIGS[name]
    ids2 = g["ids"]
    L = cfg.vis_tokens
    plan = mm_utils.build_splice(ids2, [L, L])
    assert plan["max_len"] == g["embeds"].shape[1] and plan["new_len"] == [cfg.prompt - 1 + L] * 2
    mask = mm_utils.spliced_attention_mask(torch.ones_like(ids2, dtype=torch.bool), ids2.shape[1], plan["new_len"], plan["max_len"])
    assert torch.equal(mask, g["mask"])
    labels = mm_utils.spliced_labels(ids2.clone(), ids2, [L, L], plan["max_len"])
    assert torch.equal(labels, g["labels"])
    # text rows land exactly where the reference put them
    table = synth.make_tensor("model.embed_tokens.weight", (cfg.llm.vocab, cfg.llm.hidden), "emb").float()
    emb = g["embeds"].reshape(-1, cfg.llm.hidden)
    for b, src, dst in zip(plan["text_b"], plan["text_src"], plan["text_dst"]):
        assert torch.equal(emb[dst], table[ids2[b, src]])
    assert [(m, b, p, n) for m, b, p, n in plan["mm_dst"]] == [(0, 0, 4, L), (1, 1, 9, L)]


def test_splice_plan_edge_cases():
    from videollama2_b200 import mm_utils
    segs, total, used = mm_utils.splice_plan([5, 6, 7], [10])                 # no placeholder: consumes one slot
    assert segs == [("text", 0, 3)] and total == 3 and used == 1
    segs, total, used = mm_utils.splice_plan([-201], [10])                    # only a placeholder
    assert segs == [("mm", 0, 10)] and total == 10 and used == 1
    segs, total, used = mm_utils.splice_plan([-200, 4, -202], [3, 2])         # image first, audio last
    assert segs == [("mm", 0, 3), ("text", 1, 1), ("mm", 1, 2)] and total == 6 and used == 2
    plan = mm_utils.build_splice(torch.tensor([[1, -201, 2], [3, 4, 5]]), [7, 7])
    assert plan["new_len"] == [9, 3] and plan["max_len"] == 9                 # ragged -> right padding
    m = mm_utils.spliced_attention_mask(torch.ones(2, 3, dtype=torch.bool), 3, plan["new_len"], 9)
    assert m[0].all() and m[1].tolist() == [True] * 3 + [False] * 6


def test_live_reference_splice_and_tokenizer():
    """Against the reference's tokenizer_multimodal_token as recorded by oracle/make_golden_calls.py, incl. two
    placeholders and the empty prompt."""
    from oracle.make_golden import ToyTokenizer
    from oracle.make_golden_calls import TOKENIZER_PROMPTS
    from videollama2_b200 import mm_utils
    ref = torch.load(os.path.join(GOLD, "reference_calls.pt"))["tokenizer"]
    assert [(p, t) for p, t, _ in ref] == TOKENIZER_PROMPTS
    tok = ToyTokenizer()
    for p, t, ref_ids in ref:
        assert mm_utils.tokenizer_multimodal_token(p, tok, t) == ref_ids


def test_keywords_stopping_criteria():
    from oracle.make_golden import ToyTokenizer
    from videollama2_b200.mm_utils import KeywordsStoppingCriteria
    tok = ToyTokenizer()
    kw = tok("stop now").input_ids[1:]
    sc = KeywordsStoppingCriteria(["stop now"], tok, torch.zeros(1, 3, dtype=torch.long))
    assert sc(torch.tensor([[9, 9] + kw]), None) and not sc(torch.tensor([[9, 9, 9]]), None)


def test_vision_cache_content_key():
    """The vision-feature cache key is a content checksum: equal for a copy, different after a one-element change, a
    different modality or a different shape (videollama2_arch.enable_vision_cache)."""
    from videollama2_b200.model.videollama2_arch import Videollama2MetaForCausalLM as M
    g = torch.Generator().manual_seed(5)
    x = torch.randn((4, 3, 14, 14), generator=g).to(torch.bfloat16)
    k0 = M._content_key([(x, "video")])
    assert M._content_key([(x.clone(), "video")]) == k0
    y = x.clone()
    y[3, 2, 13, 13] = y[3, 2, 13, 13] + 0.5
    assert M._content_key([(y, "video")]) != k0
    assert M._content_key([(x, "image")]) != k0
    assert M._content_key([(x.view(4, 3, 7, 28), "video")]) != k0
    z = x.clone()
    z[0], z[1] = x[1], x[0]                      # a permutation of frames keeps the plain sum, not the weighted one
    assert M._content_key([(z, "video")]) != k0
    odd = torch.arange(5, dtype=torch.uint8)      # byte count not a multiple of 8
    assert M._content_key([(odd, "video")]) == M._content_key([(odd.clone(), "video")])


def test_checkpoint_reader_handles_shards_and_bin(tmp_path):
    """`load_pretrained_model`'s checkpoint reader (model/__init__.py, reference: videollama2/model/__init__.py:165-193)
    merges sharded safetensors through the index file, reads a single safetensors file or a pytorch_model.bin, and fails
    loudly on an empty directory."""
    import json
    from safetensors.torch import save_file
    from videollama2_b200.model import _read_checkpoint
    a = {"model.layers.0.w": torch.arange(6, dtype=torch.float32).reshape(2, 3), "lm_head.weight": torch.ones(4, 2)}
    b = {"model.mm_projector.readout.0.bias": torch.full((5,), 0.5)}
    d = tmp_path / "sharded"
    d.mkdir()
    save_file(a, str(d / "model-00001-of-00002.safetensors"))
    save_file(b, str(d / "model-00002-of-00002.safetensors"))
    index = {"weight_map": {**{k: "model-00001-of-00002.safetensors" for k in a},
                            **{k: "model-00002-of-00002.safetensors" for k in b}}}
    (d / "model.safetensors.index.json").write_text(json.dumps(index))
    sd = _read_checkpoint(str(d))
    assert set(sd) == set(a) | set(b) and all(torch.equal(sd[k], {**a, **b}[k]) for k in sd)
    one = tmp_path / "single"
    one.mkdir()
    save_file(a, str(one / "model.safetensors"))
    assert set(_read_checkpoint(str(one))) == set(a)
    binp = tmp_path / "bin"
    binp.mkdir()
    torch.save(b, str(binp / "pytorch_model.bin"))
    assert torch.equal(_read_checkpoint(str(binp))["model.mm_projector.readout.0.bias"], b["model.mm_projector.readout.0.bias"])
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(FileNotFoundError):
        _read_checkpoint(str(empty))


def test_loader_rejects_unsupported_branches(tmp_path):
    from videollama2_b200.model import load_pretrained_model
    with pytest.raises(NotImplementedError):
        load_pretrained_model(str(tmp_path), load_4bit=True)
    with pytest.raises(NotImplementedError):
        load_pretrained_model(str(tmp_path), model_base="base", model_name="videollama2-lora-x")   # LoRA adapters
    (tmp_path / "config.json").write_text('{"model_type": "videollama2_mixtral"}')
    with pytest.raises(ValueError):
        load_pretrained_model(str(tmp_path))


def test_presets_flops_match_baseline():
    """The FLOP model behind every roofline fraction reproduces BASELINE.md's totals for the three 7B configs."""
    from videollama2_b200 import presets
    m = presets.make_config(presets.MISTRAL_7B, 16)
    q = presets.make_config(presets.QWEN2_7B, 16)
    assert abs(presets.flops(m, 16, 256)["total"] / 1e12 - 34.715) < 0.01
    assert abs(presets.flops(q, 16, 256)["total"] / 1e12 - 32.17) < 0.02
    assert abs(presets.flops(presets.make_config(presets.MISTRAL_7B, 8), 8, 32)["total"] / 1e12 - 17.03) < 0.02
    v21 = presets.make_config(presets.QWEN2_7B, 16, "stc_connector_v35", presets.SIGLIP_SO400M_384)
    f = presets.flops(v21, 16, 256)
    assert f["vis_tokens"] == 8 * 13 * 13 and f["S"] == 255 + 1352
    names = {n for n, _, _ in presets.state_dict_specs(v21)}
    assert "model.vision_tower.vision_tower.vision_model.embeddings.patch_embedding.bias" in names
    assert not any("class_embedding" in n for n in names)


def _my_mm_infer_call(case):
    import videollama2_b200
    from oracle.mm_infer_ref import RecordingModel, ToyChatTokenizer, summarise
    model, tok = RecordingModel(case["model_type"]), ToyChatTokenizer()
    frames = None if case["modal"] == "text" else torch.zeros((2, 3, 4, 4))
    text = videollama2_b200.mm_infer(frames, case["instruct"], model, tok, modal=case["modal"], **case["kwargs"])
    return text, summarise(model.calls[0]), model.calls[0]


def test_mm_infer_matches_reference_goldens():
    """videollama2_b200.mm_infer builds the same prompt ids / mask and hands generate() the same arguments as the
    reference's mm_infer run with the same toy tokenizer (tests/golden/mm_infer.pt, oracle/mm_infer_ref.py)."""
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mm_infer.pt"))
    for case in gold:
        text, mine, raw = _my_mm_infer_call(case)
        want = case["call"]
        assert text == case["text"]
        assert torch.equal(mine["input_ids"], want["input_ids"]) and torch.equal(mine["attention_mask"], want["attention_mask"])
        for k in ("images_modal", "n_stopping", "do_sample", "temperature", "max_new_tokens", "top_p", "use_cache", "pad_token_id"):
            assert mine[k] == want[k], (k, mine[k], want[k])
        if raw["images"] is not None:
            assert raw["images"][0][0].dtype == torch.bfloat16          # the engine's dtype (reference: .half())


def test_mm_infer_matches_live_reference():
    """The reference's mm_infer on its first case, as recorded by oracle/make_golden_calls.py."""
    from oracle import mm_infer_ref
    ref = torch.load(os.path.join(GOLD, "reference_calls.pt"))["mm_infer"]
    instruct, modal, mtype, kw = mm_infer_ref.CASES[ref["case"]]
    case = {"instruct": instruct, "modal": modal, "model_type": mtype, "kwargs": kw}
    my_text, mine, _ = _my_mm_infer_call(case)
    assert my_text == ref["text"] and torch.equal(mine["input_ids"], ref["input_ids"])
    import videollama2_b200
    with pytest.raises(ValueError):
        videollama2_b200.mm_infer(None, "x", mm_infer_ref.RecordingModel("videollama2"), mm_infer_ref.ToyChatTokenizer(), modal="audio")
    assert videollama2_b200.get_model_name_from_path("/ckpt/run1/checkpoint-500/") == "run1_checkpoint-500"


def test_sampling_warpers_match_hf():
    """generate(do_sample=True) filters the logits exactly like HF's temperature / top-k / top-p warpers (the arguments
    the reference's mm_infer passes, with GenerationConfig's default top_k = 50)."""
    lp = pytest.importorskip("transformers.generation.logits_process")
    from videollama2_b200.sampling import sample_token, warp_logits
    g = torch.Generator().manual_seed(3)
    logits = torch.randn((4, 300), generator=g) * 3
    ids = torch.zeros((4, 1), dtype=torch.long)
    for temp, k, p in [(0.2, 50, 0.9), (1.0, 50, 0.5), (0.7, 0, 0.95), (1.3, 10, 1.0), (0.2, 50, 0.01)]:
        ref = lp.TemperatureLogitsWarper(temp)(ids, logits.clone()) if temp != 1.0 else logits.clone()
        if k > 0:
            ref = lp.TopKLogitsWarper(top_k=k)(ids, ref)
        if p < 1.0:
            ref = lp.TopPLogitsWarper(top_p=p)(ids, ref)
        mine = warp_logits(logits, temp, k, p)
        assert torch.equal(torch.isinf(mine), torch.isinf(ref)), (temp, k, p)
        keep = ~torch.isinf(ref)
        assert torch.allclose(mine[keep], ref[keep], rtol=1e-6, atol=1e-6)
    assert sample_token(logits[0], 0.2, 0.9, top_k=1) == int(logits[0].argmax())          # top_k = 1 is greedy
    a = sample_token(logits[1], 1.0, 0.9, generator=torch.Generator().manual_seed(5))
    b = sample_token(logits[1], 1.0, 0.9, generator=torch.Generator().manual_seed(5))
    assert a == b
    with pytest.raises(ValueError):
        warp_logits(logits, temperature=-1.0)


def test_synthetic_checkpoint_matches_oracle_factory():
    """presets.synth_tensor / state_dict_specs (what bench.py and the full-depth GPU tests load into the engine) are
    byte-identical to oracle.synth (what the committed goldens were computed with)."""
    import torch
    from oracle import synth
    from videollama2_b200 import presets
    for name, llm in (("cfg2", presets.MISTRAL_7B), ("cfg3", presets.QWEN2_7B)):
        ocfg = synth.CONFIGS[name]
        ours = presets.state_dict_specs(presets.make_config(llm, ocfg.frames))
        theirs = synth.model_specs(ocfg)
        assert [(n, tuple(s), k) for n, s, k in ours] == [(n, tuple(s), k) for n, s, k in theirs]
    picks = [("model.layers.3.self_attn.q_proj.weight", (64, 48), "w"), ("model.norm.weight", (96,), "gain"),
             ("model.layers.0.self_attn.k_proj.bias", (40,), "bias"), ("model.embed_tokens.weight", (50, 32), "emb"),
             ("model.mm_projector.sampler.0.weight", (8, 8, 2, 2, 2), "w")]
    for name, shape, kind in picks:
        assert torch.equal(presets.synth_tensor(name, shape, kind), synth.make_tensor(name, shape, kind))
    cfg = presets.make_config(presets.MISTRAL_7B, 16)
    px, ids = presets.synthetic_inputs(cfg, 16, 256)
    opx, oids = synth.inputs(synth.CONFIGS["cfg2"])
    assert torch.equal(px, opx) and torch.equal(ids, oids)


def test_vision_config_family_defaults_and_hub_ids():
    """A SigLIP config.json that omits layer_norm_eps / hidden_act must get SigLIP's defaults (1e-6, gelu-tanh), not
    CLIP's; hub ids of the two supported towers resolve without a local directory."""
    from videollama2_b200.model.config import VisionConfig
    s = VisionConfig.from_dict({"model_type": "siglip_vision_model", "hidden_size": 1152, "num_attention_heads": 16})
    assert s.layer_norm_eps == 1e-6 and s.hidden_act == "gelu_pytorch_tanh"
    c = VisionConfig.from_dict({"vision_config": {"model_type": "clip_vision_model", "hidden_size": 1024}})
    assert c.layer_norm_eps == 1e-5 and c.hidden_act == "quick_gelu"
    so = VisionConfig.from_dir("google/siglip-so400m-patch14-384")
    assert (so.hidden_size, so.intermediate_size, so.num_hidden_layers, so.image_size, so.layer_norm_eps) == (1152, 4304, 27, 384, 1e-6)
    cl = VisionConfig.from_dir("openai/clip-vit-large-patch14-336")
    assert (cl.hidden_size, cl.num_hidden_layers, cl.image_size, cl.layer_norm_eps, cl.hidden_act) == (1024, 24, 336, 1e-5, "quick_gelu")
    with pytest.raises(FileNotFoundError):
        VisionConfig.from_dir("some/unknown-tower")


def test_assemble_state_dict_base_plus_projector(tmp_path):
    """model/__init__.py:138-164: LLM from model_base, mm_projector.bin from model_path, tower from its local directory."""
    import torch
    from safetensors.torch import save_file
    from videollama2_b200.model import assemble_state_dict
    base, path, tower = tmp_path / "base", tmp_path / "ckpt", tmp_path / "clip-tower"
    for d in (base, path, tower):
        d.mkdir()
    llm = {"model.embed_tokens.weight": torch.randn(8, 4), "lm_head.weight": torch.randn(8, 4)}
    save_file(llm, str(base / "model.safetensors"))
    proj = {"model.mm_projector.readout.0.weight": torch.randn(4, 4), "model.mm_projector.readout.0.bias": torch.randn(4)}
    torch.save(proj, str(path / "mm_projector.bin"))
    tw = {"vision_model.embeddings.class_embedding": torch.randn(4), "text_model.ignored": torch.randn(2)}
    save_file(tw, str(tower / "model.safetensors"))
    cfg = type("C", (), {"mm_vision_tower": str(tower)})()
    sd = assemble_state_dict(str(path), str(base), cfg)
    assert torch.equal(sd["lm_head.weight"], llm["lm_head.weight"])
    assert torch.equal(sd["model.mm_projector.readout.0.weight"], proj["model.mm_projector.readout.0.weight"].to(torch.float16))
    assert torch.equal(sd["model.vision_tower.vision_tower.vision_model.embeddings.class_embedding"],
                       tw["vision_model.embeddings.class_embedding"])
    assert not any("text_model" in k for k in sd)
    cfg.mm_vision_tower = "openai/clip-vit-large-patch14-336"
    with pytest.raises(FileNotFoundError):
        assemble_state_dict(str(path), str(base), cfg)
    # SFT branch: everything from model_path
    save_file({**llm, **{k: v for k, v in proj.items()}}, str(path / "model.safetensors"))
    assert set(assemble_state_dict(str(path))) == set(llm) | set(proj)


def test_keywords_stopping_criteria_decoded_text_branch_matches_reference():
    """mm_utils.py:332-337: the keyword may be spelled by different ids than tokenizer(keyword) produced; the decoded tail
    (window = longest keyword, in ids) is searched too.  Compared call by call with the reference class's answers
    recorded by oracle/make_golden_calls.py."""
    from oracle.make_golden_calls import DecodingToyTokenizer, keyword_cases
    from videollama2_b200.mm_utils import KeywordsStoppingCriteria
    tok = DecodingToyTokenizer()
    prompt = torch.zeros(1, 2, dtype=torch.long)
    ours = KeywordsStoppingCriteria(["hello"], tok, prompt)
    kw = tok("hello", add_special_tokens=False).input_ids             # ["he", "llo"]
    bang = tok("hello!", add_special_tokens=False).input_ids          # one id spelling "hello!"
    assert len(kw) == 2 and len(bang) == 1
    got = [ours(c, None) for c in keyword_cases(tok)]
    assert got[0] is True and got[2] is False and got[6] is False and got[7] is True
    assert got[1] is True          # id tail differs from tokenizer("hello"), the decoded window contains it
    assert got == torch.load(os.path.join(GOLD, "reference_calls.pt"))["keywords_hello"]
