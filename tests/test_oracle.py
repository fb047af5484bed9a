"""The CPU oracle (oracle/torch_ref.py) is pinned against (a) the committed golden fixtures produced by the REAL
reference classes (oracle/make_golden.py) and (b) the reference model's own outputs recorded by
oracle/make_golden_calls.py.  fp32 restatement vs fp32 reference: round-off only (<= 1e-5 relL2)."""
import os

import pytest
import torch

from helpers import rel

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = ["tiny", "tiny_qwen2", "tiny_v35", "tiny_siglip"]


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_reference_goldens(name):
    from oracle import synth, torch_ref
    gold = torch.load(os.path.join(GOLD, f"{name}.pt"))
    cfg = synth.CONFIGS[name]
    sd = synth.state_dict(cfg)
    px, ids = synth.inputs(cfg)
    mine = torch_ref.full_forward(sd, cfg, px, ids, torch.float32)
    g = gold["g32"]
    # fp32 on both sides; the bar leaves room for thread-count-dependent summation orders (a few 1e-6 here), nothing more
    assert mine["vit"].shape == g["vit"].shape and rel(mine["vit"], g["vit"]) < 3e-5
    assert mine["mm"].shape == g["mm"].shape == (cfg.vis_tokens, cfg.llm.hidden) and rel(mine["mm"], g["mm"]) < 3e-5
    assert mine["logits"].shape == (cfg.seq, cfg.llm.vocab) and rel(mine["logits"], g["logits"]) < 3e-5
    # the reference's greedy continuation starts with the argmax of the last prefill position
    assert int(mine["logits"][-1].argmax()) == int(gold["generate_greedy"][0, 0])
    # the bf16 run of the reference differs from its own fp32 run by the noise floor the GPU tests allow for
    h = gold["hbf16"]
    assert 1e-3 < rel(h["logits"], g["logits"]) < 5e-2


@pytest.mark.parametrize("name", NAMES)
def test_oracle_bf16_matches_reference_bf16(name):
    """Same algorithm in bf16: agreement at the bf16 noise level (different op fusion order, same roundings mostly)."""
    from oracle import synth, torch_ref
    gold = torch.load(os.path.join(GOLD, f"{name}.pt"))
    cfg = synth.CONFIGS[name]
    mine = torch_ref.full_forward(synth.state_dict(cfg), cfg, *synth.inputs(cfg), torch.bfloat16)
    assert rel(mine["vit"], gold["hbf16"]["vit"]) < 1e-2
    assert rel(mine["logits"], gold["g32"]["logits"]) < 1.5 * rel(gold["hbf16"]["logits"], gold["g32"]["logits"])


def test_oracle_vs_live_reference():
    """The reference's fp32 model on the tiny config, as recorded in golden/reference_calls.pt
    (oracle/make_golden_calls.py): logits, the STC connector alone on a batch of two videos, state-dict names/shapes."""
    from oracle import make_golden_calls, synth, torch_ref
    ref = torch.load(os.path.join(GOLD, "reference_calls.pt"))
    cfg = synth.CONFIGS["tiny"]
    sd = synth.state_dict(cfg)
    px, ids = synth.inputs(cfg)
    stc_in = make_golden_calls.stc_input(cfg)
    mine = torch_ref.full_forward(sd, cfg, px, ids, torch.float32)
    assert mine["logits"].shape == ref["tiny_logits"].shape and rel(mine["logits"], ref["tiny_logits"]) < 1e-5
    stc = torch_ref.stc_forward(sd, stc_in, 1, 4, torch.float32)      # batch of 2 videos
    assert stc.shape == ref["stc_out"].shape and rel(stc, ref["stc_out"]) < 1e-5
    # state-dict contract: names and shapes of the synthetic weights are exactly the reference model's
    mine_names = {n: tuple(s) for n, s, _ in synth.model_specs(cfg)}
    assert ref["state_dict_shapes"] == mine_names


def test_flop_model_matches_baseline_md():
    from videollama2_b200 import presets as P
    f2 = P.flops(P.make_config(P.MISTRAL_7B, 16), 16, 256)
    assert f2["S"] == 1776 and f2["vis_tokens"] == 1521
    assert abs(f2["total"] / 1e12 - 34.72) < 0.01 and abs(f2["vit"] / 1e12 - 5.86) < 0.01
    assert abs(f2["stc"] / 1e12 - 3.24) < 0.01 and abs(f2["llm"] / 1e12 - 25.62) < 0.01
    assert abs(P.flops(P.make_config(P.MISTRAL_7B, 8), 8, 32)["total"] / 1e12 - 17.03) < 0.01
    assert abs(P.flops(P.make_config(P.QWEN2_7B, 16), 16, 256)["total"] / 1e12 - 32.17) < 0.01


def test_preset_state_dict_names_match_oracle_contract():
    from oracle import synth
    from videollama2_b200 import presets as P
    from helpers import engine_config
    for name in ("tiny", "tiny_qwen2"):
        cfg = synth.CONFIGS[name]
        a = {n: tuple(s) for n, s, _ in synth.model_specs(cfg)}
        b = {n: tuple(s) for n, s, _ in P.state_dict_specs(engine_config(cfg))}
        assert a == b


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3"])
def test_fulldepth_fixtures_load_and_are_consistent(name):
    """tests/golden/full_cfg*.pt (oracle/make_golden_full.py) load with torch's default safe unpickler (the GPU box has
    no way to regenerate them) and are internally consistent: rows are what make_golden_full.tap_rows yields, the
    reference's own bf16 run agrees with its fp32 run on the arg-max token, noise floors sit where BASELINE.md §4 measured
    them (1-2e-2)."""
    import os
    from oracle import make_golden_full, synth
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"full_{name}.pt")
    fx = torch.load(path, map_location="cpu")
    cfg = synth.CONFIGS[name]
    rows = make_golden_full.tap_rows(cfg)
    assert all(torch.equal(rows[k], fx["rows"][k]) for k in rows)
    assert fx["g32"]["logits_last"].shape == (cfg.llm.vocab,) and fx["g32"]["vit"].shape == (16, cfg.vision.hidden)
    assert fx["g32"]["mm"].shape == (16, cfg.llm.hidden)
    assert fx["argmax_g32"] == fx["argmax_hbf16"] == int(fx["g32"]["logits_last"].argmax())
    assert fx["top2_margin_g32"] > 2 * fx["logit_noise_absmax"]
    assert all(5e-3 < v < 3e-2 for v in fx["noise_full"].values()), fx["noise_full"]
    assert sorted(fx["dec_tap_layers"]) == sorted(set(make_golden_full.dec_tap_layers(cfg.llm.layers)))
