"""fp8 (E4M3) decode weights, decode_weights="fp8": every decoder linear weight and lm_head streams as fp8 with one fp32
scale per output row (vl2_gemv_fp8) during KV-cache decode; prefill keeps the 16-bit weights.

The synthetic weights are untrained, so the distance between fp8 and bf16 decode says nothing about a real checkpoint.
The correctness bar is therefore equivalence with the DEQUANTISED model: a torch fp32 restatement of one decode step that
reads the engine's own KV cache and uses W8 * scale.  That restatement is first checked against the bf16 engine with the
bf16 weights at the same bar."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import engine_config, rel

FP8 = torch.float8_e4m3fn


# ---- CPU ---------------------------------------------------------------------------------------------------------
def _e4m3_table():
    """Every finite E4M3 code (0x00..0x7E and 0x80..0xFE) and its value, decoded from the bit fields."""
    codes = np.array([c for c in range(256) if (c & 0x7F) != 0x7F], dtype=np.int64)
    s, e, m = codes >> 7, (codes >> 3) & 0xF, codes & 7
    mag = np.where(e == 0, m / 8.0 * 2.0 ** -6, (1 + m / 8.0) * 2.0 ** (e - 7.0))
    return codes, np.where(s == 1, -mag, mag)


def _rows():
    g = torch.Generator().manual_seed(5)
    w = torch.randn((24, 160), generator=g) * torch.logspace(-6, 3, 24)[:, None]
    w[3] = 0.0                                              # an all-zero row
    w[7, :] = 0.0
    w[7, 11] = -2.5e-4                                      # one non-zero element: the row max is negative
    w[9] = torch.randn(160, generator=g) * 1e-3 * (torch.rand(160, generator=g) < 0.1)   # mostly zeros
    return w


def test_quantize_fp8_rows_bounds_and_codes():
    from videollama2_b200 import ops
    w = _rows()
    w8, scale = ops.quantize_fp8_rows(w)
    assert w8.dtype == FP8 and w8.shape == w.shape and scale.dtype == torch.float32 and scale.shape == (w.shape[0],)
    codes = w8.view(torch.uint8).to(torch.int64)
    assert not bool(((codes & 0x7F) == 0x7F).any())                               # no NaN code
    q = w8.float()
    zero = w.abs().amax(1) == 0
    assert bool((scale[zero] == 1).all()) and bool((q[zero] == 0).all())          # zero rows: scale 1, all zeros
    amax_i = w.abs().argmax(1)
    r = torch.arange(w.shape[0])
    peak = q[r, amax_i]
    assert bool((peak[~zero].abs() == 448).all())                                # each row's max maps to +-448 ...
    assert bool((torch.sign(peak[~zero]) == torch.sign(w[r, amax_i][~zero])).all())   # ... with its sign
    # within half an E4M3 step of the input (step at |y|: 2^(floor(log2|y|) - 3), 2^-9 in the subnormal range)
    y = w / scale[:, None]
    ay = y.abs().clamp(min=2.0 ** -6)
    step = torch.exp2(torch.floor(torch.log2(ay)) - 3)
    assert bool(((q - y).abs() <= step / 2 * (1 + 1e-6)).all())
    assert bool(((q * scale[:, None] - w).abs() <= step / 2 * scale[:, None] * (1 + 1e-5)).all())


def test_quantize_fp8_rows_is_round_to_nearest_even():
    """The codes are the nearest E4M3 value of w / scale, ties to the even code, from a table of all 254 finite codes."""
    from videollama2_b200 import ops
    w = _rows()
    w8, scale = ops.quantize_fp8_rows(w)
    codes, vals = _e4m3_table()
    order = np.argsort(vals, kind="stable")
    codes, vals = codes[order], vals[order]
    y = (w.double() / scale.double()[:, None]).clamp(-448, 448).float().double().numpy().reshape(-1)
    hi = np.clip(np.searchsorted(vals, y), 1, len(vals) - 1)
    lo = hi - 1
    dlo, dhi = np.abs(y - vals[lo]), np.abs(vals[hi] - y)
    pick = np.where(dlo < dhi, lo, np.where(dhi < dlo, hi, np.where(codes[lo] % 2 == 0, lo, hi)))
    want = vals[pick]
    got = w8.float().double().numpy().reshape(-1)
    assert np.array_equal(got, want)
    # the same as torch's own round-to-nearest-even cast of the clamped, scaled rows
    ref = (w.float() / scale[:, None]).clamp(-448, 448).to(FP8)
    assert torch.equal(w8.view(torch.uint8), ref.view(torch.uint8))


@pytest.fixture(scope="module")
def lib():
    from videollama2_b200 import _lib, build
    build.build()
    return _lib.load()


def test_gemv_fp8_argument_validation_without_gpu(lib):
    """Shape and scale checks run before any CUDA call."""
    vp = ctypes.c_void_p
    scale = vp(16)
    assert lib.vl2_gemv_fp8(vp(16), vp(16), scale, None, None, vp(16), 0, 8, 24, 0, 0.0, None) == -1   # K % 16 != 0
    assert b"K % 16" in lib.vl2_last_error()
    assert lib.vl2_gemv_fp8(vp(16), vp(16), None, None, None, vp(16), 0, 8, 32, 0, 0.0, None) == -1    # no w_scale
    assert b"w_scale" in lib.vl2_last_error()
    assert lib.vl2_gemv_fp8(vp(17), vp(16), scale, None, None, vp(16), 0, 8, 32, 0, 0.0, None) == -3   # misaligned x
    assert lib.vl2_gemv_fp8(vp(16), vp(16), scale, None, None, vp(16), 0, 7, 32, 4, 0.0, None) == -6   # SwiGLU, odd N


def test_ops_gemv_fp8_needs_scale():
    from videollama2_b200 import ops
    x = torch.zeros((1, 32), dtype=torch.bfloat16)
    w8 = torch.zeros((8, 32), dtype=FP8)
    with pytest.raises(ValueError):
        ops.gemv(x, w8)
    with pytest.raises(ValueError):
        ops.gemv(x, torch.zeros((8, 32), dtype=torch.bfloat16), w_scale=torch.ones(8))


def test_bad_decode_weights_value_is_refused():
    from oracle import synth
    from videollama2_b200.model import VLLMs, load_pretrained_model
    from videollama2_b200.model.decoder import DecoderEngine
    from videollama2_b200.model.videollama2_arch import Videollama2MetaModel
    ec = engine_config(synth.CONFIGS["tiny"])
    for bad in ("fp16", "int8", "FP8", None):
        with pytest.raises(ValueError):
            VLLMs[ec.model_type].from_state_dict(ec, {}, device="cpu", decode_weights=bad)
        with pytest.raises(ValueError):
            DecoderEngine(ec, decode_weights=bad)
    with pytest.raises(ValueError):
        load_pretrained_model("/nonexistent-checkpoint", decode_weights="e5m2")
    with pytest.raises(NotImplementedError):                 # fp8 decode with a tensor-parallel decoder
        Videollama2MetaModel(ec, tp_group=True, decode_weights="fp8")
    assert DecoderEngine(ec).decode_weights == "bf16"


# ---- GPU: the kernel ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fp8_weights(cuda):
    """fp8 test weights per (N, K, seed), shared by the modes and library builds of one shape (< 1 GB for all shapes) and
    released when this module's tests are done."""
    from videollama2_b200 import ops
    cache = {}

    def get(N, K, seed):
        if (N, K, seed) not in cache:
            g = torch.Generator(device=cuda).manual_seed(seed)
            w = torch.randn((N, K), generator=g, device=cuda) * K ** -0.5
            w *= torch.exp(torch.randn((N, 1), generator=g, device=cuda))          # rows of varied size
            w[min(3, N - 1)] = 0.0
            cache[N, K, seed] = ops.quantize_fp8_rows(w)
        return cache[N, K, seed]
    yield get
    cache.clear()
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
@pytest.mark.parametrize("N,K", [(4096, 4096), (1000, 336), (28672, 4096), (4096, 14336), (37, 16), (152064, 3584),
                                 (37888, 3584), (3584, 18944)])
@pytest.mark.parametrize("mode", ["plain", "rms_bias", "swiglu_rms", "residual", "f32out"])
def test_gemv_fp8(cuda, fp8_weights, dtype, N, K, mode):
    """fp8 GEMV against x . (W8 * scale)^T in fp32, with the epilogues of test_gemv, in both library builds."""
    from videollama2_b200 import ops
    if mode == "swiglu_rms" and N % 2:
        pytest.skip("SwiGLU needs even N")
    g = torch.Generator().manual_seed(91)
    x = (torch.randn((1, K), generator=g) * 1.5).to(dtype).to(cuda)
    w8, sc = fp8_weights(N, K, 92)
    xf, wf = x.float(), w8.float() * sc[:, None]
    eps = 1e-5
    s = torch.rsqrt((xf * xf).mean() + eps)
    if mode == "plain":
        out, ref = ops.gemv(x, w8, w_scale=sc), xf @ wf.t()
    elif mode == "rms_bias":
        b = (torch.randn((N,), generator=g) * 0.1).to(cuda)
        out, ref = ops.gemv(x, w8, w_scale=sc, bias=b, rms_eps=eps), s * (xf @ wf.t()) + b
    elif mode == "swiglu_rms":
        out = ops.gemv(x, w8, w_scale=sc, act=ops.ACT_SWIGLU, rms_eps=eps)
        y = s * (xf @ wf.t())
        ref = torch.nn.functional.silu(y[:, 0::2]) * y[:, 1::2]
    elif mode == "residual":
        r = torch.randn((1, N), generator=g).to(dtype).to(cuda)
        out, ref = ops.gemv(x, w8, w_scale=sc, residual=r), xf @ wf.t() + r.float()
    else:
        out, ref = ops.gemv(x, w8, w_scale=sc, out_dtype=torch.float32), xf @ wf.t()
        assert out.dtype == torch.float32
    assert out.shape == ref.shape and out.dtype == (torch.float32 if mode == "f32out" else dtype)
    assert rel(out, ref) < (2e-5 if mode == "f32out" else 4e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,act,rms", [(6144, 4096, 0, 1e-5), (28672, 4096, 4, 1e-5), (4096, 14336, 0, 0.0)])
def test_gemv_fp8_deterministic_and_graph_capturable(cuda, fp8_weights, N, K, act, rms):
    from videollama2_b200 import ops
    x = torch.randn((1, K), generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).to(cuda)
    w8, sc = fp8_weights(N, K, 4)
    outs = [ops.gemv(x, w8, w_scale=sc, act=act, rms_eps=rms, out_dtype=torch.float32) for _ in range(3)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    buf = torch.empty_like(outs[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.gemv(x, w8, w_scale=sc, act=act, rms_eps=rms, out=buf)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.gemv(x, w8, w_scale=sc, act=act, rms_eps=rms, out=buf)
    buf.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(buf, outs[0])


# ---- GPU: the decoder ---------------------------------------------------------------------------------------------
def _build(cfg, sd, cuda, **kw):
    from videollama2_b200.model import VLLMs
    ec = engine_config(cfg)
    return VLLMs[ec.model_type].from_state_dict(ec, sd, device=cuda, **kw)


def _embeds(model, px, ids, cuda):
    mask = torch.ones_like(ids, dtype=torch.bool)
    return model.prepare_inputs_labels_for_multimodal(ids, mask, None, None, [(px.to(cuda), "video")])[3][0]


def _decode_weights_f32(dec):
    """The weights the engine's decode streams, as fp32 (dequantised W8 * scale for fp8)."""
    layers, head = dec._decode_set()

    def f(d, k):
        return d[k].float() * d[k + "_s"][:, None] if k + "_s" in d else d[k].float()
    return ([{k: f(L, k) for k in ("wqkv", "wo", "wgu", "wd")} | ({"bqkv": L["bqkv"]} if "bqkv" in L else {})
             for L in layers], f(head, "lm_head"))


def _oracle_step(dec, Wl, Wh, x, pos):
    """fp32 restatement of one decode step at position `pos` on the engine's cache rows [0, pos): the q/k rows are in the
    engine's layout (RoPE partners (i, i + D/2) are adjacent columns (2i, 2i+1)), so RoPE rotates adjacent pairs."""
    Hq, Hkv, D, eps = dec.Hq, dec.Hkv, dec.D, dec.eps
    x = x.float().reshape(1, -1)
    inv = dec.w["inv_freq"].float()
    ang = float(pos) * inv
    cos, sin = torch.cos(ang), torch.sin(ang)

    def rms(t):
        return torch.rsqrt((t * t).mean() + eps)

    def rope(t, heads):
        t = t.view(heads, D // 2, 2)
        a, b = t[..., 0], t[..., 1]
        return torch.stack([a * cos - b * sin, b * cos + a * sin], -1).reshape(heads, D)

    for i, W in enumerate(Wl):
        qkv = rms(x) * (x @ W["wqkv"].t())[0]
        if "bqkv" in W:
            qkv = qkv + W["bqkv"]
        q = rope(qkv[: Hq * D], Hq)
        k_new = rope(qkv[Hq * D: (Hq + Hkv) * D], Hkv)
        v_new = qkv[(Hq + Hkv) * D:].view(Hkv, D)
        cache = dec.kv[i][:pos].float()
        K = torch.cat([cache[:, Hq * D: (Hq + Hkv) * D].view(pos, Hkv, D), k_new[None]], 0)
        V = torch.cat([cache[:, (Hq + Hkv) * D:].view(pos, Hkv, D), v_new[None]], 0)
        grp = Hq // Hkv
        K, V = K.repeat_interleave(grp, 1), V.repeat_interleave(grp, 1)            # [pos+1, Hq, D]
        p = torch.softmax(torch.einsum("hd,shd->hs", q, K) * D ** -0.5, -1)
        o = torch.einsum("hs,shd->hd", p, V).reshape(1, Hq * D)
        x = x + o @ W["wo"].t()
        gu = rms(x) * (x @ W["wgu"].t())
        x = x + (torch.nn.functional.silu(gu[:, 0::2]) * gu[:, 1::2]) @ W["wd"].t()
    return rms(x) * (x @ Wh.t())


DEC_CFGS = ["tiny", "tiny_qwen2", "mid"]
TEACHER = [5, 17, 3, 42, 9, 28, 11, 30]          # teacher-forced token ids (below every test vocabulary)
BAR = 1.5e-2                                     # test_kv_cache_decode_matches_recompute's bar against the fp32 oracle


@pytest.fixture(scope="module", params=DEC_CFGS)
def pair(request, cuda):
    from oracle import synth
    cfg = synth.CONFIGS[request.param]
    sd = synth.state_dict(cfg)
    px, ids = synth.inputs(cfg)
    return cfg, sd, px, ids, _build(cfg, sd, cuda), _build(cfg, sd, cuda, decode_weights="fp8")


def _teacher_forced(model, emb, cuda, steps=len(TEACHER)):
    """Prefill with the cache, then `steps` teacher-forced decode steps; per step (engine logits, oracle logits)."""
    dec = model.get_model().decoder
    dec.prefill(emb, all_logits=False, keep_cache=True, max_len=emb.shape[0] + steps + 1)
    Wl, Wh = _decode_weights_f32(dec)
    res = []
    for tok in TEACHER[:steps]:
        e = model.get_model().embed_tokens(torch.tensor([tok]))
        pos = dec.kv_len
        ref = _oracle_step(dec, Wl, Wh, e, pos)
        res.append((dec.decode_step(e).clone(), ref))
    return res


@pytest.mark.gpu
def test_fp8_decode_matches_dequantised_model(pair, cuda):
    cfg, sd, px, ids, m16, m8 = pair
    assert not m16.get_model().decoder.layers8 and m8.get_model().decoder.layers8
    emb = _embeds(m16, px, ids, cuda)
    bf16 = _teacher_forced(m16, emb, cuda)
    for got, ref in bf16:                                       # the restatement itself, on the bf16 engine
        assert rel(got, ref) < BAR
    dist = []
    for (got, ref), (g16, _) in zip(_teacher_forced(m8, emb, cuda), bf16):
        assert torch.isfinite(got).all() and rel(got, ref) < BAR
        dist.append(rel(got, g16))
    print(f"{cfg.name}: fp8-vs-bf16 decode logits relL2 per step {[round(d, 4) for d in dist]}")


@pytest.mark.gpu
def test_fp8_decode_leaves_prefill_unchanged(pair, cuda):
    cfg, sd, px, ids, m16, m8 = pair
    imgs = [(px.to(cuda), "video")]
    mask = torch.ones_like(ids)
    a, b = m16(input_ids=ids, attention_mask=mask, images=imgs), m8(input_ids=ids, attention_mask=mask, images=imgs)
    assert torch.equal(a.logits, b.logits)
    emb = _embeds(m16, px, ids, cuda)
    la, _ = m16.get_model().decoder.prefill(emb, all_logits=False)
    lb, _ = m8.get_model().decoder.prefill(emb, all_logits=False)
    assert torch.equal(la, lb)
    t16 = m16.generate(ids, images=imgs, max_new_tokens=1, do_sample=False)
    assert torch.equal(m8.generate(ids, images=imgs, max_new_tokens=1, do_sample=False), t16)


@pytest.mark.gpu
def test_fp8_graph_decode_with_l2_prefetch_fork(pair, cuda):
    """The fp8 decode graph with the forked weight-prefetch branch (vl2_l2_prefetch of the fp8 o_proj / gate-up weights
    next to the attention phase) gives the eager fp8 tokens; the budget spans all of o_proj and part of gate-up."""
    cfg, sd, px, ids, m16, m8 = pair
    imgs = [(px.to(cuda), "video")]
    dec = m8.get_model().decoder
    assert dec.layers8[0]["wo"].dtype == torch.float8_e4m3fn
    eager = m8.generate(ids, images=imgs, max_new_tokens=6, do_sample=False, eos_token_id=None)
    old = dec.decode_prefetch_mb
    dec.decode_prefetch_mb = (dec.layers8[0]["wo"].numel() + 4096) / 1e6
    m8.enable_cuda_graphs(True)
    try:
        for _ in range(2):
            assert torch.equal(m8.generate(ids, images=imgs, max_new_tokens=6, do_sample=False, eos_token_id=None), eager)
    finally:
        m8.enable_cuda_graphs(False)
        dec.decode_prefetch_mb = old


@pytest.mark.gpu
def test_fp8_graph_replay_and_sampling(pair, cuda):
    """Graph-replayed (chunked) greedy fp8 decode reproduces eager fp8 decode bit for bit, tokens and logits; sampling
    with a fixed generator gives the same tokens eagerly and graphed; forward(past_key_values=...) and batch rows follow
    the same fp8 weights."""
    cfg, sd, px, ids, m16, m8 = pair
    imgs = [(px.to(cuda), "video")]
    dec = m8.get_model().decoder
    eager = m8.generate(ids, images=imgs, max_new_tokens=7, do_sample=False, eos_token_id=None)
    emb = _embeds(m8, px, ids, cuda)
    l0, _ = dec.prefill(emb, all_logits=False, keep_cache=True, max_len=emb.shape[0] + 4)
    t0 = int(l0[0].argmax())
    eager_logits = dec.decode_step(m8.get_model().embed_tokens(torch.tensor([t0]))).clone()
    kw = dict(max_new_tokens=6, do_sample=True, temperature=1.5, top_p=0.95, eos_token_id=None)
    s_eager = m8.generate(ids, images=imgs, generator=torch.Generator(device=cuda).manual_seed(9), **kw)
    m8.enable_cuda_graphs(True)
    try:
        for chunk in (8, 3):
            assert torch.equal(m8.generate(ids, images=imgs, max_new_tokens=7, do_sample=False, eos_token_id=None,
                                           decode_chunk=chunk), eager)
        dec.prefill(emb, all_logits=False, keep_cache=True, max_len=emb.shape[0] + 4)
        dec.decode_graph_begin(t0)
        dec.decode_graph_step()
        assert torch.equal(dec.decode_graph_logits, eager_logits)
        s_graph = m8.generate(ids, images=imgs, generator=torch.Generator(device=cuda).manual_seed(9), **kw)
    finally:
        m8.enable_cuda_graphs(False)
    assert torch.equal(s_graph, s_eager)
    # forward(past_key_values=...) one token at a time
    out = m8(input_ids=ids, attention_mask=torch.ones_like(ids), images=imgs, use_cache=True)
    toks, pkv = [int(out.logits[0, -1].argmax())], out.past_key_values
    for _ in range(3):
        step = m8(input_ids=torch.tensor([[toks[-1]]]), past_key_values=pkv)
        toks.append(int(step.logits[0, -1].argmax()))
        pkv = step.past_key_values
    assert toks == eager[0, :4].tolist()
    # a batch of two identical rows decodes each row like the batch-1 call
    both = m8.generate(torch.cat([ids, ids]), images=imgs + imgs, attention_mask=torch.ones((2, ids.shape[1]), dtype=torch.bool),
                       max_new_tokens=7, do_sample=False, eos_token_id=None, pad_token_id=0)
    assert torch.equal(both[0], eager[0]) and torch.equal(both[1], eager[0])


@pytest.mark.gpu
def test_fp8_decode_fp16_build(cuda):
    """dtype=torch.float16 with decode_weights="fp8": the fp16 library's fp8 GEMV against the dequantised model."""
    from oracle import synth
    cfg = synth.CONFIGS["tiny"]
    sd = synth.state_dict(cfg)
    px, ids = synth.inputs(cfg)
    m16 = _build(cfg, sd, cuda, dtype=torch.float16)
    m8 = _build(cfg, sd, cuda, dtype=torch.float16, decode_weights="fp8")
    assert m8.get_model().decoder.dtype == torch.float16
    emb = _embeds(m16, px, ids, cuda)
    for got, ref in _teacher_forced(m16, emb, cuda):
        assert rel(got, ref) < BAR
    for got, ref in _teacher_forced(m8, emb, cuda):
        assert torch.isfinite(got).all() and rel(got, ref) < BAR


@pytest.mark.gpu
def test_fp8_decode_mistral7b_full_size(cuda):
    """Mistral-7B synthetic model: 32 fp8 tokens without NaN, and teacher-forced fp8-vs-bf16 logits within a sanity bar
    (a broken kernel gives relL2 >= 1; per-row E4M3 on these untrained weights gives ~0.1 at 4-8 layers)."""
    from videollama2_b200 import presets
    from videollama2_b200.model import VLLMs
    cfg = presets.make_config(presets.MISTRAL_7B, 16)
    sd = presets.synthetic_state_dict(cfg, cuda)
    m16 = VLLMs[cfg.model_type].from_state_dict(cfg, sd, device=cuda)
    m8 = VLLMs[cfg.model_type].from_state_dict(cfg, sd, device=cuda, decode_weights="fp8")
    del sd
    torch.cuda.empty_cache()
    ids = torch.randint(3, 32000, (1, 512), generator=torch.Generator().manual_seed(1))
    new8 = m8.generate(ids, max_new_tokens=32, do_sample=False, eos_token_id=None)
    assert new8.shape == (1, 32)
    new16 = m16.generate(ids, max_new_tokens=32, do_sample=False, eos_token_id=None)
    d16, d8 = m16.get_model().decoder, m8.get_model().decoder
    emb = m16.get_model().embed_tokens(ids)[0]
    l16, _ = d16.prefill(emb, all_logits=False, keep_cache=True, max_len=emb.shape[0] + 33)
    l8, _ = d8.prefill(emb, all_logits=False, keep_cache=True, max_len=emb.shape[0] + 33)
    assert torch.equal(l16, l8)
    dist = []
    for tok in new16[0].tolist():                          # teacher-forced with the bf16 model's greedy tokens
        e = m16.get_model().embed_tokens(torch.tensor([tok]))
        a, b = d16.decode_step(e), d8.decode_step(e)
        assert torch.isfinite(b).all()
        dist.append(rel(b, a))
    agree = sum(int(x == y) for x, y in zip(new8[0].tolist(), new16[0].tolist()))
    print(f"Mistral-7B synthetic, 32 layers: fp8-vs-bf16 teacher-forced logits relL2 mean {sum(dist) / len(dist):.4f} "
          f"max {max(dist):.4f}; greedy tokens equal at {agree}/32 positions")
    assert max(dist) < 0.25
