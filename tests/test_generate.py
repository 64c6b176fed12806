"""CPU tests of generation (quip_b200/generate.py) with the attention step injected from oracle/attn.py: ragged prompts
batched together against HF `generate` and the HF forward with a KV cache, run on each prompt alone, in fp32."""
import pytest
import torch

from oracle.attn import TorchDecodeAttention
from oracle.glue import TorchGlue
from quip_b200.generate import CudaDecodeAttention, Generator, generate, select_tokens

LENS = (3, 7, 12)
VOCAB = 199


def _model(family, arg):
    from transformers import LlamaConfig, LlamaForCausalLM, OPTConfig, OPTForCausalLM
    torch.manual_seed(0)
    if family == 'llama':
        cfg = LlamaConfig(hidden_size=128, intermediate_size=352, num_hidden_layers=2, num_attention_heads=4,
                          num_key_value_heads=arg, vocab_size=VOCAB, max_position_embeddings=64)
        return LlamaForCausalLM(cfg).float().eval()
    # word_embed_proj_dim != hidden_size exercises project_in / project_out (OPT-350m's shape)
    cfg = OPTConfig(hidden_size=64, ffn_dim=128, num_hidden_layers=2, num_attention_heads=4, vocab_size=VOCAB,
                    max_position_embeddings=64, word_embed_proj_dim=64 if arg else 48, do_layer_norm_before=arg)
    return OPTForCausalLM(cfg).float().eval()


def _prompts(seed=1):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(3, VOCAB, (n,), generator=g) for n in LENS]


MODELS = [('llama', 4, False), ('llama', 2, False), ('llama', 2, True), ('opt', True, False), ('opt', False, False)]


def _ids(c):
    return f'{c[0]}-{c[1]}' + ('-fusedglue' if c[2] else '')


@pytest.mark.parametrize('family,arg,glue', MODELS, ids=[_ids(c) for c in MODELS])
def test_greedy_generate_equals_hf_generate_on_each_prompt(family, arg, glue):
    m = _model(family, arg)
    prompts = _prompts()
    eos = m.config.eos_token_id
    with torch.no_grad():
        got = generate(m, prompts, 12, eos_token_id=eos, attn=TorchDecodeAttention(), ops=TorchGlue() if glue else None)
        for p, g in zip(prompts, got):
            want = m.generate(p[None], attention_mask=torch.ones(1, p.numel(), dtype=torch.long), max_new_tokens=12,
                              do_sample=False, eos_token_id=eos, pad_token_id=eos)[0]
            assert torch.equal(g[:want.numel()], want), (g, want)
            assert bool((g[want.numel():] == eos).all())                      # a finished row is padded with eos


@pytest.mark.parametrize('family,arg,glue', MODELS, ids=[_ids(c) for c in MODELS])
def test_step_logits_equal_hf_decode_with_kv_cache(family, arg, glue):
    """Teacher-forced: prefill of the ragged batch, then fed tokens; every row against the HF forward with a KV cache on
    that prompt alone."""
    m = _model(family, arg)
    prompts = _prompts(2)
    feed = torch.randint(3, VOCAB, (6, len(LENS)), generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        gen = Generator(m, len(LENS), 20, attn=TorchDecodeAttention(), ops=TorchGlue() if glue else None)
        got = [gen.prefill(prompts).clone()] + [gen.step(feed[i]).clone() for i in range(feed.shape[0])]
        for b, p in enumerate(prompts):
            out = m(p[None], use_cache=True)
            past, want = out.past_key_values, [out.logits[0, -1]]
            for i in range(feed.shape[0]):
                out = m(feed[i, b].view(1, 1), past_key_values=past, use_cache=True)
                past = out.past_key_values
                want.append(out.logits[0, -1])
            for i, (g, w) in enumerate(zip(got, want)):
                assert torch.allclose(g[b], w, rtol=2e-4, atol=2e-4), (b, i, float((g[b] - w).abs().max()))


def test_eos_stops_a_row_and_pads_it():
    m = _model('llama', 2)
    prompts = _prompts(4)
    with torch.no_grad():
        free = generate(m, prompts, 10, attn=TorchDecodeAttention())
        eos = int(free[0][LENS[0] + 2])                                      # the third new token of row 0
        got = generate(m, prompts, 10, eos_token_id=eos, attn=TorchDecodeAttention())
    for f, g, n in zip(free, got, LENS):
        fn, gn = f[n:].tolist(), g[n:].tolist()
        assert torch.equal(g[:n], f[:n]) and 1 <= len(gn) <= len(fn)
        cut = fn.index(eos) + 1 if eos in fn else len(fn)
        assert gn == (fn[:cut] + [eos] * len(fn))[:len(gn)], (fn, gn)
    assert len(got[0]) - LENS[0] >= 3


def test_generation_stops_early_once_every_row_has_finished():
    m = _model('llama', 4)
    prompts = _prompts(5)
    with torch.no_grad():
        free = generate(m, prompts, 4, attn=TorchDecodeAttention())
        eos = int(free[0][LENS[0]])                                          # row 0's first new token
        got = generate(m, [prompts[0]], 40, eos_token_id=eos, attn=TorchDecodeAttention(), check_every=4)
    assert got[0].numel() - LENS[0] == 4 and bool((got[0][LENS[0]:] == eos).all())


def test_overflowing_the_cache_raises():
    m = _model('opt', True)
    prompts = _prompts()
    with pytest.raises(ValueError, match='KV cache'):
        generate(m, prompts, 5, max_len=max(LENS) + 3, attn=TorchDecodeAttention())
    with torch.no_grad():
        gen = Generator(m, len(LENS), max(LENS) + 1, attn=TorchDecodeAttention())
        gen.prefill(prompts)
        gen.step()                                                            # the last free position
        with pytest.raises(ValueError, match='full'):
            gen.step()
        with pytest.raises(ValueError, match='does not fit'):
            Generator(m, len(LENS), max(LENS) - 1, attn=TorchDecodeAttention()).prefill(prompts)


def test_sampling_is_seeded_and_top_k_1_or_tiny_top_p_is_greedy():
    m = _model('llama', 2)
    prompts = _prompts(6)
    kw = dict(attn=TorchDecodeAttention())
    with torch.no_grad():
        greedy = generate(m, prompts, 8, **kw)
        a = generate(m, prompts, 8, do_sample=True, temperature=2.0, seed=11, **kw)
        b = generate(m, prompts, 8, do_sample=True, temperature=2.0, seed=11, **kw)
        c = generate(m, prompts, 8, do_sample=True, temperature=2.0, seed=12, **kw)
        k1 = generate(m, prompts, 8, do_sample=True, top_k=1, seed=3, **kw)
        p0 = generate(m, prompts, 8, do_sample=True, top_p=1e-6, seed=4, **kw)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert not all(torch.equal(x, y) for x, y in zip(a, c))
    assert all(torch.equal(x, y) for x, y in zip(k1, greedy))
    assert all(torch.equal(x, y) for x, y in zip(p0, greedy))


@pytest.mark.parametrize('temperature,top_k,top_p', [(1.0, 0, 1.0), (0.7, 0, 1.0), (1.0, 3, 1.0), (1.0, 0, 0.8)])
def test_sampled_frequencies_match_the_filtered_softmax(temperature, top_k, top_p):
    from scipy import stats
    logits = torch.tensor([2.0, 1.5, 1.0, 0.5, 0.0, -0.5, -1.0, 0.25])
    n = 40000
    g = torch.Generator().manual_seed(7)
    tok = select_tokens(logits.expand(n, -1), do_sample=True, temperature=temperature, top_k=top_k, top_p=top_p,
                        generator=g)
    counts = torch.bincount(tok, minlength=logits.numel()).double()
    p = torch.softmax(logits.double() / temperature, -1)
    order = torch.argsort(p, descending=True)
    keep = torch.zeros_like(p, dtype=torch.bool)
    if top_k:
        keep[order[:top_k]] = True
    elif top_p < 1.0:
        before = torch.cumsum(p[order], 0) - p[order]
        keep[order[before < top_p]] = True
    else:
        keep[:] = True
    p = torch.where(keep, p, 0.0)
    p = p / p.sum()
    assert float(counts[~keep].sum()) == 0.0
    exp = p[keep] * n
    chi2 = float(((counts[keep] - exp) ** 2 / exp).sum())
    assert chi2 < stats.chi2.ppf(0.999, int(keep.sum()) - 1), chi2


def test_the_cuda_step_has_no_cpu_fallback():
    m = _model('llama', 4)
    with pytest.raises(RuntimeError, match='CUDA device'):
        Generator(m, 1, 16)
    q = torch.zeros(1, 256, dtype=torch.float16)
    cache = torch.zeros(1, 4, 16, 64, dtype=torch.float16)
    with pytest.raises(RuntimeError, match='CUDA device only'):
        CudaDecodeAttention()(q, q, q, cache, cache, torch.zeros(1, dtype=torch.int32), 0.125)


def test_torch_attention_restatement_matches_a_per_sequence_loop():
    """oracle/attn.py against a plain loop over sequences and heads in float64 (ragged positions, GQA)."""
    g = torch.Generator().manual_seed(9)
    B, nh, nkv, hd, L = 3, 8, 2, 16, 10
    pos = torch.tensor([0, 4, 9])
    q, kn, vn = (torch.randn(B, n * hd, generator=g, dtype=torch.float64) for n in (nh, nkv, nkv))
    kc, vc = torch.randn(B, nkv, L, hd, generator=g, dtype=torch.float64), torch.randn(B, nkv, L, hd, generator=g, dtype=torch.float64)
    k0, v0 = kc.clone(), vc.clone()
    out = TorchDecodeAttention()(q, kn, vn, kc, vc, pos, 0.3)
    for b in range(B):
        p = int(pos[b])
        k0[b, :, p], v0[b, :, p] = kn[b].view(nkv, hd), vn[b].view(nkv, hd)
        for h in range(nh):
            kv = h // (nh // nkv)
            w = torch.softmax(0.3 * (k0[b, kv, :p + 1] @ q[b, h * hd:(h + 1) * hd]), 0)
            assert torch.allclose(out[b, h * hd:(h + 1) * hd], w @ v0[b, kv, :p + 1])
    assert torch.equal(kc, k0) and torch.equal(vc, v0)


def test_decode_attention_argument_errors_surface_before_any_launch():
    """The C entry point's shape checks (no device needed: they return before any CUDA call)."""
    from quip_b200 import _lib
    lib = _lib.load()
    p, pos = 1 << 20, 1 << 21                                                   # aligned stand-in device addresses

    def call(nh, nkv, hd, ws, q=p):
        return lib.quip_decode_attention(q, p, p, p, p, pos, 2, nh, nkv, 64, hd, 0.1, p, p, ws, None)
    assert call(8, 8, 96, 1 << 30) == 4 and b'head_dim 96' in lib.quip_last_error()
    assert call(6, 2, 64, 1 << 30) == 4 and b'3 query heads per KV head' in lib.quip_last_error()
    assert call(6, 4, 64, 1 << 30) == 1
    assert call(8, 8, 64, 16) == 2 and b'workspace' in lib.quip_last_error()
    assert call(8, 8, 64, 1 << 30, q=None) == 1
    assert call(8, 8, 64, 1 << 30, q=p + 2) == 1 and b'aligned' in lib.quip_last_error()
    need = _lib.C.c_size_t(0)
    assert lib.quip_decode_attention_workspace_bytes(2, 8, 300, 64, _lib.C.byref(need)) == 0
    assert need.value == 2 * 8 * 3 * (64 + 2) * 4                               # three 128-position splits
