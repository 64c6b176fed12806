"""quip_decode_attention (csrc/attn_decode.cu) against a float64 restatement, and generation (quip_b200/generate.py) on
packed tiny models against the HF forward with a KV cache."""
import pytest
import torch

from oracle.attn import TorchDecodeAttention

pytestmark = pytest.mark.gpu

MAX_LEN = 300                     # three 128-position splits, the last one partial
SPECIAL = [0, 1, 127, 128, 129, 255, 256, MAX_LEN - 1]


def _positions(B, g):
    if B == 1:
        return [[p] for p in SPECIAL]
    if B == 3:
        return [[0, 128, MAX_LEN - 1], [1, 127, 256]]
    rest = torch.randint(0, MAX_LEN, (B - len(SPECIAL),), generator=g).tolist()
    return [SPECIAL + rest]


@pytest.mark.parametrize('nh,nkv,hd', [(32, 32, 128), (64, 8, 128), (32, 32, 64), (56, 56, 128)])
@pytest.mark.parametrize('B', [1, 3, 32])
def test_decode_attention_matches_float64(nh, nkv, hd, B):
    from quip_b200.generate import CudaDecodeAttention
    g = torch.Generator().manual_seed(nh * 1000 + hd + B)
    attn = CudaDecodeAttention()
    scale = hd ** -0.5
    for pos_list in _positions(B, g):
        pos = torch.tensor(pos_list, dtype=torch.int32)
        q = torch.randn(B, nh * hd, generator=g).half().cuda()
        kn, vn = (torch.randn(B, nkv * hd, generator=g).half().cuda() for _ in range(2))
        k0, v0 = (torch.randn(B, nkv, MAX_LEN, hd, generator=g).half().cuda() for _ in range(2))
        kc, vc = k0.clone(), v0.clone()
        out = attn(q, kn, vn, kc, vc, pos.cuda(), scale)
        torch.cuda.synchronize()
        k64, v64 = k0.double(), v0.double()
        ref = TorchDecodeAttention()(q.double(), kn.double(), vn.double(), k64, v64, pos.cuda(), scale)
        err = (out.double() - ref).view(B, nh, hd).norm(dim=-1) / ref.view(B, nh, hd).norm(dim=-1)
        assert float(err.max()) <= 1e-3, (pos_list, float(err.max()))
        # the new rows land at pos[b] bit for bit; every other row is unchanged
        rows = torch.arange(B)
        want_k, want_v = k0.clone(), v0.clone()
        want_k[rows, :, pos.long()] = kn.view(B, nkv, hd)
        want_v[rows, :, pos.long()] = vn.view(B, nkv, hd)
        assert torch.equal(kc, want_k) and torch.equal(vc, want_v)
        # deterministic: a second run on the same inputs is bit-identical
        kc2, vc2 = k0.clone(), v0.clone()
        out2 = attn(q, kn, vn, kc2, vc2, pos.cuda(), scale)
        assert torch.equal(out, out2) and torch.equal(kc2, kc)


def test_decode_attention_rejects_unsupported_shapes():
    from quip_b200 import _lib
    from quip_b200.generate import CudaDecodeAttention
    q = torch.zeros(1, 4 * 96, dtype=torch.float16, device='cuda')
    cache = torch.zeros(1, 4, 16, 96, dtype=torch.float16, device='cuda')
    with pytest.raises(_lib.QuipError, match='head_dim 96'):
        CudaDecodeAttention()(q, q, q, cache, cache, torch.zeros(1, dtype=torch.int32, device='cuda'), 0.1)


def _packed(family, kv_heads=4):
    from transformers import LlamaConfig, OPTConfig
    from quip_b200.synth import build_synthetic_model
    if family == 'llama':
        cfg = LlamaConfig(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4,
                          num_key_value_heads=kv_heads, vocab_size=320, max_position_embeddings=128)
        seed = 5
    else:
        cfg = OPTConfig(hidden_size=256, ffn_dim=1024, num_hidden_layers=2, num_attention_heads=4, vocab_size=320,
                        max_position_embeddings=128, word_embed_proj_dim=256)
        seed = 6
    return build_synthetic_model(cfg, torch.device('cuda:0'), bits=2, incoh='blocked', rescale=True, seed=seed, seqlen=64)


def _norms(model):
    if model.config.model_type == 'llama':
        return [m for l in model.model.layers for m in (l.input_layernorm, l.post_attention_layernorm)] + [model.model.norm]
    d = model.model.decoder
    return [m for l in d.layers for m in (l.self_attn_layer_norm, l.final_layer_norm)] + [d.final_layer_norm]


LENS = (3, 7, 12)
CASES = [('llama', 4, False), ('llama', 2, False), ('llama', 2, True), ('opt', 4, False)]


@pytest.mark.parametrize('family,kv,fused_glue', CASES)
def test_generator_logits_match_hf_decode_graph_equals_eager(family, kv, fused_glue):
    """Teacher-forced ragged batch: every row against the HF forward with a KV cache on its prompt alone, within 3x what
    one-ulp flips in 3e-5 of the HF norm outputs do to the HF decode itself (tests/test_gpu_decode.py's control); graph
    replay equals the eager step bit for bit; each row equals the sequence run alone."""
    import bench
    from quip_b200 import fused
    from quip_b200.generate import Generator
    model = _packed(family, kv)
    g = torch.Generator().manual_seed(3)
    prompts = [torch.randint(0, 320, (n,), generator=g).cuda() for n in LENS]
    feed = torch.randint(0, 320, (6, len(LENS)), generator=g).cuda()
    ops = fused.CudaGlue() if fused_glue else None

    def run(prompts, feed, graph):
        gen = Generator(model, len(prompts), 32, ops=ops)
        if graph:
            gen.capture()
        res = [gen.prefill(prompts).float().clone()]
        res += [gen.step(feed[i]).float().clone() for i in range(feed.shape[0])]
        return res

    def hf(p, col, flip):
        past, res = None, []
        for i, x in enumerate([p[None]] + [feed[j, col].view(1, 1) for j in range(feed.shape[0])]):
            hooks = bench._ulp_flip_hooks(_norms(model), 3e-5, seed=i) if flip else []
            try:
                out = model(x, past_key_values=past, use_cache=True)
            finally:
                for hk in hooks:
                    hk.remove()
            past = out.past_key_values
            res.append(out.logits[0, -1].float())
        return res

    with torch.no_grad():
        eager, graph = run(prompts, feed, False), run(prompts, feed, True)
        worst = control = 0.0
        for i, (e, gr) in enumerate(zip(eager, graph)):
            assert torch.equal(e, gr), i
        for b, p in enumerate(prompts):
            want, ctrl = hf(p, b, False), hf(p, b, True)
            alone = run([p], feed[:, b:b + 1], True)
            for i, (gr, w, c, a) in enumerate(zip(graph, want, ctrl, alone)):
                worst = max(worst, float((gr[b] - w).norm() / w.norm()))
                control = max(control, float((c - w).norm() / w.norm()))
                err = float((gr[b] - a[0]).norm() / a[0].norm())
                assert err < 5e-3, (b, i, err)
    assert worst < max(2e-3, 3.0 * control), (worst, control)


@pytest.mark.parametrize('family,kv', [('llama', 2), ('opt', 4)])
def test_greedy_tokens_from_the_graph_equal_the_eager_path(family, kv):
    from quip_b200.generate import generate
    model = _packed(family, kv)
    g = torch.Generator().manual_seed(4)
    prompts = [torch.randint(0, 320, (n,), generator=g).cuda() for n in LENS]
    with torch.no_grad():
        eager = generate(model, prompts, 16, graph=False)
        graph = generate(model, prompts, 16, graph=True)
        s1 = generate(model, prompts, 16, do_sample=True, top_k=20, top_p=0.9, seed=7)
        s2 = generate(model, prompts, 16, do_sample=True, top_k=20, top_p=0.9, seed=7)
    for p, e, gr, a, b in zip(prompts, eager, graph, s1, s2):
        assert torch.equal(e, gr) and e.numel() == p.numel() + 16
        assert torch.equal(e[:p.numel()], p.cpu())
        assert torch.equal(a, b)                                   # seeded sampling replayed from the graph
