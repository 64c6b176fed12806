"""End-to-end golden fixture: a tiny random-init OPT quantized and evaluated by the LIVE reference.

Called from oracle/gen_golden.py (`--only models`).  The reference's own opt_sequential (opt.py:29-190)
quantizes the model (2-bit LDLQ with --incoh_processing semantics) under quip_b200.capture.Capture;
the reference's own opt_eval (opt.py:193-299) then prints the perplexity of the resulting dense fp16
model on CPU.  Saved: the model config, the dense fp16 state_dict after quantization (what the
reference's --save writes), every captured layer's parts, the token stream and the printed ppl.
"""
import contextlib
import io
import os
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')

TINY_OPT = dict(vocab_size=512, hidden_size=128, ffn_dim=512, num_hidden_layers=2, num_attention_heads=4,
                max_position_embeddings=64, word_embed_proj_dim=128, do_layer_norm_before=True)


def main(mods):
    quant, method, bal, vb = mods
    with contextlib.redirect_stdout(io.StringIO()):
        import opt as ref_opt                       # the reference's opt.py
    from transformers import OPTConfig, OPTForCausalLM
    from quip_b200.capture import Capture

    torch.manual_seed(0)
    np.random.seed(0)
    cfg = OPTConfig(**TINY_OPT)
    torch.set_default_dtype(torch.half)
    model = OPTForCausalLM(cfg).eval()
    torch.set_default_dtype(torch.float)
    model.seqlen = cfg.max_position_embeddings
    S = model.seqlen
    g = torch.Generator().manual_seed(1)
    calib = [(torch.randint(0, cfg.vocab_size, (1, S), generator=g), None) for _ in range(8)]
    test_ids = torch.randint(0, cfg.vocab_size, (1, 4 * S), generator=g)
    args = types.SimpleNamespace(nsamples=8, quant='ldlq', wbits=2, npasses=0, unbiased=False, qfn='b',
                                 pre_gptqH=True, pre_rescale=True, pre_proj=True, pre_proj_extra=0,
                                 percdamp=0.01, lazy_batch=False, groupsize=-1)
    dev = torch.device('cpu')
    layers_by_id = {}
    for name, mod in model.named_modules():
        if isinstance(mod, torch.nn.Linear):
            layers_by_id[id(mod)] = name
    with Capture(method, bal) as cap, contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ref_opt.opt_sequential(model, calib, dev, args)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
        ref_opt.opt_eval(model, types.SimpleNamespace(input_ids=test_ids), dev)
    ppl = float(buf.getvalue().strip().splitlines()[-1])

    out = dict(config=np.array(repr(TINY_OPT)), test_ids=test_ids.numpy(), ppl=np.float64(ppl))
    sd = model.state_dict()
    assert torch.equal(sd['lm_head.weight'], sd['model.decoder.embed_tokens.weight'])
    for k, v in sd.items():
        if k != 'lm_head.weight':                   # tied to the embedding: stored once, which keeps each file under 1 MB
            out['sd/' + k] = v.numpy()
    path = os.path.join(OUT, 'tiny_opt_2bit_incoh.npz')
    np.savez_compressed(path, **out)
    print('wrote', os.path.relpath(path, ROOT), f'{os.path.getsize(path)/1024:.0f} KiB', 'reference ppl', ppl)
    out = {}
    names = []
    for lid, parts in cap.records.items():
        name = layers_by_id[lid]
        names.append(name)
        p = 'parts/' + name + '/'
        out[p + 'codes'] = parts.codes.numpy()
        out[p + 'scales'] = parts.scales.numpy()
        out[p + 'zeros'] = parts.zeros.numpy()
        out[p + 'scaleWH'] = parts.scaleWH.numpy()
        if parts.bias is not None:
            out[p + 'bias'] = parts.bias.numpy()
        for side in 'UV':
            b = getattr(parts, side)
            out[p + side + '_B0'] = b.B0.numpy()
            out[p + side + '_B1'] = b.B1.numpy()
            out[p + side + '_p_in'] = b.p_in.numpy()
            out[p + side + '_p_out'] = b.p_out.numpy()
    out['names'] = np.array(names)
    path = os.path.join(OUT, 'tiny_opt_2bit_incoh_parts.npz')
    np.savez_compressed(path, **out)
    print('wrote', os.path.relpath(path, ROOT), f'{os.path.getsize(path)/1024:.0f} KiB', 'layers', len(names))
