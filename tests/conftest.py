import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason='no CUDA device')
    for item in items:
        if 'gpu' in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def _seeded(request):
    """Every test starts from the same generator state (CPU and CUDA), derived from its own name: a test that draws inputs
    with torch.randn(...) sees the same numbers in every run and on every box, whatever ran before it."""
    import zlib

    import torch
    torch.manual_seed(zlib.crc32(request.node.nodeid.encode()) & 0x7fffffff)   # seeds the CUDA generators too
    yield


def load_layer(name):
    """Golden layer fixture -> `parts` dict in the oracle's numpy convention."""
    import numpy as np
    z = np.load(os.path.join(GOLDEN, f'layer_{name}.npz'))
    parts = dict(bits=int(z['bits']), qfn=str(z['qfn']), codes=z['codes'], scales=z['scales'],
                 zeros=z['zeros'], bias=z['bias'] if 'bias' in z else None,
                 scaleWH=z['scaleWH'] if 'scaleWH' in z else None, U=None, V=None)
    for side in 'UV':
        if f'{side}_B0' in z:
            parts[side] = ([z[f'{side}_B0'], z[f'{side}_B1']], z[f'{side}_p_in'], z[f'{side}_p_out'])
    return parts, z


LAYER_NAMES = ['l2b_incoh', 'l2b_incoh_rg', 'l3b_incoh', 'l4b_plain', 'l2b_kron', 'l4b_noperm',
               'l3b_rescale', 'l2b_qfna_proj']


def parts_to_torch(parts):
    """numpy `parts` dict (load_layer) -> quip_b200.capture.LayerParts."""
    import torch
    from quip_b200.capture import Butterfly, LayerParts

    def bfly(b, n):
        if b is None:
            return None
        (B, p_in, p_out) = b
        return Butterfly(n, torch.from_numpy(B[0]).float(), torch.from_numpy(B[1]).float(),
                         torch.from_numpy(p_in).long(), torch.from_numpy(p_out).long())
    N, K = parts['codes'].shape
    return LayerParts(bits=parts['bits'], qfn=parts['qfn'], codes=torch.from_numpy(parts['codes']),
                      scales=torch.from_numpy(parts['scales']), zeros=torch.from_numpy(parts['zeros']),
                      bias=None if parts['bias'] is None else torch.from_numpy(parts['bias']),
                      scaleWH=None if parts['scaleWH'] is None else torch.from_numpy(parts['scaleWH']),
                      U=bfly(parts['U'], N), V=bfly(parts['V'], K))


def load_tiny_opt():
    """Tiny OPT fixture quantized + evaluated by the live reference (oracle/gen_golden_models.py).
    Returns (dense fp16 model as the reference left it, {layer name: LayerParts}, test ids, reference ppl)."""
    import ast
    import numpy as np
    import torch
    from transformers import OPTConfig
    from quip_b200.capture import Butterfly, LayerParts
    from quip_b200.opt import get_opt
    m = np.load(os.path.join(GOLDEN, 'tiny_opt_2bit_incoh.npz'))
    z = np.load(os.path.join(GOLDEN, 'tiny_opt_2bit_incoh_parts.npz'))
    cfg = OPTConfig(**ast.literal_eval(str(m['config'])))
    model = get_opt(cfg)
    sd = {k[3:]: torch.from_numpy(m[k]) for k in m.files if k.startswith('sd/')}
    sd['lm_head.weight'] = sd['model.decoder.embed_tokens.weight']      # tied in OPT: stored once
    model.load_state_dict(sd)
    parts = {}
    for name in [str(n) for n in z['names']]:
        p = 'parts/' + name + '/'
        N, K = z[p + 'codes'].shape

        def bf(side, n):
            return Butterfly(n, torch.from_numpy(z[p + side + '_B0']), torch.from_numpy(z[p + side + '_B1']),
                             torch.from_numpy(z[p + side + '_p_in']), torch.from_numpy(z[p + side + '_p_out']))
        parts[name] = LayerParts(bits=2, qfn='b', codes=torch.from_numpy(z[p + 'codes']),
                                 scales=torch.from_numpy(z[p + 'scales']), zeros=torch.from_numpy(z[p + 'zeros']),
                                 bias=torch.from_numpy(z[p + 'bias']) if (p + 'bias') in z.files else None,
                                 scaleWH=torch.from_numpy(z[p + 'scaleWH']), U=bf('U', N), V=bf('V', K))
    return model, parts, torch.from_numpy(m['test_ids']), float(m['ppl'])


def load_big_layer(name='big_1024'):
    """Golden 1024 x 1024 layer quantized by the live reference (oracle/gen_golden_big.py) -> (LayerParts, npz)."""
    import numpy as np
    import torch
    from quip_b200.capture import Butterfly, LayerParts
    z = np.load(os.path.join(GOLDEN, f'layer_{name}.npz'))
    N, K = int(z['N']), int(z['K'])
    p = z['codes2'][..., None] >> np.array([0, 2, 4, 6], dtype=np.uint8)
    codes = (p & 3).reshape(N, K).astype(np.uint8)

    def bf(s, n):
        return Butterfly(n, torch.from_numpy(z[s + '_B0']), torch.from_numpy(z[s + '_B1']),
                         torch.from_numpy(z[s + '_p_in']).long(), torch.from_numpy(z[s + '_p_out']).long())
    tp = LayerParts(bits=2, qfn='b', codes=torch.from_numpy(codes), scales=torch.from_numpy(z['scales']),
                    zeros=torch.from_numpy(z['zeros']), scaleWH=torch.from_numpy(z['scaleWH']), U=bf('U', N), V=bf('V', K))
    return tp, z
