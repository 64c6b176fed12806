"""CPU: the dense-weight restatement (quip_b200/selfcheck.reference_dense_weight, method.py:195-214) pinned against a
1024 x 1024 layer quantized by the live reference (tests/golden/layer_big_1024.npz, oracle/gen_golden_big.py)."""
import torch

from conftest import load_big_layer


def test_reference_dense_weight_reproduces_the_live_reference():
    from quip_b200.selfcheck import reference_dense_weight, rel_err
    tp, z = load_big_layer()
    W = reference_dense_weight(tp, 'cpu')
    want = torch.from_numpy(z['wref_rows'])
    same = (W[:8] == want).float().mean()
    assert float(same) > 0.99, float(same)                    # the rest: one-ulp flips from the fp32 summation order
    assert rel_err(W[:8].float(), want.float()) < 1e-4
    x = torch.from_numpy(z['x'])
    y = torch.nn.functional.linear(x.float(), W.float()).half().float()      # the reference's F.linear returns fp16
    assert rel_err(y, torch.from_numpy(z['y_ref']).float()) < 2e-4


def test_big_layer_packs_with_bit_exact_codes():
    from quip_b200 import quant as Q
    from quip_b200.incoherence import plan_side
    tp, z = load_big_layer()
    N, K = tp.codes.shape
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    uo, vo = plan_side(tp.U, 'U').order, plan_side(tp.V, 'V').order
    assert torch.equal(ql.codes(), tp.codes[uo][:, vo])
    assert int(ql.meta[1]) == 1                               # qfn 'b': symmetric grid


def test_fp32_restatement_agrees_with_the_reference_outputs_on_the_cpu():
    """quip_b200/selfcheck.restated_forward (the checker bench.py and the GPU tests use) against the live reference's y_ref of
    the golden layers and of the 1024 x 1024 layer: it is an independent, correct statement of the layer."""
    import numpy as np
    from conftest import LAYER_NAMES, load_layer, parts_to_torch
    from quip_b200 import quant as Q
    from quip_b200.selfcheck import rel_err, restated_forward
    for name in LAYER_NAMES:
        parts, z = load_layer(name)
        tp = parts_to_torch(parts)
        N, K = tp.codes.shape
        ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
        ql.pack_parts(tp)
        y = restated_forward(ql, torch.from_numpy(z['x']))
        assert rel_err(y, torch.from_numpy(z['y_ref'].astype(np.float32))) < 6e-4, name      # the reference's own fp16 roundings
    tp, z = load_big_layer()
    N, K = tp.codes.shape
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    y = restated_forward(ql, torch.from_numpy(z['x']))
    assert rel_err(y, torch.from_numpy(z['y_ref']).float()) < 6e-4
