"""The kernels of the benchmark step at the benchmark's own shapes, against independent references.

bench.py runs `qgemm_tc_kernel<2,256,false>` at (N, K, M) in {(4096, 4096), (11008, 4096), (4096, 11008)} x 2048 tokens:
256-688 tiles on 148 persistent CTAs, i.e. every CTA walks several tiles and exercises the cross-tile weight prefetch, the
ring-phase wrap and the double-buffered TMEM accumulator -- none of which the small oracle cases (<= 86 tiles) reach.
Here those launches are compared with a float64 contraction of the unpacked codes (tolerance 3e-4: the fp16 output
rounding), checked for run-to-run determinism, and whole QuantLinear forwards at the same shapes are compared with
  * the fp32 restatement of the pipeline (quip_b200/selfcheck.restated_forward),
  * the reference's own dense path F.linear(x, W_ref), W_ref = fp16(fp16(U^T Q V)/s) (method.py:195-214), restated in
    quip_b200/selfcheck.reference_dense_weight and pinned to the live reference by tests/golden/layer_big_1024.npz,
  * the live reference's y_ref of that golden layer, replicated to 2048 and 10240 tokens so it runs through the tcgen05
    route, at 10240 tokens on 320 tiles (every persistent CTA walks several).
Tolerance for whole layers: 1e-3 relative (north_star), norm-wise.
"""
import json
import os

import pytest
import torch

from conftest import ROOT, load_big_layer

pytestmark = pytest.mark.gpu

SHAPES = [(4096, 4096, 2048), (11008, 4096, 2048), (4096, 11008, 2048)]


def _report(case, **rec):
    os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
    with open(os.path.join(ROOT, 'gpurun_out', 'parity_report.jsonl'), 'a') as f:
        f.write(json.dumps(dict(case=case, **rec)) + '\n')


def _inputs(M, K, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    feat = 1.0 + 3.0 * torch.rand(K, device='cuda', generator=g)              # SURVEY 8(d) activation model
    return (torch.randn(M, K, device='cuda', generator=g) * feat).half()


@pytest.mark.parametrize('N,K,M', SHAPES + [(4096, 4096, 2048 + 77), (11008, 4096, 300)])
@pytest.mark.parametrize('symmetric', [True, False])
def test_tcgen05_gemm_at_bench_shapes_vs_float64(N, K, M, symmetric):
    from gpu_util import run_qgemm_dev
    from quip_b200.selfcheck import rel_err
    bits = 2
    g = torch.Generator(device='cuda').manual_seed(N + K + M + int(symmetric))
    codes = torch.randint(0, 4, (N, K), device='cuda', generator=g, dtype=torch.uint8)
    scales = (0.01 + 0.02 * torch.rand(N, device='cuda', generator=g)).float()
    cbar = (2 ** bits - 1) / 2.0
    zeros = scales * cbar if symmetric else scales * torch.randint(0, 4, (N,), device='cuda', generator=g).float()
    bias = None if symmetric else (0.1 * torch.randn(N, device='cuda', generator=g)).half()
    x = _inputs(M, K, N + M)
    z = run_qgemm_dev(codes, scales, zeros, bits, x, path=2, bias=bias, symmetric=symmetric)
    assert not torch.isnan(z).any()
    Qm = scales.double()[:, None] * codes.double() - zeros.double()[:, None]
    want = x.double() @ Qm.T
    if bias is not None:
        want += bias.double()
    err = rel_err(z, want)
    _report('qgemm_tc', N=N, K=K, M=M, symmetric=symmetric, rel_err_vs_float64=err)
    assert err < 3e-4, (N, K, M, symmetric, err)
    # per-tile check: no tile may be wrong while the norm hides it (128 output rows x 256 tokens per tile)
    d = (z.double() - want)
    for m0 in range(0, M, 256):
        blk = d[m0:m0 + 256].reshape(min(256, M - m0), -1)
        nb = (blk.shape[1] // 128) * 128
        e = blk[:, :nb].reshape(blk.shape[0], -1, 128).pow(2).sum((0, 2)).sqrt()
        r = want[m0:m0 + 256][:, :nb].reshape(blk.shape[0], -1, 128).pow(2).sum((0, 2)).sqrt()
        assert float((e / r).max()) < 6e-4, (m0, float((e / r).max()))
    again = run_qgemm_dev(codes, scales, zeros, bits, x, path=2, bias=bias, symmetric=symmetric)
    assert torch.equal(z, again), 'the persistent multi-tile path must be deterministic'


@pytest.mark.parametrize('K,N', [(4096, 4096), (4096, 11008), (11008, 4096)])
def test_quantlinear_at_bench_shapes(K, N):
    """Whole forward (side kernel / gather + dense 688 pass + 16-wide pass, GEMM, side) at M = 2048 and at the routes
    below it, against the fp32 restatement and against the reference's dense fp16 path."""
    from quip_b200 import quant as Q
    from quip_b200.selfcheck import reference_dense_weight, rel_err, restated_forward
    from quip_b200.synth import synth_layer_parts
    tp = synth_layer_parts(K=K, N=N, bits=2, incoh='blocked', rescale=True, bias=False, seed=K + N)
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    ql = ql.cuda()
    W_ref = reference_dense_weight(tp, 'cuda')
    x = _inputs(2048, K, K + N)
    for M in (2048, 2048 - 5, 129, 40):
        y = ql(x[:M])
        e_model = rel_err(y, restated_forward(ql, x[:M]))
        y_ref = torch.nn.functional.linear(x[:M], W_ref)                       # fp16 in, fp16 out: the reference's forward
        e_ref = rel_err(y, y_ref)
        _report('quantlinear_bench_shape', K=K, N=N, M=M, rel_err_vs_restatement=e_model, rel_err_vs_reference_dense=e_ref)
        assert e_model < 1e-3, (K, N, M, e_model)
        assert e_ref < 1e-3, (K, N, M, e_ref)
        assert torch.equal(y, ql(x[:M]))


@pytest.mark.parametrize('K,N', [(4096, 11008), (11008, 4096)])
def test_kronecker_layers_at_bench_shapes(K, N):
    """`bench.py --incoh kron`: one block per stage (method.py:38-39), every CTA of a pass reading the SAME factor -- the 688-wide
    dense pass with a shared block, the one-kernel 4096 sides with shared factors and the few-token routes."""
    from quip_b200 import quant as Q
    from quip_b200.selfcheck import reference_dense_weight, rel_err, restated_forward
    from quip_b200.synth import synth_layer_parts
    tp = synth_layer_parts(K=K, N=N, bits=2, incoh='kron', rescale=True, bias=False, seed=K + N + 1)
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    ql = ql.cuda()
    W_ref = reference_dense_weight(tp, 'cuda')
    x = _inputs(2048, K, K + N + 1)
    for M in (2048, 2043, 40, 16, 1):
        y = ql(x[:M])
        e_model = rel_err(y, restated_forward(ql, x[:M]))
        e_ref = rel_err(y, torch.nn.functional.linear(x[:M], W_ref))
        _report('quantlinear_bench_shape_kron', K=K, N=N, M=M, rel_err_vs_restatement=e_model, rel_err_vs_reference_dense=e_ref)
        assert e_model < 1e-3, (K, N, M, e_model)
        assert e_ref < 1e-3, (K, N, M, e_ref)
        assert torch.equal(y, ql(x[:M]))


def test_golden_1024_layer_from_the_live_reference():
    """tests/golden/layer_big_1024.npz: a 1024 x 1024 Linear quantized by the reference's own Balance flow (ldlq, 2 bits,
    --incoh_processing).  Its 16-token y_ref through every token-count route, including 2048 and 10240 tokens (the 16 rows
    replicated 128 and 640 times; 10240 tokens are 8 x 40 tiles on 148 persistent CTAs, so the multi-tile tcgen05 path is
    compared with the live reference's own output)."""
    from quip_b200 import quant as Q
    from quip_b200.incoherence import plan_side
    from quip_b200.selfcheck import reference_dense_weight, rel_err
    tp, z = load_big_layer()
    N, K = tp.codes.shape
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    ql = ql.cuda()
    uo, vo = plan_side(tp.U, 'U').order, plan_side(tp.V, 'V').order
    assert torch.equal(ql.codes().cpu(), tp.codes[uo][:, vo])                  # integer codes bit-exact
    x = torch.from_numpy(z['x']).cuda()
    y_ref = torch.from_numpy(z['y_ref']).cuda()
    for reps in (1, 3, 128, 640):                                               # 16, 48, 2048 and 10240 tokens
        y = ql(x.repeat(reps, 1))
        err = rel_err(y, y_ref.repeat(reps, 1))
        _report('golden_big_1024', M=16 * reps, rel_err_vs_reference=err)
        assert err < 1e-3, (reps, err)
        if reps > 1:
            assert torch.equal(y[:16], y[-16:])                                # same rows, whatever tile they land in
    for M in (1, 5):
        err = rel_err(ql(x[:M]), y_ref[:M])
        _report('golden_big_1024', M=M, rel_err_vs_reference=err)
        assert err < 1e-3, (M, err)
    # fresh activations at 10240 tokens against the dense weight restatement (pinned by tests/test_big_golden.py)
    W_ref = reference_dense_weight(tp, 'cuda')
    assert rel_err(W_ref[:8].float().cpu(), torch.from_numpy(z['wref_rows']).float()) < 1e-4
    xr = _inputs(10240, K, 7)
    err = rel_err(ql(xr), torch.nn.functional.linear(xr, W_ref))
    _report('golden_big_1024', M=10240, fresh_inputs=True, rel_err_vs_reference=err)
    assert err < 1e-3, err


@pytest.mark.parametrize('K,N', [(8192, 8192), (8192, 1024), (8192, 28672), (28672, 8192), (7168, 7168), (7168, 28672),
                                 (28672, 7168), (2048, 2048), (2048, 8192), (8192, 2048)])
def test_other_model_shapes_at_2048_tokens(K, N):
    """Layer shapes of BASELINE configs[1], [3], [4] (OPT-1.3b, OPT-30b, Llama-2-70B: sides 2048 = 64 x 32, 7168 = 224 x 32,
    8192 = 128 x 64, 28672 = 448 x 64, 1024 = 32 x 32) through the many-token route -- dense tcgen05 passes for the wide
    blocks, small-block passes, the one-kernel side where both blocks are 32 / 64 wide -- against the fp32 restatement."""
    from quip_b200 import quant as Q
    from quip_b200.selfcheck import rel_err, restated_forward
    from quip_b200.synth import synth_layer_parts
    tp = synth_layer_parts(K=K, N=N, bits=2, incoh='blocked', rescale=True, bias=(K in (7168, 2048) or N in (7168, 2048)), seed=K + N)
    ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp))
    ql.pack_parts(tp)
    ql = ql.cuda()
    x = _inputs(2048, K, K + N)
    for M in (2048, 333):
        y = ql(x[:M])
        err = rel_err(y, restated_forward(ql, x[:M]))
        _report('quantlinear_other_shapes', K=K, N=N, M=M, rel_err_vs_restatement=err)
        assert err < 1e-3, (K, N, M, err)
