"""Kernel launches per QuantLinear forward (quip_launch_count, the `gpu_launches` of every bench line), pinned per token
count.  The counts follow from the routing of quip_qlinear_forward with the library defaults:

  * M > 32: a side of 64 x 64 blocks is one fused kernel (gather, both passes, row sums); an 11008 side (688 x 16
    blocks) is a gather plus a dense 688 pass plus a 16-wide pass; the contraction is one tcgen05 launch.
  * M <= 32: each pass is one few-token launch, the K-side gather riding on the first pass when its blocks are at most
    128 wide and the N-side gather + bias on the last pass; the contraction is one qgemv (<= 8 tokens) or split-K launch.
"""
import ctypes as C

import pytest
import torch

from quip_b200 import _lib, quant as Q
from quip_b200.synth import synth_layer_parts

pytestmark = pytest.mark.gpu

# (K, N, bits, incoh, qfn): the 4096 x 4096 layer is the decode bench's 2-bit blocked layer with rescale
LAYERS = {
    '2b_4096': (4096, 4096, 2, 'blocked', 'b'),
    '2b_4096_11008': (4096, 11008, 2, 'blocked', 'b'),
    '2b_11008_4096': (11008, 4096, 2, 'blocked', 'b'),
    '3b_4096_asym': (4096, 4096, 3, 'blocked', 'a'),
    '4b_plain_bias': (4096, 4096, 4, None, 'b'),
}

# (layer, M) -> launches of one forward
EXPECTED = {
    # V pass (+gather), V pass, qgemv / split-K, U pass, U pass (+scatter, bias) -- fused side, tcgen05, fused side
    ('2b_4096', 1): 5, ('2b_4096', 5): 5, ('2b_4096', 8): 5, ('2b_4096', 16): 5, ('2b_4096', 32): 5,
    ('2b_4096', 33): 3, ('2b_4096', 2048): 3,
    # N side of 11008: 16-wide pass, 688 pass (+scatter) few-token; 16-wide pass, dense 688 pass, gather above 32
    ('2b_4096_11008', 1): 5, ('2b_4096_11008', 2048): 5,
    # K side of 11008: its first pass is 688 wide, so the gather is a launch of its own at every token count
    ('2b_11008_4096', 1): 6, ('2b_11008_4096', 2048): 5,
    # asymmetric grid: the fused K side also writes the row sums the tcgen05 kernel needs
    ('3b_4096_asym', 1): 5, ('3b_4096_asym', 2048): 3,
    # no incoherence: the 1/s gather, then the contraction with the bias
    ('4b_plain_bias', 1): 2, ('4b_plain_bias', 300): 2,
}

_modules = {}


def _layer(name):
    if name not in _modules:
        K, N, bits, incoh, qfn = LAYERS[name]
        tp = synth_layer_parts(K=K, N=N, bits=bits, incoh=incoh, rescale=True, bias=incoh is None, seed=K + N + bits,
                               qfn=qfn)
        ql = Q.QuantLinear(infeatures=K, outfeatures=N, **Q.spec_from_parts(tp)).cuda()
        ql.pack_parts(tp)
        _modules[name] = ql
    return _modules[name]


def _counted(fn):
    lib = _lib.load()
    torch.cuda.synchronize()
    before = lib.quip_launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, lib.quip_launch_count() - before


@pytest.mark.parametrize('name,M', sorted(EXPECTED))
def test_launches_per_forward(name, M):
    ql = _layer(name)
    x = torch.randn(M, ql.infeatures, device='cuda').half()
    ql(x)                                                  # descriptors and workspace are set up on the first call
    y, launches = _counted(lambda: ql(x))
    assert launches == EXPECTED[(name, M)], (name, M, launches)
    assert bool(torch.isfinite(y).all())


def test_launches_of_pack_and_fp16_qgemv():
    """quip_pack_codes is one launch; quip_qgemm(path=1) at six tokens is one fp16 qgemv launch."""
    from gpu_util import stream
    lib = _lib.load()
    N, K = 4096, 4096
    codes = torch.randint(0, 4, (N, K), dtype=torch.uint8, device='cuda')
    qw, launches = _counted(lambda: Q.pack_codes(codes, 2))
    assert launches == 1
    sc = torch.full((N,), 0.01, device='cuda')
    ze = sc * 1.5
    d = _lib.QuipLinearDesc()
    d.K, d.N, d.bits, d.flags = K, N, 2, _lib.QUIP_FLAG_SYMMETRIC
    d.qweight, d.scales, d.zeros = qw.data_ptr(), sc.data_ptr(), ze.data_ptr()
    M = 6
    need = C.c_size_t()
    _lib.check(lib.quip_qlinear_workspace_bytes(C.byref(d), M, C.byref(need)))
    ws = torch.zeros(need.value, dtype=torch.uint8, device='cuda')
    x = torch.randn(M, K, device='cuda').half()
    z = torch.empty(M, N, dtype=torch.float16, device='cuda')
    _, launches = _counted(lambda: _lib.check(lib.quip_qgemm(C.byref(d), _lib.ptr(x), None, None, _lib.ptr(z), M, 1,
                                                             _lib.ptr(ws), ws.numel(), stream())))
    assert launches == 1
    want = (x.float() @ ((Q.unpack_codes(qw, N, K, 2).float() - 1.5) * 0.01).t())
    assert float((z.float() - want).norm() / want.norm()) < 1e-3


@pytest.mark.parametrize('name', ['2b_4096', '2b_11008_4096', '4b_plain_bias'])
def test_one_token_without_pdl_is_bit_identical(name):
    """quip_config('pdl', 0) launches the same kernels without the programmatic-dependent-launch attribute: same
    count, same bits."""
    lib = _lib.load()
    ql = _layer(name)
    x = torch.randn(1, ql.infeatures, device='cuda').half()
    ql(x)
    try:
        y1, n1 = _counted(lambda: ql(x).clone())
        _lib.check(lib.quip_config(b'pdl', 0))
        y0, n0 = _counted(lambda: ql(x).clone())
    finally:
        _lib.check(lib.quip_config(b'pdl', 1))
    assert n0 == n1 == EXPECTED[(name, 1)]
    assert torch.equal(y0, y1)
