"""Independent restatements of one packed linear in plain torch, for checking -- never used to compute a result.

Two checkers, both built from data the CUDA path does not share with them beyond the stored buffers:

  * `restated_forward(ql, x)`: fp32 restatement of QuantLinear.forward from the module's own buffers and pass descriptors
    (gather, 1/s, block-diagonal passes, Q = scales*codes - zeros, passes, gather, bias) with no fp16 rounding between the
    stages.  bench.py runs it on the layers of the model it times and reports the error in its JSON line; the GPU tests
    use it at the Llama-2-7B shapes.
  * `reference_dense_weight(parts)`: the dense fp16 weight the reference leaves behind after `postproc`
    (method.py:195-214): W_ref = fp16( fp16(U^T Qhat V) / scaleWH ), Qhat the fp16 grid values; the reference's effective
    forward is then F.linear(x, W_ref, bias) (bal.py:44-45, opt.py:263-264).  Pinned against the live reference by
    tests/golden/layer_big_1024.npz.

Neither is a fallback: QuantLinear.forward raises without the CUDA library.
"""
import torch

from .capture import Butterfly, LayerParts


@torch.no_grad()
def restated_forward(ql, x):
    from . import quant as Q
    d = ql._descriptor()
    K, N = ql.infeatures, ql.outfeatures
    dev = x.device

    def side(sd, h, name):
        n = sd.n
        for i in range(sd.npass if n else 0):
            ps = sd.passes[i]
            F_ = getattr(ql, f'{name}_f{i}').float()
            p, nblk = ps.p, ps.nblk
            if F_.shape[0] == 1 and nblk > 1:
                F_ = F_.expand(nblk, p, p)
            if ps.strided:
                h3 = h.reshape(-1, p, nblk)                                   # element j of block b at j*nblk + b
                h = torch.einsum('bij,mjb->mib', F_, h3).reshape(-1, n)
            else:
                h3 = h.reshape(-1, nblk, p)
                h = torch.einsum('bij,mbj->mbi', F_, h3).reshape(-1, n)
        return h

    h = x.float().reshape(-1, K)
    if d.V.n or d.inv_scale:
        idx = ql.v_idx.long() if (d.V.n and d.V.idx) else torch.arange(K, device=dev)
        h = h[:, idx] * (ql.inv_scale.float()[idx] if d.inv_scale else 1.0)
    h = side(d.V, h, 'v')
    codes = Q.unpack_codes(ql.qweight, N, K, ql.bits).float()
    Qm = ql.scales.float().reshape(-1, 1) * codes - ql.zeros.float().reshape(-1, 1)
    z = h @ Qm.T
    z = side(d.U, z, 'u')
    if d.U.n and d.U.idx:
        z = z[:, ql.u_idx.long()]
    if ql.bias is not None:
        z = z + ql.bias.float()
    return z


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def _bf_to(bf: Butterfly, dev):
    return Butterfly(bf.n, bf.B0.to(dev), bf.B1.to(dev), bf.p_in.to(dev), bf.p_out.to(dev))


@torch.no_grad()
def reference_dense_weight(parts: LayerParts, device):
    """W_ref (N, K) fp16 as the reference's postproc leaves it (method.py:195-214), from the captured parts."""
    from .quantize import butterfly_apply_t
    codes = parts.codes.to(device).float()
    grid = (parts.scales.to(device).float().reshape(-1, 1) * codes - parts.zeros.to(device).float().reshape(-1, 1)).half()
    w = grid.float()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        if parts.U is not None:
            U, V = _bf_to(parts.U, device), _bf_to(parts.V, device)
            w = butterfly_apply_t(U, w)                       # U^T @ Q
            w = butterfly_apply_t(V, w.T.contiguous()).T      # (V^T Q'^T)^T = Q' V
        w = w.half()                                          # method.py:204  w.to(fp16)
        if parts.scaleWH is not None:
            w = (w / parts.scaleWH.to(device).float()[None, :]).half()      # method.py:210-213 (fp16 / fp32 -> fp32 -> fp16)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return w.contiguous()
