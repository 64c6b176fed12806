"""Golden 1024 x 1024 layer quantized by the LIVE reference (build container only).

Run:  python -m oracle.gen_golden_big [--method ldlq|nearest] [--n 1024 --k 1024]

The small golden layers (oracle/gen_golden.py) never exceed K = 640.  This fixture is a whole Linear through the
reference's own flow (`Balance.preproc` with --pre_gptqH --pre_rescale --pre_proj, method.py:139-193; `fasterquant`,
bal.py:21-48; `postproc`, method.py:195-214), so that the multi-tile persistent path (its 16 tokens replicated to
thousands), the 32 x 32 butterflies and the one-kernel sides are checked against the reference's own dense fp16 output
`F.linear(x, W_ref)`.  1024 x 1024 keeps the file under 1 MB; a 4096 x 4096 layer needs 8 MB of codes and factors.

To stay small the file keeps what the packer needs (codes as 2-bit planes, grid parameters, scaleWH, butterfly factors
and permutations) plus a 16-token x / y_ref slice and eight rows of W_ref -- not W_ref itself.
"""
import argparse
import contextlib
import io
import os
import time

import numpy as np
import torch
import torch.nn as nn

from oracle.gen_golden import OUT, ROOT, import_reference, synth_inputs


def pack2(codes):
    """(N, K) uint8 codes < 4 -> (N, K/4) uint8, code k at bits 2*(k % 4) of byte k // 4."""
    c = codes.astype(np.uint8).reshape(codes.shape[0], -1, 4)
    return (c[..., 0] | (c[..., 1] << 2) | (c[..., 2] << 4) | (c[..., 3] << 6)).astype(np.uint8)


def unpack2(packed):
    p = packed[..., None] >> np.array([0, 2, 4, 6], dtype=np.uint8)
    return (p & 3).reshape(packed.shape[0], -1).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--method', default='ldlq')
    ap.add_argument('--n', type=int, default=1024)
    ap.add_argument('--k', type=int, default=1024)
    ap.add_argument('--tokens', type=int, default=2048)
    ap.add_argument('--name', default='big_1024')
    a = ap.parse_args()
    mods = import_reference()
    quant, method, bal, _ = mods
    from quip_b200.capture import Capture
    N, K, seed = a.n, a.k, 4096
    torch.manual_seed(seed)
    np.random.seed(seed)
    layer = nn.Linear(K, N, bias=False).half()                      # Llama: no bias
    X = synth_inputs(K, a.tokens, seed + 1)
    t0 = time.time()
    with Capture(method, bal) as cap:
        qm = bal.Balance(layer)
        qm.configure(a.method, 2, 0, False)                          # bal.py:15
        qm.quantizer = quant.Quantizer()
        qm.quantizer.configure(2, perchannel=True, sym=False, qfn='b', mse=False)      # opt.py:124-128
        qm.add_batch(X.unsqueeze(0), None)                           # method.py:98-120
        qm.post_batch()
        qm.preproc(preproc_gptqH=True, percdamp=0.01, preproc_rescale=True, preproc_proj=True,
                   preproc_proj_extra=0)                             # opt.py:154-157 as --incoh_processing runs it
        with contextlib.redirect_stderr(io.StringIO()):
            qm.fasterquant(lazy_batch=False)                         # opt.py:161
        parts = cap.parts_for(layer)
    print(f'reference quantization ({a.method}) of {N} x {K}: {time.time() - t0:.1f} s')
    x = synth_inputs(K, 16, seed + 2)
    with torch.no_grad():
        W_ref = layer.weight.data
        y_ref = nn.functional.linear(x, W_ref, None)                 # the reference's effective forward
    codes = parts.codes.numpy()
    assert codes.max() < 4 and np.array_equal(unpack2(pack2(codes)), codes)
    d = dict(bits=np.int32(2), qfn=np.array('b'), method=np.array(a.method), N=np.int32(N), K=np.int32(K),
             codes2=pack2(codes), scales=parts.scales.numpy(), zeros=parts.zeros.numpy(),
             scaleWH=parts.scaleWH.numpy(), x=x.numpy(), y_ref=y_ref.numpy(), wref_rows=W_ref[:8].numpy())
    for side in 'UV':
        b = getattr(parts, side)
        d.update({f'{side}_B0': b.B0.numpy().astype(np.float32), f'{side}_B1': b.B1.numpy().astype(np.float32),
                  f'{side}_p_in': b.p_in.numpy().astype(np.int32), f'{side}_p_out': b.p_out.numpy().astype(np.int32)})
    path = os.path.join(OUT, f'layer_{a.name}.npz')
    np.savez_compressed(path, **d)
    print('wrote', os.path.relpath(path, ROOT), f'{os.path.getsize(path) / 2 ** 20:.1f} MiB')


if __name__ == '__main__':
    main()
