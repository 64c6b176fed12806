"""TEST INFRASTRUCTURE -- torch restatement of quip_decode_attention (quip_b200/csrc/attn_decode.cu).

One decode step of attention for B sequences over the static cache: sequence b stores k_new / v_new at pos[b] of the
cache and attends to positions 0 .. pos[b], softmax and sums in fp32 (float64 inputs stay float64), the query heads of a
KV head being consecutive.  It is the `attn` provider quip_b200.generate.Generator takes in the CPU tests, in the way
oracle/glue.py's TorchGlue stands in for fused.CudaGlue; the product never imports it.
"""
import torch


class TorchDecodeAttention:
    def __call__(self, q, k_new, v_new, k_cache, v_cache, pos, scale):
        """q (B, nh*hd), k_new / v_new (B, nkv*hd); k_cache / v_cache (B, nkv, max_len, hd), updated in place; pos (B,)
        int.  Returns out (B, nh*hd) in q's dtype."""
        B, nkv, max_len, hd = k_cache.shape
        nh = q.shape[-1] // hd
        rows = torch.arange(B, device=q.device)
        pos = pos.long()
        k_cache[rows, :, pos] = k_new.reshape(B, nkv, hd).to(k_cache.dtype)
        v_cache[rows, :, pos] = v_new.reshape(B, nkv, hd).to(v_cache.dtype)
        acc = torch.float64 if q.dtype == torch.float64 else torch.float32
        qh = q.reshape(B, nkv, nh // nkv, hd).to(acc)
        s = scale * (qh @ k_cache.to(acc).transpose(-1, -2))                          # (B, nkv, G, max_len)
        valid = torch.arange(max_len, device=q.device)[None, :] <= pos[:, None]         # (B, max_len)
        s = s.masked_fill(~valid[:, None, None, :], float('-inf'))
        o = torch.softmax(s, dim=-1) @ v_cache.to(acc)                                   # (B, nkv, G, hd)
        return o.reshape(B, nh * hd).to(q.dtype)
