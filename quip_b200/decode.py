"""Token-by-token decode of a packed Llama or OPT model from one CUDA graph.

The reference's `benchmark()` (opt.py:431-482, llama.py via the same code) times an eager HF forward per
token with a growing KV cache; with the few-token kernels of this package one token's GPU work is a few
milliseconds while the eager Python path around it costs more than that in launch overhead.  `GraphDecoder`
is the same computation with everything a CUDA graph needs made static:

  * a KV cache of fixed length `max_len` per layer, written at the current position with `index_copy_`;
  * the position as a device tensor (advanced inside the graph), rotary cos/sin gathered from a table;
  * attention over the whole cache under a mask `arange(max_len) <= position`.

The decoder layers' own modules are reused (input_layernorm, the seven QuantLinear / nn.Linear projections,
post_attention_layernorm, final norm, lm_head): same weights, same kernels as `model(...)`; only the glue
between them is restated.  Llama (MHA or GQA; torch glue or the kernels of csrc/glue.cu) and OPT (the model benchmark() is
written for, opt.py:431-482: learned positions, LayerNorm with bias, ReLU MLP; torch glue).
"""
import math

import torch
import torch.nn.functional as F


def _rotate_half(x):
    h = x.shape[-1] // 2
    return torch.cat((-x[..., h:], x[..., :h]), dim=-1)


class GraphDecoder:
    def __init__(self, model, max_len=256, batch=1, ops=None, layer_range=None, first=True, last=True):
        """ops: provider of the fused glue kernels (quip_b200.fused.CudaGlue; picked up automatically when
        QUIP_FUSED_LAYER=1 on a CUDA device), None for the torch glue.

        layer_range=(lo, hi), first, last: one STAGE of a layer pipeline (the reference's opt_multigpu / llama_multigpu
        placement, opt.py:384-428) -- decoder layers lo..hi-1 with their own KV cache; a stage that is not the first reads
        the hidden state of the token from `h_in`, one that is not the last leaves it in `h_out` (static buffers, so the
        stage is still one graph); quip_b200.pipeline.PipelinedDecoder moves them between ranks."""
        cfg = model.config
        assert cfg.model_type in ('llama', 'opt'), 'GraphDecoder covers the Llama and OPT families'
        self.family = cfg.model_type
        self.model, self.max_len, self.batch = model, int(max_len), int(batch)
        self.dev = next(iter(model.parameters())).device
        self.nh = cfg.num_attention_heads
        dt = model.get_input_embeddings().weight.dtype     # fp16 on the GPU path; fp32 in the CPU tests
        self.first, self.last = bool(first), bool(last)
        if self.family == 'llama':
            self.layers = list(model.model.layers)
            self.nkv = getattr(cfg, 'num_key_value_heads', None) or self.nh
            self.hd = getattr(cfg, 'head_dim', None) or cfg.hidden_size // self.nh
            # rotary table with the model's own module (HF default rope: positions 0 .. max_len-1)
            pos = torch.arange(self.max_len, device=self.dev)[None, :]
            with torch.no_grad():
                cos, sin = model.model.rotary_emb(torch.zeros(1, 1, cfg.hidden_size, device=self.dev, dtype=dt), pos)
            self.cos, self.sin = cos[0].to(dt).contiguous(), sin[0].to(dt).contiguous()        # (max_len, head_dim)
        else:
            dec = model.model.decoder
            assert self.max_len <= cfg.max_position_embeddings, 'OPT has learned positions: max_len beyond the table'
            self.layers = list(dec.layers)
            self.nkv = self.nh
            self.hd = cfg.hidden_size // self.nh
        lo, hi = layer_range or (0, len(self.layers))
        assert 0 <= lo < hi <= len(self.layers), (lo, hi)
        self.layers = self.layers[lo:hi]
        L, B = len(self.layers), self.batch
        self.h_in = None if self.first else torch.zeros(B, 1, cfg.hidden_size, dtype=dt, device=self.dev)
        self.h_out = None if self.last else torch.zeros(B, 1, cfg.hidden_size, dtype=dt, device=self.dev)
        self.k_cache = torch.zeros(L, B, self.nkv, self.max_len, self.hd, dtype=dt, device=self.dev)
        self.v_cache = torch.zeros_like(self.k_cache)
        self.position = torch.zeros(1, dtype=torch.long, device=self.dev)
        self.tokens = torch.zeros(B, dtype=torch.long, device=self.dev)
        self.logits = None
        self.graph = None
        self._arange = torch.arange(self.max_len, device=self.dev)
        self._pos_host = 0
        # q/k/v and gate/up read the same input: their chains of few-token kernels run on parallel branches
        self._side = [torch.cuda.Stream(device=self.dev) for _ in range(2)] if self.dev.type == 'cuda' else None
        if self.family != 'llama':
            ops = None                                     # the fused glue kernels are the Llama layer's
        elif ops is None and self.dev.type == 'cuda':
            from . import fused
            if fused.enabled() and getattr(cfg, 'hidden_act', 'silu') == 'silu' and self.hd % 16 == 0:
                ops = fused.CudaGlue()
        self.ops = ops

    def _parallel(self, x, mods):
        """[m(x) for m in mods] with every module after the first on its own stream (graph branches when capturing)."""
        if self._side is None:
            return [m(x) for m in mods]
        main = torch.cuda.current_stream(self.dev)
        outs = [None] * len(mods)
        for i, m in enumerate(mods[1:], 1):
            st = self._side[i - 1]
            st.wait_stream(main)
            with torch.cuda.stream(st):
                outs[i] = m(x)
        outs[0] = mods[0](x)
        for i in range(1, len(mods)):
            main.wait_stream(self._side[i - 1])
        return outs

    def reset(self):
        self._pos_host = 0
        self.position.zero_()
        self.k_cache.zero_()
        self.v_cache.zero_()

    # ---- attention of the step, shared by the three kinds of glue (quip_b200.generate.Generator overrides both)
    def _attn_context(self):
        """What _attend needs of the step's positions, computed once per step: the mask over the static cache."""
        return (self._arange <= self.position)[None, None, None, :]                     # (1, 1, 1, max_len)

    def _attend(self, li, q, k, v, scale, mask):
        """q (B, nh, 1, hd), k, v (B, nkv, 1, hd) of the step: store k, v at the position in layer li's cache and attend over
        the whole cache under the mask.  Returns (B, nh, 1, hd)."""
        pos = self.position
        self.k_cache[li].index_copy_(2, pos, k)
        self.v_cache[li].index_copy_(2, pos, v)
        kk, vv = self.k_cache[li], self.v_cache[li]
        if self.nkv != self.nh:
            kk = kk.repeat_interleave(self.nh // self.nkv, dim=1)
            vv = vv.repeat_interleave(self.nh // self.nkv, dim=1)
        return F.scaled_dot_product_attention(q, kk, vv, attn_mask=mask, scale=scale)

    def _graph_generators(self):
        """Random generators the step draws from, registered with the graph so that each replay advances them."""
        return ()

    # ---- the layers of the stage, three kinds of glue.  Each takes the hidden state entering the stage and returns
    # (h, pend): the residual stream and a branch output still to be added to it (None when already added).

    # csrc/glue.cu: 4 launches per layer instead of ~30 (at one token every torch elementwise op is a launch-latency-bound
    # graph node); the residual add of a branch rides on the next RMSNorm
    def _layers_fused(self, h):
        ops = self.ops
        B, nh, nkv, hd = self.batch, self.nh, self.nkv, self.hd
        pos = self.position
        h = h.contiguous()
        cos = self.cos.index_select(0, pos).expand(B, hd).contiguous()                     # one row per sequence
        sin = self.sin.index_select(0, pos).expand(B, hd).contiguous()
        ctx = self._attn_context()
        pend = None
        for li, layer in enumerate(self.layers):
            a, mlp = layer.self_attn, layer.mlp
            n1, n2 = layer.input_layernorm, layer.post_attention_layernorm
            if pend is None:
                x = ops.rmsnorm(h, n1.weight, n1.variance_epsilon)
            else:
                h, x = ops.rmsnorm(h, n1.weight, n1.variance_epsilon, residual=pend)
            q, k, v = self._parallel(x, [a.q_proj, a.k_proj, a.v_proj])
            ops.rope_(q, k, cos, sin, hd)
            o = self._attend(li, q.view(B, 1, nh, hd).transpose(1, 2), k.view(B, 1, nkv, hd).transpose(1, 2),
                             v.view(B, 1, nkv, hd).transpose(1, 2), 1.0 / math.sqrt(hd), ctx)
            o = o.transpose(1, 2).reshape(B, 1, nh * hd)
            h, x = ops.rmsnorm(h, n2.weight, n2.variance_epsilon, residual=a.o_proj(o))
            gate, up = self._parallel(x, [mlp.gate_proj, mlp.up_proj])
            pend = mlp.down_proj(ops.silu_mul(gate, up))
        return h, pend

    def _layers_llama(self, h):
        B, nh, nkv, hd = self.batch, self.nh, self.nkv, self.hd
        pos = self.position
        cos = self.cos.index_select(0, pos).view(-1, 1, 1, hd)                             # (1 or B, 1, 1, hd)
        sin = self.sin.index_select(0, pos).view(-1, 1, 1, hd)
        ctx = self._attn_context()
        for li, layer in enumerate(self.layers):
            a = layer.self_attn
            x = layer.input_layernorm(h)
            q, k, v = self._parallel(x, [a.q_proj, a.k_proj, a.v_proj])
            q = q.view(B, 1, nh, hd).transpose(1, 2)                                       # (B, nh, 1, hd)
            k = k.view(B, 1, nkv, hd).transpose(1, 2)
            v = v.view(B, 1, nkv, hd).transpose(1, 2)
            q = q * cos + _rotate_half(q) * sin
            k = k * cos + _rotate_half(k) * sin
            o = self._attend(li, q, k, v, 1.0 / math.sqrt(hd), ctx)
            o = o.transpose(1, 2).reshape(B, 1, nh * hd)
            h = h + a.o_proj(o)
            x = layer.post_attention_layernorm(h)
            mlp = layer.mlp
            gate, up = self._parallel(x, [mlp.gate_proj, mlp.up_proj])
            h = h + mlp.down_proj(F.silu(gate) * up)
        return h, None

    # OPT (modeling_opt.OPTDecoderLayer): pre- or post-LayerNorm, q scaled before the dot product, ReLU between fc1 and fc2;
    # biases live inside the (Quant)Linear modules
    def _layers_opt(self, h):
        B, nh, hd = self.batch, self.nh, self.hd
        ctx = self._attn_context()
        for li, layer in enumerate(self.layers):
            a, before = layer.self_attn, layer.do_layer_norm_before
            x = layer.self_attn_layer_norm(h) if before else h
            q, k, v = self._parallel(x, [a.q_proj, a.k_proj, a.v_proj])
            q = (q * a.scaling).view(B, 1, nh, hd).transpose(1, 2)                         # scaled first, as the HF module does
            o = self._attend(li, q, k.view(B, 1, nh, hd).transpose(1, 2), v.view(B, 1, nh, hd).transpose(1, 2), 1.0, ctx)
            h = h + a.out_proj(o.transpose(1, 2).reshape(B, 1, nh * hd))
            if not before:
                h = layer.self_attn_layer_norm(h)
            x = layer.final_layer_norm(h) if before else h
            h = h + layer.fc2(layer.activation_fn(layer.fc1(x)))
            if not before:
                h = layer.final_layer_norm(h)
        return h, None

    def _embed(self):
        """Token (and, for OPT, learned position: index position + 2) embeddings of the step: (B, 1, hidden)."""
        if self.family == 'llama':
            return self.model.model.embed_tokens(self.tokens)[:, None, :]
        d = self.model.model.decoder
        h = d.embed_tokens(self.tokens)[:, None, :]
        if d.project_in is not None:
            h = d.project_in(h)
        return h + F.embedding(self.position + d.embed_positions.offset, d.embed_positions.weight)[:, None]

    def _head(self, h, pend):
        """Final norm (fused with the pending residual add on the glue-kernel path) -> lm_head: logits (B, vocab)."""
        if self.family == 'llama':
            fn = self.model.model.norm
            if self.ops is not None:
                _, h = self.ops.rmsnorm(h, fn.weight, fn.variance_epsilon, residual=pend)
            else:
                h = fn(h)
        else:
            d = self.model.model.decoder
            if d.final_layer_norm is not None:
                h = d.final_layer_norm(h)
            if d.project_out is not None:
                h = d.project_out(h)
        return self.model.lm_head(h)[:, 0, :]

    # one decode step of the stage on the static buffers (what the graph records)
    def _step(self):
        h = self._embed() if self.first else self.h_in
        if self.family == 'opt':
            h, pend = self._layers_opt(h)
        elif self.ops is not None:
            h, pend = self._layers_fused(h)
        else:
            h, pend = self._layers_llama(h)
        if self.last:
            self.logits = self._head(h, pend)
        else:
            self.h_out.copy_(h if pend is None else h + pend)   # fp16 add: the rounding the fused residual add performs
        self.position.add_(1)

    def capture(self):
        """Record one step.  The cache and position are restored afterwards, so capture is side-effect free."""
        from .quant import QuantLinear
        for mod in self.model.modules():                   # sibling groups launch on side streams: not while capturing
            if isinstance(mod, QuantLinear) and getattr(mod, '_group', None) is not None:
                raise RuntimeError('dissolve the sibling groups (quant.SiblingGroup.dissolve) before capturing')
        pos0, k0, v0 = self.position.clone(), self.k_cache.clone(), self.v_cache.clone()
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.no_grad(), torch.cuda.stream(side):
            for _ in range(2):                             # lazy set-up (descriptors, workspaces) outside the graph
                self._step()
            self.position.copy_(pos0)
            self.graph = torch.cuda.CUDAGraph()
            for gen in self._graph_generators():
                self.graph.register_generator_state(gen)
            with torch.cuda.graph(self.graph, stream=side, capture_error_mode='thread_local'):
                self._step()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        self.position.copy_(pos0)
        self.k_cache.copy_(k0)
        self.v_cache.copy_(v0)
        return self

    def step(self, tokens):
        """tokens (B,) -> logits (B, vocab) for the next position; advances the cache."""
        if self._pos_host >= self.max_len:
            raise ValueError(f'KV cache of {self.max_len} positions is full')
        self._pos_host += 1
        self.tokens.copy_(tokens.reshape(-1))
        if self.graph is None:
            with torch.no_grad():
                self._step()
        else:
            self.graph.replay()
        return self.logits


def graph_decode_benchmark(model, input_ids, max_len=None, check=False):
    """`decode_benchmark` (reference benchmark(), opt.py:431-482) through the graph: median seconds per token and,
    with check, the perplexity of the fed sequence."""
    import time

    import numpy as np
    ids = input_ids.reshape(-1).to(next(iter(model.parameters())).device)
    dec = GraphDecoder(model, max_len=max_len or int(ids.numel()), batch=1).capture()
    times, tot = [], 0.0
    for i in range(ids.numel()):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        logits = dec.step(ids[i:i + 1])
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        if check and i != ids.numel() - 1:
            tot += float(F.cross_entropy(logits.float(), ids[i + 1:i + 2]))
    ppl = float(np.exp(tot / (ids.numel() - 1))) if check else None
    return float(np.median(times)), ppl


def graph_decode_throughput(model, batch, steps=32, max_len=64, seed=0):
    """Aggregate tokens/s of `steps` graph-replayed decode steps with `batch` independent sequences (random token ids)."""
    dev = next(iter(model.parameters())).device
    dec = GraphDecoder(model, max_len=max_len, batch=batch).capture()
    gen = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, model.config.vocab_size, (steps + 2, batch), generator=gen).to(dev)
    for i in range(2):
        dec.step(ids[i])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        dec.step(ids[2 + i])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return batch * 1e3 / ms, ms
