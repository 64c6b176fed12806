"""Generation from prompts with a packed Llama or OPT model: the prompt in one pass, new tokens from one CUDA graph.

    from quip_b200.generate import generate
    out = generate(model, [ids_a, ids_b], max_new_tokens=64)          # list of 1-D tensors: prompt + new tokens

  * Prefill.  The prompts are right-padded into (B, P) and run once through the model's many-token path (the HF forward
    of the base model, so the packed linears see B*P tokens); the K / V it produces are copied into the static cache.
    With right padding and the causal mask no real token attends to padding.  The first new token comes from the
    lm_head of each sequence's last real row only.
  * Decode.  `Generator` is `GraphDecoder` (quip_b200/decode.py) with a position per sequence: rotary rows (Llama) or
    learned positions (OPT) are gathered per row, and attention runs through quip_decode_attention, which reads only the
    cache rows 0 .. pos[b] of each sequence and reads a GQA KV head once for its group of query heads.  The token is
    chosen on the device (greedy, or temperature / top-k / top-p sampling from a seeded generator), written to the
    step's input and to the output buffer, rows that produced eos_token_id keep emitting it, and the positions advance:
    the whole step is one graph, T new tokens are T replays.  The host synchronises only to ask whether every row has
    finished, every `check_every` steps.

`attn` is the provider of the attention step: `CudaDecodeAttention` (the C ABI, CUDA only) or, in the CPU tests, the
torch restatement under oracle/ -- which this module never imports.
"""

import torch

from . import _lib
from .decode import GraphDecoder


class CudaDecodeAttention:
    """quip_decode_attention of the C ABI on torch tensors (fp16, CUDA).  The fp32 workspace of the split partials is
    allocated on the first call and reused (it is the same for every layer of a model)."""

    def __init__(self):
        self._ws = None

    def __call__(self, q, k_new, v_new, k_cache, v_cache, pos, scale):
        """q (B, nh*hd), k_new / v_new (B, nkv*hd); k_cache / v_cache (B, nkv, max_len, hd), updated at pos; pos (B,)
        int32.  Returns out (B, nh*hd)."""
        for t in (q, k_new, v_new, k_cache, v_cache, pos):
            if not t.is_cuda:
                raise RuntimeError('quip_decode_attention runs on a CUDA device only (there is no CPU fallback)')
        if any(t.dtype != torch.float16 for t in (q, k_new, v_new, k_cache, v_cache)) or pos.dtype != torch.int32:
            raise ValueError('quip_decode_attention takes fp16 q / k / v / caches and int32 positions')
        if not (k_cache.is_contiguous() and v_cache.is_contiguous() and pos.is_contiguous()):
            raise ValueError('quip_decode_attention takes contiguous caches and positions')
        q, k_new, v_new = q.contiguous(), k_new.contiguous(), v_new.contiguous()
        B, nkv, max_len, hd = k_cache.shape
        nh = q.shape[-1] // hd
        lib = _lib.load()
        need = _lib.C.c_size_t(0)
        _lib.check(lib.quip_decode_attention_workspace_bytes(B, nh, max_len, hd, _lib.C.byref(need)))
        if self._ws is None or self._ws.numel() < need.value or self._ws.device != q.device:
            self._ws = torch.empty(need.value, dtype=torch.uint8, device=q.device)
        out = torch.empty_like(q)
        with torch.cuda.device(q.device):
            _lib.check(lib.quip_decode_attention(q.data_ptr(), k_new.data_ptr(), v_new.data_ptr(), k_cache.data_ptr(),
                                                 v_cache.data_ptr(), pos.data_ptr(), B, nh, nkv, max_len, hd,
                                                 _lib.C.c_float(scale), out.data_ptr(), self._ws.data_ptr(),
                                                 self._ws.numel(), torch.cuda.current_stream(q.device).cuda_stream))
        return out


def select_tokens(logits, do_sample=False, temperature=1.0, top_k=0, top_p=1.0, generator=None):
    """logits (B, vocab) -> token ids (B,) on the device, without a host synchronisation (so a graph can record it).
    Greedy: argmax.  Sampling: logits / temperature, keep the top_k largest (0: all), then the smallest set of the most
    likely tokens whose probability reaches top_p (the most likely always stays), and draw from the renormalised
    softmax with `generator` (argmax of p / E with E ~ Exp(1): an exact draw from p)."""
    x = logits.float()
    if not do_sample:
        return x.argmax(-1)
    x = x / temperature
    if top_k > 0:
        kth = x.topk(min(top_k, x.shape[-1]), dim=-1).values[:, -1:]
        x = x.masked_fill(x < kth, float('-inf'))
    if top_p < 1.0:
        sx, si = x.sort(dim=-1, descending=True)
        p = sx.softmax(-1)
        drop = (p.cumsum(-1) - p) >= top_p                 # the mass before a token already reaches top_p
        x = x.scatter(-1, si, sx.masked_fill(drop, float('-inf')))
    p = x.softmax(-1)
    e = torch.empty_like(p).exponential_(generator=generator).clamp_min_(torch.finfo(torch.float32).tiny)
    return (p / e).argmax(-1)


class Generator(GraphDecoder):
    """GraphDecoder over B sequences of their own lengths, with prefill and on-device token selection (module doc)."""

    def __init__(self, model, batch, max_len, attn=None, ops=None, do_sample=False, temperature=1.0, top_k=0,
                 top_p=1.0, eos_token_id=None):
        """attn: the attention provider (CudaDecodeAttention on a CUDA device when None; no CPU fallback).  ops: the glue
        provider, as for GraphDecoder."""
        super().__init__(model, max_len=max_len, batch=batch, ops=ops)
        if attn is None:
            if self.dev.type != 'cuda':
                raise RuntimeError('Generator: quip_decode_attention needs a CUDA device (there is no CPU fallback); '
                                   'pass attn= to run elsewhere')
            attn = CudaDecodeAttention()
        self.attn = attn
        if do_sample and not temperature > 0:
            raise ValueError('temperature must be positive when sampling')
        self.sampling = dict(do_sample=bool(do_sample), temperature=float(temperature), top_k=int(top_k),
                             top_p=float(top_p))
        self.eos = eos_token_id
        B = self.batch
        self.position = torch.zeros(B, dtype=torch.long, device=self.dev)           # per sequence
        self.finished = torch.zeros(B, dtype=torch.bool, device=self.dev)
        self.out = torch.zeros(B, self.max_len, dtype=torch.long, device=self.dev)   # new tokens, column t per step
        self.t = torch.zeros(1, dtype=torch.long, device=self.dev)
        self.rng = torch.Generator(device=self.dev)
        self.lens = None

    # ---- GraphDecoder's attention of the step, through quip_decode_attention with a position per row
    def _attn_context(self):
        return self.position.to(torch.int32)

    def _attend(self, li, q, k, v, scale, pos32):
        B = self.batch
        o = self.attn(q.transpose(1, 2).reshape(B, -1), k.transpose(1, 2).reshape(B, -1),
                      v.transpose(1, 2).reshape(B, -1), self.k_cache[li], self.v_cache[li], pos32, scale)
        return o.view(B, 1, self.nh, self.hd).transpose(1, 2)

    def _graph_generators(self):
        return (self.rng,) if self.sampling['do_sample'] else ()

    def _take(self, logits):
        """Choose the next token of every row from logits (B, vocab); finished rows repeat eos_token_id."""
        tok = select_tokens(logits, generator=self.rng, **self.sampling)
        if self.eos is not None:
            tok = tok.masked_fill(self.finished, self.eos)
            self.finished |= tok == self.eos
        self.tokens.copy_(tok)
        self.out.index_copy_(1, self.t, tok[:, None])
        self.t.add_(1)

    def _step(self):
        super()._step()
        self._take(self.logits)

    def capture(self):
        """Record one step (prefill is not part of it).  Every buffer the step writes is restored afterwards."""
        saved = [t.clone() for t in (self.tokens, self.finished, self.out, self.t)]
        super().capture()
        for t, s in zip((self.tokens, self.finished, self.out, self.t), saved):
            t.copy_(s)
        return self

    def prefill(self, prompts):
        """prompts: B 1-D id tensors.  Runs them in one pass, fills the cache, chooses the first new token.  Returns the
        logits of each sequence's last prompt token (B, vocab)."""
        B = self.batch
        if len(prompts) != B:
            raise ValueError(f'{len(prompts)} prompts for a batch of {B}')
        lens = [int(p.numel()) for p in prompts]
        if min(lens) < 1:
            raise ValueError('empty prompt')
        P = max(lens)
        if P > self.max_len:
            raise ValueError(f'a prompt of {P} tokens does not fit a KV cache of {self.max_len} positions')
        ids = torch.zeros(B, P, dtype=torch.long, device=self.dev)
        for b, p in enumerate(prompts):
            ids[b, :lens[b]] = p.reshape(-1).to(self.dev)
        lens_d = torch.tensor(lens, device=self.dev)
        mask = (torch.arange(P, device=self.dev)[None, :] < lens_d[:, None]).long()
        with torch.no_grad():
            out = self.model.model(input_ids=ids, attention_mask=mask, use_cache=True)
            for li, layer in enumerate(out.past_key_values.layers):
                self.k_cache[li, :, :, :P].copy_(layer.keys)
                self.v_cache[li, :, :, :P].copy_(layer.values)
            h = out.last_hidden_state[torch.arange(B, device=self.dev), lens_d - 1]          # last real row only
            logits = self.model.lm_head(h)
            self.position.copy_(lens_d)
            self.finished.zero_()
            self.t.zero_()
            self._take(logits)
        self._pos_host = P
        self.lens = lens
        return logits

    def step(self, tokens=None):
        """One decode step (a graph replay once captured): feeds `tokens` (B,) when given (teacher forcing), else the
        tokens chosen by the previous step.  Returns the logits (B, vocab) of the fed tokens."""
        if tokens is not None:
            tokens = tokens.reshape(-1)
        return super().step(self.tokens if tokens is None else tokens)

    def new_tokens(self):
        """The tokens chosen so far, (B, n)."""
        return self.out[:, :int(self.t)]


def generate(model, prompts, max_new_tokens, do_sample=False, temperature=1.0, top_k=0, top_p=1.0, seed=0,
             eos_token_id=None, max_len=None, attn=None, ops=None, graph=None, check_every=8):
    """Prompt + up to max_new_tokens new tokens for each prompt (a list of 1-D id tensors), as a list of 1-D tensors.
    Rows that emit eos_token_id continue with it until every row has (then generation stops).  max_len: positions of
    the static cache (default: the longest prompt + max_new_tokens).  graph: replay one CUDA graph per step (default:
    on a CUDA device).  attn / ops: providers of the attention step and of the Llama glue (Generator)."""
    lens = [int(p.numel()) for p in prompts]
    if max_new_tokens < 1:
        return [p.reshape(-1).clone() for p in prompts]
    need = max(lens) + max_new_tokens - 1                  # positions written: the prompt, then every fed new token
    max_len = int(max_len) if max_len is not None else need
    if need > max_len:
        raise ValueError(f'{max(lens)} prompt tokens + {max_new_tokens} new tokens need a KV cache of {need} positions, '
                         f'max_len is {max_len}')
    gen = Generator(model, len(prompts), max_len, attn=attn, ops=ops, do_sample=do_sample, temperature=temperature,
                    top_k=top_k, top_p=top_p, eos_token_id=eos_token_id)
    if graph is None:
        graph = gen.dev.type == 'cuda'
    if graph:
        gen.capture()
    gen.rng.manual_seed(seed)
    gen.prefill(prompts)
    for i in range(1, max_new_tokens):
        if eos_token_id is not None and i % check_every == 0 and bool(gen.finished.all()):
            break
        gen.step()
    new = gen.new_tokens().cpu()
    return [torch.cat((p.reshape(-1).cpu(), new[b])) for b, p in enumerate(prompts)]
