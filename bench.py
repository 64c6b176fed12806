"""bench.py -- tokens/s of the packed 2-bit Llama-2-7B eval path on N B200s (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    ... bench.py --model llama70b|opt30b|opt1.3b [--parallelism pp]     the other BASELINE.json configs (not the headline)

Workload (BASELINE.json configs[2], the config `metric` is quoted on): Llama-2-7B architecture, every
decoder Linear a 2-bit packed QuantLinear with the as-run blocked incoherence butterflies + rescale
(`--incoh_processing`), synthetic 2048-token samples, random-init weights / random codes (no network).
A *step* = one 2048-token sample through the per-layer eval path (embed -> 32 decoder layers, 7 packed
linears each -> final norm -> lm_head -> CE loss), i.e. one pass of llama_eval's inner loop.

  value   whole-job tokens/s with token ids already resident in HBM (CUDA events, barrier + sync on both
          sides, max over ranks).  Data parallel over samples: each rank runs K steps (weak scaling); the
          path's only collective, one all-reduce of the summed NLL, is inside the timed region.
  e2e     the same metric through the public API quip_b200.llama.llama_eval with HOST token ids: every step
          copies its ids from pinned host memory and reads the scalar result back.
  roofline  the dominant kernel (tcgen05 packed GEMM): algorithmic flops of its launches / their summed
          device time, measured with CUDA events around every launch inside the timed region.
  config.glue  which glue ran between the packed linears (HF torch launches or the fused kernels of csrc/glue.cu), chosen
          in the run by `pick_glue`: every fused op against the HF module it replaces (bit-exact except the norm's summation
          order), two real layers both ways judged against a control (the HF layers with one-ulp flips in their own norm
          outputs -- a random-init transformer amplifies rounding noise), fused only if also faster; then the whole-model NLL
          of the step to be timed is compared with the HF-glue value.
  decode  extras, N=1 only: the 224 QuantLinear calls of one token from a CUDA graph, the packed contraction alone in
          steady state against the HBM peak, eager HF decode, graph decode and its batch sweep.
  selfcheck  outputs of packed linears of the timed model (layer 0: q_proj, down_proj) on a real sample against the fp32 torch
          restatement of the pipeline (quip_b200/selfcheck.py), relative error; the run aborts above 1e-3.
  --parallelism pp  the layer pipeline (BASELINE configs[3], [4]): contiguous layer ranges per rank (opt.py:424-426), one
          CUDA-graph replay per stage per sample, NCCL send/recv of the hidden states on per-link communicators; a step is
          one sample through all stages, `pipeline` reports the stage times and the fill/drain bubble.
  cpu_baseline / --impl reference: the reference's effective path (HF decoder layer with dense fp16
          weights, the per-layer loop of llama.py:174-253 ported in oracle/evalloop.py) on the host cores,
          on a bounded sample (1 decoder layer x 1 sample), extrapolated to 32 layers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEQ = 2048
N_LAYERS = 32


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tflops_burst=d['bf16_tflops'], tflops_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe: -lms 200).  The process is
    started BEFORE the warm-up steps -- nvidia-smi's own start-up (NVML init under the driver lock) slowed the first
    timed steps by ~25 % whenever it coincided with them -- and only the rows that arrive between mark_start() and
    mark_end() are summarised."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.all_rows, self.t0, self.t1 = [], None, None

    def mark_start(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.all_rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()        # exact PID we started
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = (self.t1 if self.t1 is not None else time.perf_counter()) + 0.25
        self.rows = [r for (ts, r) in self.all_rows if t0 <= ts <= t1] or [r for (_, r) in self.all_rows[-2:]]
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith('active') for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=float(self.rows[0][1]), reasons=reasons, samples=len(sm),
                    power_w_max=max(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace('.', '').isdigit()))


def decode_leg(model, dev, pk):
    """One token through every QuantLinear of the model (7 per decoder layer, every layer its own weights, so the
    packed words and factors come from HBM), replayed from one CUDA graph: the few-token kernels of the path
    (qgemv int8 tensor-core GEMV, few-token passes, programmatic dependent launch) against the HBM roofline of the
    bytes they must read.  Attention, norms and the KV cache are not part of this leg."""
    from quip_b200.quant import QuantLinear
    layers = model.model.layers
    names = ('self_attn.q_proj', 'self_attn.k_proj', 'self_attn.v_proj', 'self_attn.o_proj', 'mlp.gate_proj',
             'mlp.up_proj', 'mlp.down_proj')

    def get(layer, name):
        m = layer
        for part in name.split('.'):
            m = getattr(m, part)
        return m
    mods = [[get(l, n) for n in names] for l in layers]
    assert all(isinstance(m, QuantLinear) for row in mods for m in row)
    nbytes = 0
    for row in mods:
        for m in row:
            for bname, buf in m.named_buffers():
                if bname not in ('meta',):
                    nbytes += buf.numel() * buf.element_size()
    x = torch.randn(1, mods[0][0].infeatures, device=dev).half()
    sides = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def fan(h, members):
        """Sibling linears read the same input: independent chains, one graph branch each (as GraphDecoder runs them)."""
        main = torch.cuda.current_stream(dev)
        outs = [None] * len(members)
        for i, m in enumerate(members[1:], 1):
            sides[i - 1].wait_stream(main)
            with torch.cuda.stream(sides[i - 1]):
                outs[i] = m._forward_impl(h)
        outs[0] = members[0]._forward_impl(h)
        for i in range(1, len(members)):
            main.wait_stream(sides[i - 1])
        return outs

    def step_serial():
        h = x
        for q, k, v, o, g, u, d in mods:
            a = q._forward_impl(h); k._forward_impl(h); v._forward_impl(h)
            h2 = o._forward_impl(a)
            gg = g._forward_impl(h2); u._forward_impl(h2)
            h = d._forward_impl(gg)
        return h

    def step_branches():
        h = x
        for q, k, v, o, g, u, d in mods:
            a = fan(h, [q, k, v])[0]
            h2 = o._forward_impl(a)
            gg = fan(h2, [g, u])[0]
            h = d._forward_impl(gg)
        return h

    def replay_ms(step):
        with torch.no_grad():
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side, capture_error_mode='thread_local'):
                    step()
            torch.cuda.current_stream().wait_stream(side)
            graph.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for _ in range(reps):
                graph.replay()
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    ms_serial = replay_ms(step_serial)
    ms = replay_ms(step_branches)
    gbs = nbytes / (ms / 1e3) / 1e9
    return dict(tokens=1, what='all %d QuantLinear.forward calls of one decode step from one CUDA graph: q/k/v and gate/up of a '
                               'layer on parallel graph branches (they read the same input), the four groups of a layer and '
                               'the layers in sequence; no attention / KV cache' % (len(mods) * 7),
                ms_per_token_linears=ms, tokens_per_s_linears=1e3 / ms, bytes_per_token=nbytes, achieved_gbs=gbs,
                hbm_peak_gbs=pk['hbm_gbs'], hbm_frac=gbs / pk['hbm_gbs'],
                ms_per_token_linears_fully_serial=ms_serial, hbm_frac_fully_serial=nbytes / (ms_serial / 1e3) / 1e9 / pk['hbm_gbs'],
                roofline_tokens_per_s=pk['hbm_gbs'] * 1e9 / nbytes)


def contraction_leg(dev, pk):
    """The packed contraction alone in steady state: one token (and two) against the 2-bit gate/up/down-sized matrices of
    all 32 layers stacked into one (352256 x 4096) matrix, so the launch ramp is amortised and every packed word comes from
    HBM (360 MB per matrix, two matrices alternated).  Algorithmic bytes = packed codes + fp16 activations in and out
    (SURVEY section 8d B_codes); this is the figure the north star's ">= 70 % of the HBM roofline" refers to."""
    from quip_b200 import _lib
    from quip_b200.quant import packed_words
    lib = _lib.load()
    N, K, bits, copies = 32 * 11008, 4096, 2, 2
    qw = torch.randint(-2 ** 31, 2 ** 31 - 1, (copies, packed_words(N, K, bits)), dtype=torch.int32, device=dev)
    sc = torch.full((N,), 0.01, device=dev)
    ze = sc * 1.5
    res = {}
    for M in (1, 2):
        x = torch.randn(M, K, device=dev).half()
        z = torch.empty(M, N, dtype=torch.float16, device=dev)
        descs = []
        for c in range(copies):
            d = _lib.QuipLinearDesc()
            d.K, d.N, d.bits, d.flags = K, N, bits, _lib.QUIP_FLAG_SYMMETRIC
            d.qweight, d.scales, d.zeros = qw[c].data_ptr(), sc.data_ptr(), ze.data_ptr()
            descs.append(d)
        need = C.c_size_t()
        _lib.check(lib.quip_qlinear_workspace_bytes(C.byref(descs[0]), M, C.byref(need)))
        ws = torch.zeros(max(need.value, 1 << 20), dtype=torch.uint8, device=dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def run(i):
            _lib.check(lib.quip_qgemm(C.byref(descs[i % copies]), _lib.ptr(x), None, None, _lib.ptr(z), M, 1,
                                      _lib.ptr(ws), ws.numel(), st))
        for i in range(4):
            run(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for i in range(reps):
            run(i)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / reps * 1e3
        nbytes = N * K * bits / 8 + 2 * M * K + 2 * M * N
        res[str(M)] = dict(us=us, gbs=nbytes / us / 1e3, hbm_frac=nbytes / us / 1e3 / pk['hbm_gbs'])
    return dict(what='quip_qgemm, 2-bit, (352256 x 4096) stacked matrix, tokens -> {us, GB/s of codes + activations, fraction of '
                     'the measured HBM peak}', kernel='qgemv_i8_stream_kernel (int8 tensor-core GEMV, three-limb tokens)', tokens=res)


def _device_ms(fn, reps, warm):
    """Average device milliseconds of fn() over `reps` calls (CUDA events on the current stream)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _replay_ms(fn, reps=3):
    """Device milliseconds of fn() replayed from a CUDA graph: what the timed step does, and independent of the host (eager
    launches of several ranks on a host with few cores are host-bound, which says nothing about the kernels).  Falls back to
    eager timing when the capture fails."""
    try:
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side, capture_error_mode='thread_local'):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    except Exception:
        torch.cuda.synchronize()
        return _device_ms(fn, reps=reps, warm=2)


def _ulp_flip_hooks(mods, rate, seed=0):
    """Forward hooks that move a random fraction `rate` of each module's fp16 outputs by one ulp: the control of pick_glue."""
    gens = {}

    def fn(m, inp, out):
        gen = gens.get(out.device)
        if gen is None:
            gen = gens[out.device] = torch.Generator(device=out.device).manual_seed(seed)
        it, expmask, absmask = ((torch.int16, 0x7C00, 0x7FFF) if out.dtype == torch.float16 else (torch.int32, 0x7F800000, 0x7FFFFFFF))
        if out.dtype not in (torch.float16, torch.float32):
            return out
        bits = out.contiguous().view(it)
        mask = torch.rand(bits.shape, device=out.device, generator=gen) < rate
        finite = (bits & expmask) != expmask
        step = torch.where(torch.rand(bits.shape, device=out.device, generator=gen) < 0.5, 1, -1).to(it)
        return torch.where(mask & finite & ((bits & absmask) > 1), bits + step, bits).view(out.dtype).view(out.shape)
    return [m.register_forward_hook(fn) for m in mods]


def pick_glue(model, prime):
    """Which glue runs between the packed linears of a decoder layer in this run: the HF modules' own torch launches, or the
    fused kernels of csrc/glue.cu (quip_b200/fused.py).  QUIP_FUSED_LAYER=0/1 forces one; otherwise the fused stack must
    pass, on this model and one real sample:
      ops      every fused op against the HF module / function it replaces, on the real tensors of layer 0: rotary, SiLU*up
               and the residual add bit-exact; RMSNorm within one fp16 ulp on < 1e-3 of the positions (the fp32 mean is
               summed in a different order -- the only arithmetic difference between the two glues);
      stack    the first two decoder layers both ways, relative difference of the hidden states;
      control  the HF layers against THEMSELVES with one-ulp flips injected into their norm outputs at the rate measured
               under `ops`.  A random-init transformer amplifies such flips (peaked softmax: logits of standard deviation
               ~5), so the stack difference is judged against this control (<= 3x, or < 1e-3 outright), not in absolute
               terms: the kernels cannot be closer to the HF layers than the HF layers are to their own rounding noise;
      speed    the fused stack must be faster.
    Later the whole-model NLL of the step to be timed is compared with the HF-glue value (main).  Returns a dict for the
    JSON line; sets QUIP_FUSED_LAYER for the rest of the process."""
    from quip_b200 import evalloop, fused
    forced = os.environ.get('QUIP_FUSED_LAYER')
    if forced is not None:
        return dict(mode='fused' if forced == '1' else 'hf', chosen_by='QUIP_FUSED_LAYER=' + forced)
    info = dict(mode='hf', chosen_by='in-run check')
    try:
        with torch.no_grad():
            h, kw = evalloop.layer_inputs(model, evalloop.LLAMA, prime)
            if not fused.supports(model, h, kw):
                info['why'] = 'model not supported by the fused stack'
                return info
            layers = list(model.model.layers)[:2]
            glue = fused.CudaGlue()
            L, S = layers[0], h.shape[1]
            att, mlp = L.self_attn, L.mlp
            hd = att.head_dim

            def diff(a, b):
                d = (a.view(torch.int16).int() - b.view(torch.int16).int()).abs()      # same-sign neighbours differ by 1
                return dict(frac_differ=float((d != 0).float().mean()), max_ulps=int(d.max()))
            ops = {}
            hc = h.contiguous()
            x_hf = L.input_layernorm(hc)
            ops['rmsnorm'] = diff(glue.rmsnorm(hc, L.input_layernorm.weight, L.input_layernorm.variance_epsilon), x_hf)
            q, k = att.q_proj(x_hf), att.k_proj(x_hf)
            cos, sin = kw['position_embeddings']
            from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
            nq, nkv = q.shape[-1] // hd, k.shape[-1] // hd
            q_hf, k_hf = apply_rotary_pos_emb(q.view(1, S, nq, hd).transpose(1, 2), k.view(1, S, nkv, hd).transpose(1, 2), cos, sin)
            q2, k2 = q.clone(), k.clone()
            glue.rope_(q2, k2, cos[0].contiguous(), sin[0].contiguous(), hd)
            ops['rope_q'] = diff(q2, q_hf.transpose(1, 2).reshape(q.shape).contiguous())
            ops['rope_k'] = diff(k2, k_hf.transpose(1, 2).reshape(k.shape).contiguous())
            g, u = mlp.gate_proj(x_hf), mlp.up_proj(x_hf)
            ops['silu_mul'] = diff(glue.silu_mul(g, u), (mlp.act_fn(g) * u).contiguous())
            n2 = L.post_attention_layernorm
            s_f, y_f = glue.rmsnorm(hc, n2.weight, n2.variance_epsilon, residual=q)
            ops['residual_add'] = diff(s_f, (hc + q).contiguous())
            ops['add_rmsnorm'] = diff(y_f, n2(hc + q))
            exact = all(ops[n]['max_ulps'] == 0 for n in ('rope_q', 'rope_k', 'silu_mul', 'residual_add'))
            norm_ok = all(ops[n]['max_ulps'] <= 1 and ops[n]['frac_differ'] < 1e-3 for n in ('rmsnorm', 'add_rmsnorm'))
            info['ops'] = ops

            def hf():
                r = h
                for layer in layers:
                    r = evalloop._call_layer(layer, r, kw)
                return r

            def fu():
                return fused.llama_stack(layers, h.clone(), kw)

            ref, got = hf().float(), fu().float()
            err = float((got - ref).norm() / ref.norm())
            rate = max(ops['rmsnorm']['frac_differ'], ops['add_rmsnorm']['frac_differ'], 1e-6)
            norms = [m for layer in layers for m in (layer.input_layernorm, layer.post_attention_layernorm)]
            ctrl = []
            for seed in range(3):
                hooks = _ulp_flip_hooks(norms, rate, seed)
                try:
                    ctrl.append(float((hf().float() - ref).norm() / ref.norm()))
                finally:
                    for hk in hooks:
                        hk.remove()
            control = sorted(ctrl)[1]
            timer = _replay_ms if h.is_cuda else (lambda fn: _device_ms(fn, reps=3, warm=2))
            times = {name: timer(fn) / len(layers) for name, fn in (('hf', hf), ('fused', fu))}
            info.update(rel_err_vs_hf_layers=err, control_rel_err_hf_vs_hf_with_ulp_flips=control, control_runs=ctrl,
                        control_flip_rate=rate, ms_per_layer_hf=times['hf'], ms_per_layer_fused=times['fused'],
                        note='CUDA-graph replays (device time), first two decoder layers, one 2048-token sample; control = the HF layers with '
                             'one-ulp flips in their norm outputs at the measured rate (median of 3 seeds)')
            stack_ok = err < 1e-3 or err <= 3.0 * control
            if exact and norm_ok and stack_ok and times['fused'] < times['hf']:
                info['mode'] = 'fused'
            else:
                info['why'] = f'exact ops {exact}, norms {norm_ok}, stack {stack_ok}, faster {times["fused"] < times["hf"]}'
    except Exception as e:                                  # any failure keeps the HF glue
        info['why'] = repr(e)[:200]
    os.environ['QUIP_FUSED_LAYER'] = '1' if info['mode'] == 'fused' else '0'
    return info


def decode_glue_ok(model, dev):
    """The decode step with the fused glue (GraphDecoder._layers_fused) against the torch-glue step on the same model: eight
    tokens, two sequences.  As in pick_glue the two differ only by one-ulp flips of the norm outputs, which 32 random-init
    layers amplify; the logits difference is therefore judged against a control -- the torch-glue step against itself with
    such flips injected at the measured rate (<= 3x the control, or < 2e-3 outright)."""
    from quip_b200.decode import GraphDecoder
    from quip_b200.fused import CudaGlue
    ids = torch.randint(0, model.config.vocab_size, (8, 2), generator=torch.Generator().manual_seed(7)).to(dev)
    norms = [m for layer in model.model.layers for m in (layer.input_layernorm, layer.post_attention_layernorm)] + [model.model.norm]
    with torch.no_grad():
        os.environ['QUIP_FUSED_LAYER'] = '0'
        plain = GraphDecoder(model, max_len=16, batch=2)
        fusedd = GraphDecoder(model, max_len=16, batch=2, ops=CudaGlue())
        ctrl = GraphDecoder(model, max_len=16, batch=2)
        worst = control = 0.0
        for i in range(ids.shape[0]):
            a, b = plain.step(ids[i]).float(), fusedd.step(ids[i]).float()
            hooks = _ulp_flip_hooks(norms, 3e-5, seed=i)
            try:
                c = ctrl.step(ids[i]).float()
            finally:
                for hk in hooks:
                    hk.remove()
            worst = max(worst, float((a - b).norm() / a.norm()))
            control = max(control, float((a - c).norm() / a.norm()))
    return (worst < 2e-3 or worst <= 3.0 * control), worst, control


_CPU_THREADS = None


def cpu_threads():
    """One thread-count policy for both places the CPU path is timed (--impl reference and the cpu_baseline leg): the count,
    among 8 / 16 / 32 / 64 / all usable cores, at which the host's fp16 GEMM of a layer's shape runs fastest (on a 128-core
    host all cores are 7x SLOWER than 16: the policy is "the fastest the CPU path can be made", not "as many as exist")."""
    global _CPU_THREADS
    if _CPU_THREADS is None:
        ncpu = os.cpu_count() or 1
        try:
            ncpu = len(os.sched_getaffinity(0))
        except Exception:
            pass
        probe_x, probe_w = torch.randn(SEQ, 4096).half(), torch.randn(4096, 4096).half()
        best = (float('inf'), ncpu)
        for nt in sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)}):
            torch.set_num_threads(nt)
            torch.nn.functional.linear(probe_x, probe_w)
            dt = float('inf')
            for _ in range(5):                                  # best of five: one timing is too noisy to choose by
                t0 = time.perf_counter()
                torch.nn.functional.linear(probe_x, probe_w)
                dt = min(dt, time.perf_counter() - t0)
            if dt < 0.9 * best[0]:                              # more threads only for a clear (> 10 %) gain
                best = (dt, nt)
        _CPU_THREADS = best[1]
    return _CPU_THREADS


def cpu_reference_arm(steps, warmup, model_name='llama7b'):
    """The reference's own implementation of the path on the host cores: dense fp16 decoder layer through
    the reference loop (oracle/evalloop.py).  Bounded sample: ONE decoder layer x ONE 2048-token sample per
    step; tokens/s extrapolated to the whole stack (attention, norms and MLP included; embedding and
    lm_head excluded, as they are not on the quantized path).  Returns value, seconds per layer, cores, a description and
    the number of steps / seconds actually timed."""
    from oracle.evalloop import reference_eval
    from quip_b200.synth import MODELS, model_config
    cores = cpu_threads()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    family = MODELS[model_name][0]
    full = model_config(model_name)
    n_layers = full.num_hidden_layers
    cfg = model_config(model_name, num_hidden_layers=1)
    if family == 'llama':
        from quip_b200.llama import get_llama
        model = get_llama(cfg, seqlen=SEQ)
    else:
        from quip_b200.opt import get_opt
        model = get_opt(cfg)
        model.seqlen = SEQ
    ids = torch.randint(0, cfg.vocab_size, (1, SEQ), generator=torch.Generator().manual_seed(0))
    times = []
    for i in range(warmup + steps):
        timing = {}
        reference_eval(model, ids, nlayers=1, timing=timing)
        if i >= warmup:
            times.append(timing['layer_loop_s'])
    per_layer = sum(times) / len(times)
    value = SEQ / (per_layer * n_layers)
    sample = (f'1 decoder layer x 1 sample of {SEQ} tokens per step (dense fp16 nn.Linear on CPU, {cores} threads), '
              f'{per_layer:.3f} s/layer, extrapolated x{n_layers} layers; {len(times)} steps timed ({sum(times):.2f} s)')
    return value, per_layer, cores, sample, len(times), sum(times), n_layers


def selfcheck_model(model, arch, prime):
    """Packed linears of the model that is about to be timed, on the real hidden states of one sample, against the fp32 torch
    restatement (quip_b200/selfcheck.restated_forward).  Layer 0: one linear per distinct (K, N) shape."""
    from quip_b200 import evalloop
    from quip_b200.quant import QuantLinear
    from quip_b200.selfcheck import rel_err, restated_forward
    res = {}
    with torch.no_grad():
        h, kw = evalloop.layer_inputs(model, arch, prime)
        layer0 = arch.layers(model)[0]
        seen = {}
        hooks = []
        for name, mod in layer0.named_modules():
            if isinstance(mod, QuantLinear) and (mod.infeatures, mod.outfeatures) not in seen:
                seen[(mod.infeatures, mod.outfeatures)] = name

                def fn(m, inp, outp, name=name):
                    x = inp[0]
                    res[name] = dict(K=m.infeatures, N=m.outfeatures, M=int(x.numel() // m.infeatures),
                                     rel_err_vs_fp32_restatement=rel_err(outp, restated_forward(m, x).reshape(outp.shape)))
                hooks.append(mod.register_forward_hook(fn))
        try:
            evalloop._call_layer(layer0, h, kw)
        finally:
            for hk in hooks:
                hk.remove()
    worst = max((r['rel_err_vs_fp32_restatement'] for r in res.values()), default=None)
    return dict(what='layer-0 packed linears of the timed model, real sample, vs fp32 torch restatement', worst=worst,
                tolerance=1e-3, layers=res)


def pp_main(a, base, rank, world):
    """--parallelism pp: the layer pipeline over all ranks (quip_b200.pipeline.PipelineStage)."""
    import torch.distributed as dist
    from quip_b200 import _lib, evalloop, pipeline
    from quip_b200.synth import MODELS, build_synthetic_model, model_config
    assert world > 1, 'the layer pipeline needs more than one rank (torchrun --nproc-per-node N)'
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    family = MODELS[a.model][0]
    arch = evalloop.LLAMA if family == 'llama' else evalloop.OPT
    cfg = model_config(a.model) if not a.layers else model_config(a.model, num_hidden_layers=a.layers)
    L = cfg.num_hidden_layers
    lo, hi = pipeline.stage_ranges(L, world)[rank]
    model = build_synthetic_model(cfg, dev, bits=2, incoh=a.incoh, rescale=True, seed=0, seqlen=SEQ, layer_range=(lo, hi),
                                  head=(rank == world - 1))
    model.seqlen = SEQ
    from quip_b200.quant import group_siblings
    groups = group_siblings(model)
    if family == 'llama' and os.environ.get('QUIP_FUSED_LAYER') is None:
        os.environ['QUIP_FUSED_LAYER'] = '1'
    total = a.warmup + a.steps
    gen = torch.Generator().manual_seed(1234)
    ids_host = torch.randint(0, cfg.vocab_size, (total, 1, SEQ), generator=gen).pin_memory()
    with torch.no_grad():
        stage = pipeline.PipelineStage(model, arch, lo, hi, dev, ids_host[0])
        check = selfcheck_stage(stage) if hi > lo else None

        def barrier():
            dist.barrier()
            torch.cuda.synchronize()
        # stage body alone (device time of one replay): the pipeline's steady state is paced by the slowest stage
        est = _device_ms(stage._compute, reps=2, warm=2)
        stage_ms = _device_ms(stage._compute, reps=max(3, min(60, int(2000.0 / max(est, 1e-3)))), warm=0)   # ~2 s: sustained clocks
        stage.run([ids_host[i] for i in range(a.warmup)])
        barrier()
        launches0 = lib.quip_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            barrier()
            clk.mark_start()
            e0.record()
            nll = stage.run([ids_host[i] for i in range(a.warmup, total)])
            t = torch.stack([nll, torch.tensor(float(a.steps * SEQ), device=dev)]) if rank == world - 1 else torch.zeros(2, device=dev)
            dist.all_reduce(t)
            e1.record()
            barrier()
            clk.mark_end()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        allst = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(allst, torch.tensor([stage_ms], device=dev))
        worst = torch.tensor([check['worst'] if check and check['worst'] is not None else 0.0], device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        n_launch = int(stage_launches(stage, lib) * a.steps)
        decode = None
        if not a.no_decode:
            # the reference's benchmark() on the placed model (opt.py:384-482): token-by-token decode across the stages
            try:
                for g in groups:
                    g.dissolve()
                r = pipeline.pp_decode_benchmark(model, arch, ids_host[0][:, :48], dev, max_len=64)
                decode = dict(tokens_per_s=1.0 / r['latency_s'], median_ms_per_token=r['latency_s'] * 1e3,
                              teacher_forced_tokens_per_s=1.0 / r['pipelined_s'], tokens=r['tokens'], stages=r['stages'],
                              note='quip_b200.pipeline.PipelinedDecoder: one GraphDecoder stage (CUDA graph, own KV cache of 64) '
                                   'per rank, (1, 1, hidden) fp16 hidden state over the per-link communicators; tokens_per_s = '
                                   'all ranks synchronised around every token (host clock), teacher_forced = free-running feed '
                                   'of given ids (stages overlap across tokens), batch 1')
            except Exception as e:
                decode = dict(error=repr(e)[:200])
    if rank == 0:
        ms = float(ms[0])
        stages = [float(x[0]) for x in allst]
        value = a.steps * SEQ / (ms / 1e3)
        ideal = SEQ / (max(stages) / 1e3)
        out = dict(base, value=value, ms_per_step=ms / a.steps, dtype='f16', impl='ours', scaling='strong',
                   gpu_launches=n_launch,
                   e2e=dict(value=value, unit='tokens/s', h2d_bytes_per_step=SEQ * 8, d2h_bytes_per_step=4,
                            api='quip_b200.pipeline.PipelineStage.run (host token ids, pinned)'),
                   pipeline=dict(stages=world, layers_per_stage=[list(r) for r in pipeline.stage_ranges(L, world)],
                                 stage_ms=stages, samples=a.steps,
                                 bubble_fill_drain=(world - 1) / (a.steps + world - 1),
                                 steady_state_tokens_per_s=ideal, efficiency_vs_slowest_stage=value / ideal,
                                 transfers='isend/irecv of (1, %d, %d) fp16 per link, per-link NCCL communicators, receive one '
                                           'sample ahead, sends double-buffered' % (SEQ, cfg.hidden_size)),
                   selfcheck=dict(worst_rel_err_over_stages=float(worst[0]), tolerance=1e-3), clocks=clk.summary())
        out['config'] = dict(base['config'], parallelism=f'pp{world}')
        if decode is not None:
            out['decode'] = decode
        print(json.dumps(out))
    dist.destroy_process_group()


def selfcheck_stage(stage):
    """selfcheck_model for a pipeline stage: its first decoder layer on its own (random) input buffer."""
    from quip_b200.quant import QuantLinear
    from quip_b200.selfcheck import rel_err, restated_forward
    from quip_b200 import evalloop
    res = {}
    layer0 = stage.layers[0]
    hooks, seen = [], set()
    for name, mod in layer0.named_modules():
        if isinstance(mod, QuantLinear) and (mod.infeatures, mod.outfeatures) not in seen:
            seen.add((mod.infeatures, mod.outfeatures))

            def fn(m, inp, outp, name=name):
                res[name] = rel_err(outp, restated_forward(m, inp[0]).reshape(outp.shape))
            hooks.append(mod.register_forward_hook(fn))
    try:
        h = torch.randn_like(stage.h_in)
        evalloop._call_layer(layer0, h, stage.kw)
    finally:
        for hk in hooks:
            hk.remove()
    return dict(worst=max(res.values(), default=None), layers=res)


def stage_launches(stage, lib):
    """Kernels of this library in one stage body (counted from one eager run of the body)."""
    n0 = lib.quip_launch_count()
    stage._body()
    torch.cuda.synchronize()
    return lib.quip_launch_count() - n0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--layers', type=int, default=0, help=argparse.SUPPRESS)   # debugging only
    ap.add_argument('--model', default='llama7b', choices=['llama7b', 'llama70b', 'opt1.3b', 'opt30b', 'opt125m'],
                    help='llama7b = BASELINE configs[2], the headline; the others are the remaining configs')
    ap.add_argument('--parallelism', default='dp', choices=['dp', 'pp'])
    ap.add_argument('--incoh', default='blocked', choices=['blocked', 'kron'],
                    help="butterfly structure of U / V: 'blocked' = one orthogonal block per position, what --incoh_processing runs "
                         "(opt.py:596, method.py:34-35; the headline); 'kron' = one block per stage (pre_proj_extra 1, method.py:38-39): "
                         "the factor bytes drop from n(p1+p2) to p1^2+p2^2 per side (not the headline configuration)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-decode', action='store_true', help='skip the one-token decode legs (quick runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps write what the last timed step returned (the NLL of its sample, float32) to '
                         'DIR/nll.npy; the inputs are fixed by seeds, so two builds can be compared output for output')
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != 'ours' or a.parallelism != 'dp'):
        ap.error('--dump-outputs covers the timed data-parallel path (--impl ours --parallelism dp)')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    structure = 'blocked butterflies' if a.incoh == 'blocked' else 'Kronecker butterflies (pre_proj_extra 1): NOT the headline structure'
    pretty = {'llama7b': 'Llama-2-7B', 'llama70b': 'Llama-2-70B', 'opt1.3b': 'OPT-1.3b', 'opt30b': 'OPT-30b', 'opt125m': 'OPT-125m'}[a.model]
    base = dict(metric=f'tokens/sec 2-bit {pretty} (per-layer eval path, seq 2048)', unit='tokens/s', n_gpus=a.gpus,
                steps=a.steps, warmup=a.warmup, higher_is_better=True, scaling='weak', vs_baseline=None, data='synthetic',
                config=dict(workload=f'{pretty} 2-bit --incoh_processing ({structure} + rescale), seq 2048, batch 1 '
                                     'per step, random codes / random orthogonal factors / random-init embeddings',
                            parallelism=f'dp{a.gpus}', l2='inputs larger than L2: each step streams 3.5 GB of packed '
                                                          'weights + butterfly factors',
                            setup='descriptors, fragment-order factor copies and per-stream workspaces are built by two '
                                  'untimed priming passes before the W warm-up steps; the decoder stack of a step is then '
                                  'captured once in a CUDA graph and replayed (QUIP_NO_GRAPH=1 for eager launches)'))

    if a.impl == 'reference':
        if rank != 0:
            return
        value, per_layer, cores, sample, nsteps, secs, n_layers = cpu_reference_arm(max(1, min(a.steps, 3)), 1, a.model)
        base.update(steps=nsteps, warmup=1, steps_requested=a.steps, timed_seconds=secs)
        out = dict(base, impl='reference', value=value, ms_per_step=per_layer * n_layers * 1e3, dtype='f16',
                   cpu_baseline=dict(value=value, unit='tokens/s', cores=cores, kind='port', sample=sample),
                   e2e=dict(value=value, unit='tokens/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(out))
        return

    assert a.warmup >= 3, 'timing rules: at least 3 warm-up steps'
    from quip_b200 import _lib, evalloop, pipeline
    from quip_b200.synth import MODELS, build_synthetic_model, model_config
    family = MODELS[a.model][0]
    arch = evalloop.LLAMA if family == 'llama' else evalloop.OPT
    if family == 'llama':
        from quip_b200.llama import llama_eval as model_eval
    else:
        from quip_b200.opt import opt_eval as model_eval
    # NCCL writes its debug output (the version banner at NCCL_DEBUG=VERSION/WARN) to stdout: send it to stderr so that
    # stdout carries the one JSON line only
    os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
    pipeline.init_distributed()
    import torch.distributed as dist
    if a.parallelism == 'pp':
        return pp_main(a, base, rank, world)
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    lib = _lib.load()

    cfg = model_config(a.model) if not a.layers else model_config(a.model, num_hidden_layers=a.layers)
    model = build_synthetic_model(cfg, dev, bits=2, incoh=a.incoh, rescale=True, seed=rank, seqlen=SEQ)
    model.seqlen = SEQ
    groups = []
    if os.environ.get('QUIP_NO_OVERLAP') != '1':
        from quip_b200.quant import group_siblings
        groups = group_siblings(model)  # q/k/v and gate/up chains run concurrently on side streams
    # one-time set-up outside the W warm-up steps: descriptors, fragment-order factor copies, per-stream workspaces
    # and first-launch module loads (two untimed passes; the W warm-up steps below still follow)
    with torch.no_grad():
        prime = torch.randint(0, cfg.vocab_size, (1, SEQ), device=dev)
        for _ in range(2):
            nll_prime = float(evalloop.sample_nll(model, arch, prime))       # HF glue: the reference value below
    torch.cuda.synchronize()
    check = selfcheck_model(model, arch, prime)
    assert check['worst'] is not None and check['worst'] < 1e-3, f'self-check of the timed model failed: {check}'
    glue = pick_glue(model, prime) if family == 'llama' else dict(mode='hf', why='fused glue kernels cover the Llama layer only')
    if glue['mode'] == 'fused':
        with torch.no_grad():                               # first-launch set-up of the fused path, outside the warm-up
            evalloop.sample_nll(model, arch, prime)
        torch.cuda.synchronize()
    base['config']['glue'] = glue
    # the decoder stack of a step as one CUDA graph (QUIP_NO_GRAPH=1: eager launches, as the roofline replay leg uses)
    stepper = None
    if os.environ.get('QUIP_NO_GRAPH') != '1':
        for attempt in range(2):
            try:
                stepper = evalloop.enable_graphed_eval(model, arch, prime)
                break
            except Exception as e:
                model._quip_graph_step = None
                stepper = None
                if glue['mode'] == 'fused' and attempt == 0:   # capture the HF-glue step instead
                    print(f'bench: capture of the fused stack failed ({e!r}); using the HF glue', file=sys.stderr)
                    os.environ['QUIP_FUSED_LAYER'] = '0'
                    glue.update(mode='hf', why='capture of the fused stack failed: ' + repr(e)[:160])
                    continue
                print(f'bench: graph capture failed ({e!r}); falling back to eager launches', file=sys.stderr)
                break
    step_fn = stepper if stepper is not None else (lambda ids: evalloop.sample_nll(model, arch, ids))
    if glue['mode'] == 'fused' and 'rel_err_vs_hf_layers' in glue:
        # whole model, end to end: the NLL of the priming sample through the step that will be timed, against the HF-glue
        # value from the priming pass; a disagreement beyond the perplexity tolerance puts the HF glue back
        with torch.no_grad():
            d = abs(float(step_fn(prime)) - nll_prime) / abs(nll_prime)
        glue['nll_rel_diff_vs_hf_glue'] = d
        # the loss is an fp16 number (opt.py:292-294: CrossEntropy on fp16 logits), so d moves in steps of ~7.5e-4: allow two
        if not d < 2e-3:
            os.environ['QUIP_FUSED_LAYER'] = '0'
            glue.update(mode='hf', why='NLL of the fused step differs from the HF-glue step')
            model._quip_graph_step = None
            stepper = None
            if os.environ.get('QUIP_NO_GRAPH') != '1':
                try:
                    stepper = evalloop.enable_graphed_eval(model, arch, prime)
                except Exception:
                    model._quip_graph_step = None
                    stepper = None
            step_fn = stepper if stepper is not None else (lambda ids: evalloop.sample_nll(model, arch, ids))
    gen = torch.Generator().manual_seed(1234 + rank)
    total = a.warmup + a.steps
    ids_host = torch.randint(0, cfg.vocab_size, (total, 1, SEQ), generator=gen).pin_memory()
    ids_dev = ids_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        return ms

    # ---- device-resident timing ----
    with torch.no_grad(), ClockSampler(local) as clk:
        for i in range(a.warmup):
            step_fn(ids_dev[i])
        barrier()
        launches0 = lib.quip_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        profiling = os.environ.get('QUIP_PROFILE') == '1'     # ncu --profile-from-start off: timed region only
        barrier()
        if profiling:
            torch.cuda.profiler.start()
        clk.mark_start()
        e0.record()
        nll = torch.zeros((), device=dev)
        for i in range(a.warmup, total):
            last = step_fn(ids_dev[i])
            nll += last
        if world > 1:
            dist.all_reduce(nll)
        e1.record()
        barrier()
        clk.mark_end()
        if profiling:
            torch.cuda.profiler.stop()
    if a.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, 'nll.npy'), last.float().cpu().numpy())
    with torch.no_grad():
        ms = max_over_ranks(e0.elapsed_time(e1))
        launches = lib.quip_launch_count() - launches0       # eager launches; a replayed graph is counted below

        # ---- roofline leg: per-launch CUDA-event timing of the dominant kernel over the same K steps.  The
        # sibling overlap is switched off for this replay: concurrent kernels share the SMs, so a per-launch
        # duration is only meaningful when the launch has the GPU to itself. ----
        for g in groups:
            g.dissolve()
        lib.quip_timing_reset()
        lib.quip_timing_enable(1)
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        r0.record()
        for i in range(a.warmup, total):
            evalloop.sample_nll(model, arch, ids_dev[i])
        r1.record()
        barrier()
        serial_ms = r0.elapsed_time(r1)
        if stepper is not None:
            # the graph replays exactly the launches of an eager step: count them from this eager replay of the same K steps
            launches = lib.quip_launch_count() - launches0 - launches
        lib.quip_timing_enable(0)
        tms, tn, tfl, tby = C.c_double(), C.c_int64(), C.c_double(), C.c_double()
        _lib.check(lib.quip_timing_read(2, C.byref(tms), C.byref(tn), C.byref(tfl), C.byref(tby)))
        lib.quip_timing_reset()
        if groups:
            from quip_b200.quant import group_siblings
            groups = group_siblings(model)

        # ---- end to end through the public API, host token ids ----
        for i in range(2):
            model_eval(model, ids_host[i], dev, verbose=False)
        barrier()
        t0 = time.perf_counter()
        for i in range(a.warmup, total):
            model_eval(model, ids_host[i], dev, verbose=False)      # H2D of the ids, D2H of the ppl scalar inside
        barrier()
        e2e_s = time.perf_counter() - t0
        e2e_ms = max_over_ranks(e2e_s * 1e3)

    if world > 1:
        t = torch.tensor([float(launches)], device=dev)
        dist.all_reduce(t)
        launches = int(t[0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    value = world * a.steps * SEQ / (ms / 1e3)
    e2e_value = world * a.steps * SEQ / (e2e_ms / 1e3)
    achieved = tfl.value / (tms.value / 1e3) / 1e12 if tms.value > 0 else None
    traffic, traffic_note = None, None
    prof = os.path.join(ROOT, 'profiles', 'ncu_qgemm_tc_latest.json')
    if os.path.exists(prof):
        pj = json.load(open(prof))
        traffic = pj.get('dram_bytes_per_launch')
        traffic_note = ('dram__bytes_read+write of one ncu --set full capture, %s: algorithmic %.1f MB (the activations '
                        'stay largely L2-resident between the kernels of one linear)' % (pj.get('shape'), pj.get('algorithmic_bytes', 0) / 1e6))
    out = dict(base, value=value, ms_per_step=ms / a.steps, dtype='f16', impl='ours', gpu_launches=int(launches),
               e2e=dict(value=e2e_value, unit='tokens/s', h2d_bytes_per_step=SEQ * 8, d2h_bytes_per_step=4,
                        api='quip_b200.llama.llama_eval' if family == 'llama' else 'quip_b200.opt.opt_eval'),
               roofline=dict(bound='tensor', kernel='qgemm_tc_kernel<2,256> (tcgen05 packed GEMM)', achieved=achieved,
                             peak=pk['tflops_sustained'], unit='TFLOP/s', frac=(achieved / pk['tflops_sustained']) if achieved else None,
                             traffic=traffic, traffic_note=traffic_note, launches_timed=int(tn.value), kernel_ms_per_step=tms.value / a.steps,
                             share_of_step=tms.value / ms, share_of_serial_replay=tms.value / serial_ms,
                             measured_in=('serial replay of the same K steps with CUDA events around every launch '
                                          '(sibling-stream overlap off, eager launches: %.2f ms/step, host gaps included); '
                                          'share_of_step = its summed launch time / the timed step (one graph replay, overlap '
                                          'on); the ncu launch list of the same command: profiles/launches_r02.json' % (serial_ms / a.steps)), peak_source=pk['source'] + ', sustained bf16 (kernel timed inside a long step)'),
               selfcheck=check, clocks=clk.summary())
    if world == 1 and not a.no_decode and a.model == 'llama7b':
        try:
            for g in groups:
                g.dissolve()
            out['decode'] = decode_leg(model, dev, pk)
            if glue['mode'] == 'fused':                          # the decode step has its own fused variant: check it too
                try:
                    ok, worst, control = decode_glue_ok(model, dev)
                except Exception as e:
                    ok, worst, control = False, repr(e)[:160], None
                os.environ['QUIP_FUSED_LAYER'] = '1' if ok else '0'
                out['decode']['glue'] = dict(mode='fused' if ok else 'hf', rel_err_vs_torch_glue_step=worst,
                                             control_torch_glue_vs_itself_with_ulp_flips=control)
            try:
                out['decode']['contraction_kernel'] = contraction_leg(dev, pk)
            except Exception as e:
                out['decode']['contraction_kernel'] = dict(error=repr(e)[:160])
            # the reference's benchmark() (opt.py:431-482): token-by-token through the whole HF model with a KV cache
            sec, _ = evalloop.decode_benchmark(model, ids_dev[0][:, :48])
            out['decode']['hf_decode'] = dict(tokens_per_s=1.0 / sec, median_ms_per_token=sec * 1e3, tokens=48,
                                              note='quip_b200.evalloop.decode_benchmark: eager HF forward per token '
                                                   '(host launch overhead included), batch 1')
            from quip_b200.decode import graph_decode_benchmark
            gsec, _ = graph_decode_benchmark(model, ids_dev[0][:, :48], max_len=64)
            from quip_b200.decode import graph_decode_throughput
            sweep = {}
            for bsz in (1, 2, 4, 8, 16, 32):                    # BASELINE configs[4]: batch 1-32 sweep
                try:
                    tps, step_ms = graph_decode_throughput(model, bsz, steps=24, max_len=32)
                    sweep[str(bsz)] = dict(tokens_per_s=tps, ms_per_step=step_ms)
                except Exception as e:                          # keep the sizes that ran
                    sweep[str(bsz)] = dict(error=repr(e)[:160])
            out['decode']['graph_decode_batch_sweep'] = sweep
            out['decode']['graph_decode'] = dict(tokens_per_s=1.0 / gsec, median_ms_per_token=gsec * 1e3, tokens=48,
                                                 note='quip_b200.decode.GraphDecoder: the same decode step (attention, norms, '
                                                      'static KV cache of 64, lm_head) replayed from one CUDA graph, batch 1')
        except Exception as e:                      # the decode leg is an extra; never lose the headline over it
            out['decode'] = dict(error=repr(e)[:200])
    if world == 1 and not a.no_decode and family == 'opt':
        # the model the reference's benchmark() is written for (opt.py:431-482): eager HF decode and the graph decode
        try:
            for g in groups:
                g.dissolve()
            from quip_b200.decode import graph_decode_benchmark, graph_decode_throughput
            sec, _ = evalloop.decode_benchmark(model, ids_dev[0][:, :48])
            gsec, _ = graph_decode_benchmark(model, ids_dev[0][:, :48], max_len=64)
            sweep = {}
            for bsz in (1, 8, 32):
                tps, step_ms = graph_decode_throughput(model, bsz, steps=24, max_len=32)
                sweep[str(bsz)] = dict(tokens_per_s=tps, ms_per_step=step_ms)
            out['decode'] = dict(hf_decode=dict(tokens_per_s=1.0 / sec, median_ms_per_token=sec * 1e3, tokens=48),
                                 graph_decode=dict(tokens_per_s=1.0 / gsec, median_ms_per_token=gsec * 1e3, tokens=48,
                                                   note='quip_b200.decode.GraphDecoder (OPT step, torch glue), static KV cache of 64'),
                                 graph_decode_batch_sweep=sweep)
        except Exception as e:
            out['decode'] = dict(error=repr(e)[:200])
    if world == 1 and not a.no_cpu_baseline:
        v, per_layer, cores, sample = cpu_reference_arm(1, 1, a.model)[:4]
        out['cpu_baseline'] = dict(value=v, unit='tokens/s', cores=cores, kind='port', sample=sample)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
