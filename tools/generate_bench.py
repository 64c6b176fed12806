"""Generation benchmark on Llama-2-7B shapes (2-bit synthetic packed model): prefill, graph-replayed decode with
quip_decode_attention, and the attention step alone against GraphDecoder's masked SDPA over the same cache.

    python tools/generate_bench.py --out DIR [--prompt 512 2048] [--batch 1 8 32] [--new 128] [--layers 32]

For every (prompt length, batch): prefill ms (one pass of B x P tokens, after one warm-up pass); decode ms per token and
tokens/s over new-1 graph replays (the first new token comes from the prefill); and, at the first and the last position
the decode writes, the attention of one layer: quip_decode_attention alone, and GraphDecoder._attend (index_copy_ +
masked SDPA over all max_len positions) on the same cache.  Each is recorded as a CUDA graph of `reps` calls, as it runs
inside the decode step, and the two graphs are replayed alternately in rounds (CUDA events, median round).  The calls
rotate through the layers' caches so that the working set is larger than the 126 MB L2.  Bytes of the kernel are the
valid K / V rows (2 * B * (ctx+1) * nkv * hd * 2) plus q, k_new, v_new and out.  Writes DIR/generate_bench.json with the
GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def hbm_peak_gbs():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 7700.0, 'HGX B200 data sheet, one GPU'


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def attention_compare(gen, ctx, rounds=11, reps=64):
    """us per layer of the kernel and of GraphDecoder's masked SDPA at position ctx of every row."""
    from types import SimpleNamespace

    from quip_b200.decode import GraphDecoder
    from quip_b200.generate import CudaDecodeAttention
    B, nh, nkv, hd, L = gen.batch, gen.nh, gen.nkv, gen.hd, len(gen.layers)
    g = torch.Generator(device='cuda').manual_seed(0)
    q = torch.randn(B, nh * hd, device='cuda', generator=g).half()
    kn = torch.randn(B, nkv * hd, device='cuda', generator=g).half()
    vn = torch.randn(B, nkv * hd, device='cuda', generator=g).half()
    pos32 = torch.full((B,), ctx, dtype=torch.int32, device='cuda')
    attn, scale = CudaDecodeAttention(), hd ** -0.5
    ref = SimpleNamespace(position=torch.tensor([ctx], device='cuda'), k_cache=gen.k_cache, v_cache=gen.v_cache,
                          nh=nh, nkv=nkv)
    mask = GraphDecoder._attn_context(SimpleNamespace(_arange=torch.arange(gen.max_len, device='cuda'),
                                                      position=ref.position))
    q4 = q.view(B, 1, nh, hd).transpose(1, 2)
    k4, v4 = kn.view(B, 1, nkv, hd).transpose(1, 2), vn.view(B, 1, nkv, hd).transpose(1, 2)

    def kern(i):
        attn(q, kn, vn, gen.k_cache[i % L], gen.v_cache[i % L], pos32, scale)

    def sdpa(i):
        GraphDecoder._attend(ref, i % L, q4, k4, v4, scale, mask)

    # each side recorded as one graph of `reps` calls, as they run inside the decode step: device time, not enqueue time
    graphs = []
    for fn in (kern, sdpa):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn(0)                                          # warm-up outside the graph: workspace, SDPA backend
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=side):
                for i in range(reps):
                    fn(i)
        torch.cuda.current_stream().wait_stream(side)
        graphs.append(gr)
    torch.cuda.synchronize()
    tk, ts = [], []
    for _ in range(rounds):
        tk.append(events_ms(lambda i: graphs[0].replay(), 1) / reps)
        ts.append(events_ms(lambda i: graphs[1].replay(), 1) / reps)
    tk.sort()
    ts.sort()
    us_k, us_s = 1e3 * tk[len(tk) // 2], 1e3 * ts[len(ts) // 2]
    nbytes = 2 * B * (ctx + 1) * nkv * hd * 2 + 2 * B * nh * hd * 2 + 2 * B * nkv * hd * 2
    return dict(context=ctx, kernel_us_per_layer=us_k, masked_sdpa_us_per_layer=us_s, kernel_bytes=nbytes,
                kernel_gbs=nbytes / (us_k * 1e-6) / 1e9, sdpa_cache_positions=gen.max_len)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--prompt', type=int, nargs='+', default=[512, 2048])
    ap.add_argument('--batch', type=int, nargs='+', default=[1, 8, 32])
    ap.add_argument('--new', type=int, default=128)
    ap.add_argument('--layers', type=int, default=32)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('generate_bench.py measures on a CUDA device; none is visible')
    from quip_b200 import fused
    from quip_b200.generate import Generator
    from quip_b200.synth import build_synthetic_model, model_config
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device('cuda:0')
    t0 = time.time()
    cfg = model_config('llama7b', num_hidden_layers=a.layers)
    model = build_synthetic_model(cfg, dev, bits=2, incoh='blocked', rescale=True, seed=0, seqlen=max(a.prompt))
    build_s = time.time() - t0
    peak, peak_src = hbm_peak_gbs()
    res = dict(model='llama7b shapes, 2-bit synthetic (synth.build_synthetic_model)', layers=a.layers, new_tokens=a.new,
               gpu=gpu_info(), fused_glue=fused.enabled(), hbm_peak_gbs=peak, hbm_peak_source=peak_src,
               model_build_s=build_s, runs=[])
    g = torch.Generator().manual_seed(1)
    for P in a.prompt:
        for B in a.batch:
            prompts = [torch.randint(0, cfg.vocab_size, (P,), generator=g).to(dev) for _ in range(B)]
            with torch.no_grad():
                gen = Generator(model, B, P + a.new - 1).capture()
                gen.prefill(prompts)                                   # warm-up pass
                for _ in range(4):
                    gen.step()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                gen.prefill(prompts)
                e1.record()
                torch.cuda.synchronize()
                prefill_ms = e0.elapsed_time(e1)
                steps = a.new - 1
                decode_ms = events_ms(lambda i: gen.step(), steps)
                # the first and the last position the decode writes
                att = [attention_compare(gen, ctx) for ctx in (P, P + a.new - 2)]
            for x in att:
                x['kernel_share_of_hbm_peak'] = x['kernel_gbs'] / peak
            run = dict(prompt=P, batch=B, prefill_ms=prefill_ms, decode_ms_per_token=decode_ms,
                       decode_tokens_per_s=B * 1e3 / decode_ms, attention=att)
            print(json.dumps(run), flush=True)
            res['runs'].append(run)
            del gen
            torch.cuda.empty_cache()
    path = os.path.join(a.out, 'generate_bench.json')
    with open(path, 'w') as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == '__main__':
    main()
