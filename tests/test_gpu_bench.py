"""bench.py end to end at two decoder layers: --steps sets the number of timed steps, and --dump-outputs writes the NLL the
last timed step returned, which an eager pass of the same sample through the same model reproduces."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def test_bench_dumps_what_the_last_timed_step_returned(tmp_path):
    from quip_b200 import evalloop
    from quip_b200.synth import build_synthetic_model, model_config
    steps, warmup, layers = 2, 3, 2
    out = tmp_path / 'dump'
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', str(steps),
                        '--warmup', str(warmup), '--layers', str(layers), '--no-decode', '--no-cpu-baseline',
                        '--dump-outputs', str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d['steps'] == steps and d['warmup'] == warmup
    got = np.load(out / 'nll.npy')
    assert got.dtype == np.float32 and got.shape == () and np.isfinite(got)
    # bench.py's inputs: the synthetic model of rank 0 (seed 0) and one seeded sample per warm-up and timed step
    dev = torch.device('cuda:0')
    cfg = model_config('llama7b', num_hidden_layers=layers)
    model = build_synthetic_model(cfg, dev, bits=2, incoh='blocked', rescale=True, seed=0, seqlen=2048)
    ids = torch.randint(0, cfg.vocab_size, (warmup + steps, 1, 2048), generator=torch.Generator().manual_seed(1234))
    want = float(evalloop.sample_nll(model, evalloop.LLAMA, ids[-1].to(dev)))
    # the loss is an fp16 number (~7.5e-4 relative per ulp); the timed step may run the fused glue: allow two ulps
    assert abs(float(got) - want) / abs(want) < 2e-3, (float(got), want)
