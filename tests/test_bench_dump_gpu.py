"""bench.py on the B200: --steps sets the number of timed steps, and --dump-outputs writes a fixed float32 sample of
what the last timed step returned, equal to the public op's results on the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_fro

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, H, D = 4096, 32, 128
NAMES = ("out", "dq", "dk", "dv")


def _bench(steps, dump_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--seq", str(S), "--steps",
                        str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-vqgan", "--no-parity",
                        "--dump-outputs", str(dump_dir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {n: np.load(os.path.join(str(dump_dir), n + ".npy")) for n in NAMES}


def test_steps_and_dumped_outputs(tmp_path):
    one, d1 = _bench(1, tmp_path / "one")
    three, d3 = _bench(3, tmp_path / "three")
    assert one["steps"] == 1 and three["steps"] == 3
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    assert sorted(os.listdir(tmp_path / "one")) == sorted(n + ".npy" for n in NAMES)
    assert sum(os.path.getsize(tmp_path / "one" / (n + ".npy")) for n in NAMES) <= 64 << 20
    for n in NAMES:
        assert d1[n].dtype == np.float32 and d1[n].shape == (512, H, D)
        assert np.isfinite(d1[n]).all() and np.abs(d1[n]).max() > 0
        assert rel_fro(d3[n], d1[n]) < 1e-3, n

    # the same op on the same inputs in this process, sampled the same way
    from lwm_b200 import ringattention as ra
    from lwm_b200 import synthetic as syn
    q, k, v, do = [syn.shard(n_, 0, S, H, D, 1234).cuda() for n_ in ("q", "k", "v", "do")]
    q, k, v = [t.requires_grad_(True) for t in (q, k, v)]
    out = ra.ringattention(q, k, v, None, None, axis_name="sp", float32_logits=True, cache_idx=None,
                           blockwise_kwargs=dict(causal_block_size=1, deterministic=True, dropout_rng=None,
                                                 attn_pdrop=0.0, query_chunk_size=1024, key_chunk_size=1024,
                                                 dtype=torch.bfloat16, policy=None, precision=None, prevent_cse=True))
    out.backward(do)
    rows = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:512].sort().values.cuda()
    for n, t in zip(NAMES, (out, q.grad, k.grad, v.grad)):
        want = t.detach()[0].index_select(0, rows).float().cpu().numpy()
        assert rel_fro(d1[n], want) < 1e-3, n
