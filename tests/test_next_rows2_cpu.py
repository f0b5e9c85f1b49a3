"""CPU tests of two host mirrors next to the hot paths (SURVEY.md §8f rows 1 and 4): the sequence-sharded KV cache
update (lwm/llama.py:440-492) under gloo, and frame preprocessing (lwm/vision_chat.py:59-74) pinned against a
fixture produced by the reference's own function (tools/make_golden_next_rows_from_reference.py)."""
import os
import socket

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "process_frame_reference.npz")


def _images():
    from PIL import Image
    rng = np.random.RandomState(3)
    out = []
    for (w, h) in ((320, 240), (240, 320), (256, 256), (517, 300), (301, 777)):
        out.append(Image.fromarray(rng.randint(0, 256, size=(h, w, 3)).astype(np.uint8)))
    return out


def test_process_frame_matches_the_reference_fixture():
    from lwm_b200.vision_frames import process_frame, process_frames
    gold = np.load(GOLD)
    ims = _images()
    for i, im in enumerate(ims):
        got = process_frame(im, 64)
        assert got.shape == (64, 64, 3) and got.dtype == np.float32
        assert np.array_equal(got, gold["frame_%d" % i])
    assert process_frames(ims[:2]).shape == (2, 256, 256, 3)       # default size: the VQGAN's 256 x 256 input
    assert float(got.min()) >= -1.0 and float(got.max()) <= 1.0


def _cache_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from lwm_b200.kv_cache import ShardedKVCache
        B, H, D, max_len, prompt = 2, 2, 4, 16 * world, 5 * world
        g = torch.Generator().manual_seed(0)
        k_new = torch.randn(B, prompt, H, D, generator=g)
        v_new = torch.randn(B, prompt, H, D, generator=g)
        steps = [(torch.randn(B, 1, H, D, generator=g), torch.randn(B, 1, H, D, generator=g)) for _ in range(world * 6)]
        cache = ShardedKVCache(B, max_len, H, D, dtype=torch.float32, device="cpu")
        ql = prompt // world
        cache.concatenate(k_new[:, rank * ql:(rank + 1) * ql], v_new[:, rank * ql:(rank + 1) * ql])     # prefill
        for (kk, vv) in steps:                                                                          # decode
            ck, cv = cache.concatenate(kk, vv)
        ret[rank] = (ck.numpy(), cv.numpy(), cache.cache_index)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2, 4])
def test_sharded_kv_cache_matches_the_unsharded_update(world):
    import torch.multiprocessing as mp
    B, H, D, max_len, prompt = 2, 2, 4, 16 * world, 5 * world
    g = torch.Generator().manual_seed(0)
    k_new = torch.randn(B, prompt, H, D, generator=g)
    v_new = torch.randn(B, prompt, H, D, generator=g)
    steps = [(torch.randn(B, 1, H, D, generator=g), torch.randn(B, 1, H, D, generator=g)) for _ in range(world * 6)]
    ref_k, ref_v = torch.zeros(B, max_len, H, D), torch.zeros(B, max_len, H, D)
    ref_k[:, :prompt], ref_v[:, :prompt] = k_new, v_new          # dynamic_update_slice at index 0 (llama.py:485-487)
    idx = prompt
    for (kk, vv) in steps:
        ref_k[:, idx], ref_v[:, idx] = kk[:, -1], vv[:, -1]      # .at[:, cur_index].set(key[:, -1]) (llama.py:461-462)
        idx += 1
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_cache_worker, args=(world, port, ret), nprocs=world, join=True)
    L = max_len // world
    for r in range(world):
        ck, cv, ci = ret[r]
        assert ci == idx
        assert np.array_equal(ck, ref_k[:, r * L:(r + 1) * L].numpy())
        assert np.array_equal(cv, ref_v[:, r * L:(r + 1) * L].numpy())
