#!/usr/bin/env python
"""bench.py — headline benchmark of the lwm_b200 hot paths (see BASELINE.json / DESIGN.md §Measurement).

Workload (config.workload): ring attention forward+backward of ONE LWM-7B layer
(H=32, D=128, hidden 4096, B=1, causal) at S=131072 tokens, bf16 in / fp32 accumulate, sequence
sharded over N GPUs (N=1: the whole 128K sequence on one B200). A "step" is one forward+backward
pass of that layer's attention through the public `ringattention` op. STRONG scaling: total
work is fixed as N grows.

  value   tokens/s of the attention path of a 32-layer 7B model = S / (32 * t_step), inputs resident
          in HBM, device-timed (CUDA events, barrier + synchronize on both sides, max over ranks)
  e2e     same metric through the same public op with HOST (pinned) q/k/v/dout: H2D copies of the
          inputs and D2H copies of out/dq/dk/dv inside the timed region
  roofline   tensor-bound: algorithmic causal FLOPs of the dominant kernel (attn_bwd_kernel) per
          launch / its CUDA-event duration, against the measured cuBLAS bf16 peak
  gpu_launches   C-ABI compute calls into liblwm_b200.so (each launches at least one of this repo's kernels) made by
          rank 0 inside the timed region, counted by lwm_b200._lib.launch_count()
  cpu_baseline / --impl reference   the CPU restatement of the reference algorithm (oracle/),
          timed on the host cores on a bounded sample of the same workload.
  parity  before anything is timed, the SAME op on the SAME inputs (all N ranks) is checked against the float64
          row-wise oracle (oracle/attn_rows.py): out / dq of one sampled query row per 128-row tile and dk / dv of
          every key row, two heads, fp32 read-out; max relative Frobenius error over ranks (north_star bound 1e-3)
  reference_probe   whether the reference's own JAX implementation (jax + the un-vendored `ringattention` package)
          is importable on this box — if it ever is, the oracle is pinned against it on a small case right here

--dump-outputs DIR writes what the last timed step returned to its caller (out, dq, dk, dv) as float32 .npy files, a
fixed seeded sample of token rows (see dump_outputs), so that two builds can be compared output for output: the inputs
depend only on the arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S_TOTAL = 131072
H, D, LAYERS = 32, 128, 32
METRIC = "ring_attn_fwd_bwd_tokens_per_s_attention_only_7B_128K"
UNIT = "tokens/s"


def f_fwd(S):
    """algorithmic causal forward FLOPs of one layer (SURVEY.md §8d): 4*B*H*D*S(S+1)/2."""
    return 4.0 * H * D * S * (S + 1) / 2.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=float(d["bf16_tflops"]), sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    hbm=float(d["hbm_gbs"]), source="MEASURED_PEAKS.json")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        clocks, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [x.strip() for x in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                clocks.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        clocks.sort()
        med = clocks[len(clocks) // 2] if clocks else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(clocks)}


# ------------------------------------------------------------------------------------------------
# CPU restatement timed on the host cores (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------------
def cpu_sample_step(S, rows, heads, chunk=1024):
    """Blockwise online-softmax forward + recompute backward (SURVEY.md Appendix A) for the LAST
    `rows` query rows of an S-token causal sequence and `heads` heads, fp32, torch CPU matmuls.
    Returns (seconds, flops)."""
    import torch
    from oracle import ring_blockwise as rb
    g = torch.Generator().manual_seed(0)
    q = torch.randn(1, rows, heads, D, generator=g)
    k = torch.randn(1, S, heads, D, generator=g)
    v = torch.randn(1, S, heads, D, generator=g)
    do = torch.randn(1, rows, heads, D, generator=g)
    t0 = time.perf_counter()
    rb.torch_blockwise_fwd_bwd(q, k, v, do, q_pos0=S - rows, chunk=chunk)
    dt = time.perf_counter() - t0
    # full (not causal-halved) tiles except the diagonal chunk: count exact visible pairs
    vis = sum(min(S, (S - rows) + i + 1) for i in range(rows))
    flops = 3.5 * 4.0 * heads * D * vis
    return dt, flops


def workload_name(S):
    """one string for both arms (the reference arm runs on 'your arm's config')"""
    return "LWM-7B ring attention fwd+bwd, one layer, S=%d B=1 H=32 D=128 causal" % S


def run_reference_arm(args, rank):
    """`--impl reference`: the reference's own (CPU) algorithm for this path, restated in oracle/
    (the un-vendored JAX package cannot be installed offline — DESIGN.md), all host threads."""
    if rank != 0:
        return
    import torch
    cores = min(len(os.sched_getaffinity(0)), 32)
    torch.set_num_threads(cores)
    rows, heads = 2048, 2        # a fixed sample of the 128K problem: 9.5e11 FLOP per step (~4 s on the box's 32 cores)
    times, flops = [], 0.0
    for i in range(args.warmup + args.steps):
        dt, flops = cpu_sample_step(S_TOTAL, rows, heads)
        if i >= args.warmup:
            times.append(dt)
    times.sort()
    t = times[len(times) // 2]   # median: the host cores are shared with whatever else runs on the box
    full = 3.5 * f_fwd(S_TOTAL)
    t_layer = t * full / flops                      # extrapolated time of one whole layer
    value = S_TOTAL / (LAYERS * t_layer)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(S_TOTAL),
                   "tokens_per_s_definition": "S / (32 layers * t_step), attention only",
                   "note": "CPU restatement of the reference algorithm (oracle/ring_blockwise.py); the JAX "
                           "reference cannot be installed offline"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "last %d query rows x %d head of the 128K causal problem per step, fwd+bwd, "
                                   "extrapolated by FLOPs (x%.0f) to one layer" % (rows, heads, full / flops)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_gflops": flops / t / 1e9, "cpu_seconds_per_step": t, "cpu_step_spread": [times[0], times[-1]],
    }
    print(json.dumps(line))


def probe_reference():
    """SURVEY.md §8c: the ring-attention arithmetic lives in the un-vendored JAX package `ringattention`. If this box can
    import it (it cannot in the stock image: no jax, no network), run its CPU path on a small case and pin
    oracle/ring_blockwise.py against it; otherwise say why not."""
    try:
        import jax  # noqa: F401
        import jax.numpy as jnp
        from ringattention import ringattention_jax  # noqa: F401
    except Exception as e:      # noqa: BLE001
        return {"importable": False, "why": "%s: %s" % (type(e).__name__, str(e)[:120]),
                "oracle_pinned_against_reference": False}
    try:
        import numpy as np
        from oracle.attn_dense import attention_dense
        rng = np.random.RandomState(0)
        qn, kn, vn = [rng.randn(1, 512, 2, 64).astype(np.float32) for _ in range(3)]
        bias = jnp.zeros((1, 1, 1, 512), jnp.float32)
        out = ringattention_jax(jnp.asarray(qn), jnp.asarray(kn), jnp.asarray(vn), bias, None, axis_name=None,
                                float32_logits=True, cache_idx=None,
                                blockwise_kwargs=dict(causal_block_size=1, deterministic=True, dropout_rng=None,
                                                      attn_pdrop=0.0, query_chunk_size=128, key_chunk_size=128,
                                                      dtype=jnp.float32, policy=None, precision=None, prevent_cse=True))
        ref = attention_dense(qn, kn, vn, causal=True)
        err = float(np.linalg.norm(np.asarray(out, dtype=np.float64) - ref) / np.linalg.norm(ref))
        return {"importable": True, "oracle_vs_reference_rel_err": err, "oracle_pinned_against_reference": bool(err < 1e-5)}
    except Exception as e:      # noqa: BLE001
        return {"importable": True, "why": "reference call failed: %s" % str(e)[:160],
                "oracle_pinned_against_reference": False}


VQ_FLOPS_ENC, VQ_FLOPS_DEC = 216.6e9, 477.4e9           # per 256x256 frame (SURVEY.md Appendix C)
VQ_BYTES_ENC = 815.5e6                                   # minimum activation traffic per frame, fp32 activations (SURVEY.md §8d)


def bench_vqgan(dev, peaks, world, rank, with_cpu=True):
    """BASELINE 'VQGAN frames/s': encode of a 16-frame 256x256 clip, synthetic weights and pixels, default precision
    mode, same contract as the attention record: `value` with the clip resident in HBM, `e2e` from pinned host pixels to
    host codes (copies inside the timed region), `roofline` against the HBM roof north_star names (algorithmic bytes =
    SURVEY.md §8d minimum-traffic model with fp32 activations, 815.5 MB / frame) with the tensor-pipe fraction beside
    it, `cpu_baseline` = the CPU restatement (oracle/vqgan_ref.py) on a bounded sample, `parity` on that same sample.
    Replicas only across GPUs (frames are independent: no collective)."""
    import numpy as np
    import torch
    from lwm_b200.vqgan import VQGAN, init_params
    params = init_params(seed=0, codebook="normal")
    g = torch.Generator().manual_seed(1234)
    hx = (torch.rand(16, 256, 256, 3, generator=g) * 2 - 1).pin_memory()
    x = hx.to(dev)
    tok = VQGAN(params, device=str(dev))
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b2 = ev(), ev()
        a.record()
        for _ in range(n):
            fn()
        b2.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b2) / n
    ms = timed(lambda: tok.encode(x), 10)
    hidx = torch.empty(16, 16, 16, dtype=torch.int32).pin_memory()

    def e2e():
        xd = hx.to(dev, non_blocking=True)
        _, idx = tok.encode(xd)
        hidx.copy_(idx.reshape(16, 16, 16), non_blocking=True)
        torch.cuda.current_stream().synchronize()       # the caller reads the codes on the host
    ms_e2e = timed(e2e, 10)
    codes = torch.randint(0, 8192, (16, 16, 16), dtype=torch.int32, device=dev)
    ms_dec = timed(lambda: tok.decode(codes), 5)
    fps = 16 / (ms * 1e-3)
    gbs = 16 * VQ_BYTES_ENC / (ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_vqgan_encode16_r02.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_total_bytes_per_clip")
    passes = 2.15        # FLOP-weighted MMA work of the mixed mode (2 on the >= 64x64 levels, 3 below)
    rec = {
        "metric": "vqgan_encode_frames_per_s_256x256x16f", "value": world * fps, "unit": "frames/s", "n_gpus": world,
        "scaling": "replicas (frames independent, no collective)", "ms_per_clip": ms, "frames_per_s_per_gpu": fps,
        "dtype": "f16 tensor-core operands (activation fp16, weights fp16 hi+lo), fp32 accumulate, fp32 activations in HBM",
        "config": {"workload": "VQGAN encode, 16 frames 256x256x3, LWM VQGANConfig defaults (58.7M encoder params)",
                   "precision": "fp16x2 (mixed: 2-MMA fp16 scheme on the >=64x64 levels, 3-MMA split-bf16 below)",
                   "l2": "every conv streams 34 MB .. 537 MB of activations per clip: larger than the 126 MB L2 on the "
                         "levels that carry 90 % of the bytes"},
        "roofline": {"bound": "hbm", "kernel": "whole encode (dominant: conv_umma_kernel)", "achieved": gbs,
                     "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"], "traffic": traffic,
                     "algorithmic_bytes_per_clip": 16 * VQ_BYTES_ENC,
                     "tensor": {"algorithmic_tflops": 16 * VQ_FLOPS_ENC / (ms * 1e-3) / 1e12,
                                "issued_tflops": passes * 16 * VQ_FLOPS_ENC / (ms * 1e-3) / 1e12,
                                "frac_of_bf16_peak_issued": passes * 16 * VQ_FLOPS_ENC / (ms * 1e-3) / 1e12 / peaks["sustained"]},
                     "note": "north_star quotes the HBM roof; the 3x3 convs are tensor-bound (AI >= 576 FLOP/B), so the "
                             "composite floor is max(bytes/HBM, issued FLOPs/tensor peak)"},
        "e2e": {"value": world * 16 / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_clip": ms_e2e,
                "h2d_bytes_per_step": hx.numel() * 4, "d2h_bytes_per_step": hidx.numel() * 4,
                "copies": "pinned host fp32 pixels -> device, int32 codes -> pinned host, host waits for the codes"},
        "decode": {"ms_per_clip": ms_dec, "frames_per_s_per_gpu": 16 / (ms_dec * 1e-3),
                   "algorithmic_tflops": 16 * VQ_FLOPS_DEC / (ms_dec * 1e-3) / 1e12},
    }
    if with_cpu and rank == 0:
        from oracle import vqgan_ref as vr
        cores = min(len(os.sched_getaffinity(0)), 32)
        torch.set_num_threads(cores)
        nfr = 2
        t0 = time.perf_counter()
        ref_zq, ref_idx, ref_h = vr.encode(hx[:nfr], params)
        dt = time.perf_counter() - t0
        _, idx = tok.encode(x[:nfr])
        h = tok.model.ops.conv_gn(tok.model.encoder(x[:nfr].contiguous()), tok.model.p["quant_conv"])
        torch.cuda.synchronize()
        lat = float(np.linalg.norm(h.cpu().numpy().astype(np.float64) - ref_h) / np.linalg.norm(ref_h))
        rec["cpu_baseline"] = {"value": nfr / dt, "unit": "frames/s", "cores": cores, "kind": "port",
                               "sample": "oracle/vqgan_ref.py encode (torch CPU fp32) of the clip's first %d frames: "
                                         "%.1f s of CPU work" % (nfr, dt)}
        rec["parity"] = {"latent_rel": lat, "tol": 1e-3, "frames": nfr,
                         "index_agreement": float((idx.cpu().numpy().astype(np.int32) == ref_idx).mean()),
                         "note": "codes are bit-exact at the VectorQuantizer boundary (tests/test_vqgan_gpu.py); end to "
                                 "end a code can differ only where the oracle's two nearest codes tie within the latent "
                                 "error"}
    return rec


DUMP_ROWS = 512     # token rows sampled per output: 4 outputs x 512 rows x 32 heads x 128 x fp32 = 32 MB


def dump_outputs(dirname, outputs, rank, world):
    """Write the step's outputs ([1, S/N, H, D] each, 1 GiB apiece at 128K tokens on one GPU) as DIR/<name>.npy, float32,
    shape [rows, H, D]: the same seeded sample of DUMP_ROWS token rows of the local shard (sorted, every head and channel)
    in every run. With N ranks each writes DUMP_ROWS / N rows of its own shard as <name>_rank<r>.npy."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    g = torch.Generator().manual_seed(0)
    rows = torch.randperm(outputs[0].shape[1], generator=g)[:max(1, DUMP_ROWS // world)].sort().values
    suffix = "" if world == 1 else "_rank%d" % rank
    for name, t in zip(("out", "dq", "dk", "dv"), outputs):
        a = t.detach()[0].index_select(0, rows.to(t.device)).float().cpu().numpy()
        np.save(os.path.join(dirname, name + suffix + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="lwm_b200")
    ap.add_argument("--seq", type=int, default=S_TOTAL, help="(debug) override the total sequence length")
    ap.add_argument("--layout", default="auto")
    ap.add_argument("--precision", default=None, choices=[None, "bf16", "fp16"],
                    help="attention precision mode (default: the package default, bf16)")
    ap.add_argument("--e2e-serial", action="store_true",
                    help="e2e leg with the host<->device copies serialised with the kernels instead of double-buffered "
                         "(default: step i+1's uploads and step i-1's downloads overlap step i's kernels)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="(debug) skip the oracle check that precedes the timing")
    ap.add_argument("--no-vqgan", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's out / dq / dk / dv to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from lwm_b200 import ringattention as ra

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: lwm_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")   # NCCL copy kernels must be able to preempt
        dist.init_process_group("nccl", device_id=dev)
    S = args.seq
    assert S % world == 0
    Sl = S // world
    W, K = max(args.warmup, 3), args.steps
    peaks = load_peaks()

    from lwm_b200 import synthetic as syn
    torch.set_num_threads(max(1, min(len(os.sched_getaffinity(0)), 64) // world))
    # N(0,1) rounded to bf16; every (tensor, rank, head) has its own seeded stream so that any rank can rebuild any
    # head of the whole sequence for the oracle check
    hq, hk, hv, hdo = [syn.shard(n_, rank, Sl, H, D, 1234).pin_memory() for n_ in ("q", "k", "v", "do")]
    q, k, v, do = [t.to(dev) for t in (hq, hk, hv, hdo)]
    kwargs = dict(axis_name="sp", float32_logits=True, cache_idx=None,
                  blockwise_kwargs=dict(causal_block_size=1, deterministic=True, dropout_rng=None, attn_pdrop=0.0,
                                        query_chunk_size=1024, key_chunk_size=1024, dtype=torch.bfloat16,
                                        policy=None, precision=None, prevent_cse=True), layout=args.layout,
                  precision=args.precision)
    from lwm_b200 import _lib

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    kern_ms = {"fwd": [], "bwd": []}

    def step():
        qq, kk, vv = [t.detach().requires_grad_(True) for t in (q, k, v)]
        out = ra.ringattention(qq, kk, vv, None, None, **kwargs)
        out.backward(do)
        return out, qq.grad, kk.grad, vv.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity of exactly this op / sharding / precision mode on exactly these inputs, before anything is timed
    parity = None
    if not args.no_parity:
        from lwm_b200.selftest import sampled_parity
        # (a failure here is reported in the line, it must not take the measurement down with it; every rank takes the
        # same branch: an exception on one rank would leave the others in the all_reduce below)
        try:
            pe = sampled_parity(S, H, [0, H - 1], lambda a, b, c: ra.ringattention(a, b, c, None, None, **kwargs), dev,
                                rank, world, 1234, shards=dict(q=q, k=k, v=v, do=do))
        except Exception as e:      # noqa: BLE001
            if world > 1:
                raise               # a multi-rank failure cannot be papered over: the other ranks are inside the op
            pe = {"out": 9.0, "dq": 9.0, "dk": 9.0, "dv": 9.0, "dq_unsampled_abs": 9.0, "rows": 0, "keys": 0}
            print("parity check failed: %s: %s" % (type(e).__name__, str(e)[:300]), file=sys.stderr)
        worst = max(pe[n_] for n_ in ("out", "dq", "dk", "dv"))
        tp = torch.tensor([pe["out"], pe["dq"], pe["dk"], pe["dv"], pe["dq_unsampled_abs"], worst], device=dev)
        tn = torch.tensor([float(pe["rows"]), float(pe["keys"])], device=dev)
        if world > 1:
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            dist.all_reduce(tn, op=dist.ReduceOp.SUM)
        tp, tn = tp.tolist(), tn.tolist()
        parity = {"max_rel": tp[5], "tol": 1e-3, "ok": bool(tp[5] < 1e-3 and tp[4] == 0.0),
                  "per_tensor": {"out": tp[0], "dq": tp[1], "dk": tp[2], "dv": tp[3]},
                  "rows": int(tn[0]), "key_rows": int(tn[1]), "heads_checked": [0, H - 1],
                  "oracle": "oracle/attn_rows.py (float64, row-wise restatement of oracle/attn_dense.py); fp32 read-out "
                            "of the op on the bench inputs, dO zero outside the sampled query rows; max over %d rank(s)"
                            % world}
        torch.set_num_threads(max(1, min(len(os.sched_getaffinity(0)), 64)))
    for _ in range(W):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t0, t1 = ev(), ev()
    barrier()
    calls0 = _lib.launch_count()
    t0.record()
    for i in range(K):
        last = step()
        if i + 1 < K:
            last = None         # only the last step's results outlive their step
    t1.record()
    barrier()
    gpu_launches = _lib.launch_count() - calls0      # C-ABI compute calls of this rank in the timed region
    ms = t0.elapsed_time(t1) / K
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, rank, world)
    last = None
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        tm = torch.tensor([ms], device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms = float(tm.item())

    # ---- dominant-kernel timing (single GPU): the raw fwd / bwd tile kernels, CUDA events on their stream
    roof = None
    if world == 1:
        out = torch.empty_like(q)
        lse = torch.empty(1, H, Sl, dtype=torch.float32, device=dev)
        delta = torch.empty_like(lse)
        dq = torch.zeros(1, Sl, H, D, dtype=torch.float32, device=dev)
        dk = torch.zeros_like(dq)
        dv = torch.zeros_like(dq)
        prec = args.precision or ra._DEFAULT_PRECISION
        if prec == "fp16":      # the tile kernels of the default mode: fp16 operand copies + their scales
            (kq, sq_), (kk, sk_), (kv, sv_), (kdo, sd_) = [ra.to_f16(t) for t in (q, k, v, do)]
            fsc, bsc = (sq_, sk_, sv_), (sq_, sk_, sv_, sd_)
        else:
            kq, kk, kv, kdo, fsc, bsc = q, k, v, do, None, None
        ra.fwd_step(kq, kk, kv, out, lse, None, None, None, 0, 0, True, None, None, True, True, scales=fsc)
        ra.bwd_prep(out, do, delta)
        nlse2 = ra.lse_for_bwd(lse, f16=(prec == "fp16"))
        for name, fn in (("fwd", lambda: ra.fwd_step(kq, kk, kv, out, lse, None, None, None, 0, 0, True, None, None,
                                                     True, True, scales=fsc)),
                         ("bwd", lambda: ra.bwd_step(kq, kk, kv, kdo, nlse2, delta, dq, dk, dv, 0, 0, True, None, None,
                                                     scales=bsc))):
            fn()
            torch.cuda.synchronize()
            a, b2 = ev(), ev()
            a.record()
            for _ in range(3):
                fn()
            b2.record()
            torch.cuda.synchronize()
            kern_ms[name] = a.elapsed_time(b2) / 3
        del dq, dk, dv
        fl_bwd = 2.5 * f_fwd(S)
        ach = fl_bwd / (kern_ms["bwd"] * 1e-3) / 1e12
        traffic = None   # dram__bytes_read+write of one attn_bwd_kernel launch at S=131072 (ncu --set full capture)
        tp = os.path.join(ROOT, "profiles", "ncu_attn_128k_r02.json")
        if S == S_TOTAL and os.path.exists(tp):
            traffic = json.load(open(tp))["attn_bwd_kernel"]["dram_total_bytes"]
        roof = {"bound": "tensor", "kernel": "attn_bwd_kernel<%s>" % ("fp16 operands" if prec == "fp16" else "bf16 operands"),
                "achieved": ach, "peak": peaks["sustained"],
                "unit": "TFLOP/s", "frac": ach / peaks["sustained"], "traffic": traffic,
                "traffic_note": "bytes per launch from profiles/ncu_attn_128k_r02.json; algorithmic minimum ~17 GB "
                                "(q,k,v,dout once + dq/dk/dv fp32 read-modify-write); tensor-bound, HBM < 2 % busy",
                "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step); burst=%.1f"
                % peaks["burst"],
                "fwd_kernel": {"achieved": f_fwd(S) / (kern_ms["fwd"] * 1e-3) / 1e12,
                               "frac": f_fwd(S) / (kern_ms["fwd"] * 1e-3) / 1e12 / peaks["sustained"],
                               "ms": kern_ms["fwd"]},
                "bwd_kernel_ms": kern_ms["bwd"], "share_of_step": (kern_ms["bwd"]) / ms}

    # ---- end-to-end through the public op with host buffers
    hout = torch.empty_like(hq).pin_memory()
    hdq, hdk, hdv = [torch.empty_like(hq).pin_memory() for _ in range(3)]

    def e2e_step():
        qd = hq.to(dev, non_blocking=True).requires_grad_(True)
        kd = hk.to(dev, non_blocking=True).requires_grad_(True)
        vd = hv.to(dev, non_blocking=True).requires_grad_(True)
        dod = hdo.to(dev, non_blocking=True)
        o = ra.ringattention(qd, kd, vd, None, None, **kwargs)
        o.backward(dod)
        hout.copy_(o.detach(), non_blocking=True)
        hdq.copy_(qd.grad, non_blocking=True)
        hdk.copy_(kd.grad, non_blocking=True)
        hdv.copy_(vd.grad, non_blocking=True)

    # the caller's persistent device staging buffers and copy streams (allocated once, outside the timed region)
    e2e_state = {}

    def e2e_setup():
        e2e_state["up"], e2e_state["down"] = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        e2e_state["dbuf"] = [[torch.empty_like(q) for _ in range(4)] for _ in range(2)]

    def e2e_pipelined(n):
        """Same copies per step, but double-buffered: two copy streams move step i+1's inputs up and step i-1's results
        down while step i's kernels run (what a caller streaming layers / micro-batches through the op would do).
        Results stay referenced until the main stream has waited for their download, so the allocator never hands a
        block that a copy is still reading to the next step (no record_stream, no allocation churn)."""
        main = torch.cuda.current_stream(dev)
        up, down, dbuf = e2e_state["up"], e2e_state["down"], e2e_state["dbuf"]
        up.wait_stream(main)
        up_done, free, down_done, keep = [None, None], [None, None], [None, None], [None, None]

        def upload(slot):
            with torch.cuda.stream(up):
                if free[slot] is not None:
                    up.wait_event(free[slot])
                for dst, src in zip(dbuf[slot], (hq, hk, hv, hdo)):
                    dst.copy_(src, non_blocking=True)
                up_done[slot] = up.record_event()
        upload(0)
        for i in range(n):
            s = i % 2
            if i + 1 < n:
                upload(1 - s)
            main.wait_event(up_done[s])
            if down_done[s] is not None:        # the results of step i-2 have left the device: their memory may be reused
                main.wait_event(down_done[s])
                keep[s] = None
            qd, kd, vd = [t.detach().requires_grad_(True) for t in dbuf[s][:3]]
            o = ra.ringattention(qd, kd, vd, None, None, **kwargs)
            o.backward(dbuf[s][3])
            free[s] = main.record_event()
            keep[s] = (o, qd, kd, vd)
            with torch.cuda.stream(down):
                down.wait_event(free[s])
                for dst, src in ((hout, o.detach()), (hdq, qd.grad), (hdk, kd.grad), (hdv, vd.grad)):
                    dst.copy_(src, non_blocking=True)
                down_done[s] = down.record_event()
        main.wait_stream(down)
        keep[0] = keep[1] = None

    e2e_step()
    n_e2e = K
    if not args.e2e_serial:
        e2e_setup()
        e2e_pipelined(2)            # warm-up of the pipelined path (untimed)
    barrier()
    a, b2 = ev(), ev()
    a.record()
    if not args.e2e_serial:
        e2e_pipelined(n_e2e)
    else:
        for _ in range(n_e2e):
            e2e_step()
    b2.record()
    barrier()
    ms_e2e = a.elapsed_time(b2) / n_e2e
    if world > 1:
        tm = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms_e2e = float(tm.item())
    bytes_in = 4 * hq.numel() * 2
    bytes_out = 4 * hq.numel() * 2

    # ---- VQGAN encode: 16 frames of 256x256 (replicas: every rank encodes its own clip, no collective)
    vq = None
    if not args.no_vqgan:
        try:
            vq = bench_vqgan(dev, peaks, world, rank, with_cpu=not args.no_cpu_baseline)
        except Exception as e:      # noqa: BLE001  (the attention line must still be printed)
            vq = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}

    if rank == 0:
        total_flops = 3.5 * f_fwd(S)
        line = {
            "metric": METRIC, "value": S / (LAYERS * ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(S), "sharding": "sequence over %d GPU(s)" % world,
                       "layout": args.layout, "precision": args.precision or ra._DEFAULT_PRECISION, "l2": "inputs (>=1 GiB per tensor at N=1) larger than the 126 MB L2",
                       "tokens_per_s_definition": "S / (32 layers * t_step), attention only"},
            "tflops_per_gpu": total_flops / (ms * 1e-3) / 1e12 / world,
            "frac_of_bf16_peak_per_gpu": total_flops / (ms * 1e-3) / 1e12 / world / peaks["sustained"],
            "e2e": {"value": S / (LAYERS * ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
                    "steps": n_e2e,
                    "copies": "serialised with the kernels" if args.e2e_serial else
                    "double-buffered: step i+1's uploads and step i-1's downloads overlap step i's kernels; all copies "
                    "(first upload and last download included) inside the timed region"},
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "reference_probe": probe_reference(),
        }
        if parity:
            line["parity"] = parity
        if roof:
            line["roofline"] = roof
        if vq:
            line["vqgan"] = vq
        if not args.no_cpu_baseline:
          try:
            cores = min(len(os.sched_getaffinity(0)), 32)   # more threads only add contention at this size
            torch.set_num_threads(cores)
            cpu_sample_step(1024, 1024, 4, chunk=512)       # warm the thread pool
            dt, fl = cpu_sample_step(4096, 4096, 32, chunk=1024)
            line["cpu_baseline"] = {
                "value": 4096 / (LAYERS * dt), "unit": UNIT, "cores": cores, "kind": "port",
                "gflops": fl / dt / 1e9,
                "sample": "oracle blockwise fwd+bwd (torch CPU fp32) of one full layer at S=4096 (BASELINE configs[0]; "
                          "32 heads, causal); %.1f s of CPU work; tokens/s = 4096 / (32 layers * t)" % dt}
          except Exception as e:      # noqa: BLE001
            line["cpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
