#!/usr/bin/env python
"""bench.py - H-Codec-2.0 encode + RVQ + decode throughput on B200 (BASELINE.json configs[1]).

A "step" = one pass of the hot path (Codec.encode -> Codec.decode) over one synthetic batch of
B=64 clips x 10 s at the shipped 48 kHz configuration (480 000 samples / clip, 125 tokens / stream),
seeded random weights of the shipped architecture (large_12.5hz_config.yaml).  No pretrained
weights / datasets exist offline, hence `data: synthetic`.

  python bench.py --gpus 1 --steps 5 --warmup 3            # our arm (CUDA kernels via the C ABI)
  python bench.py --impl reference --steps 2 --warmup 1     # the reference's CPU path (oracle port)
  torchrun ... bench.py --gpus N ...                        # one rank per GPU, weak scaling
  python bench.py --steps 5 --warmup 3 --dump-outputs DIR   # also write the last timed step's outputs as DIR/<name>.npy

Prints ONE JSON line (see README / DESIGN.md "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "hcodec2_encode_rvq_decode_samples_per_s"
UNIT = "samples/s"
# SURVEY 8(d): algorithmic FLOPs per 50 Hz frame (multiply-add = 2), encoder+semantic+RVQ+decoder
FLOP_PER_FRAME = 2245.8e6

H2_FULL = dict(
    sampling_rate=48000,
    encoder_config=dict(dim=1536, intermediate_dim=4608, dimension=512, n_fft=1920, hop_length=960,
                        convnext_layers=24, transformer_layers=2, target_frame_rate=12.5, causal=False),
    decoder_config=dict(input_channels=1024, dim=1536, intermediate_dim=4608, convnext_layers=32, n_fft=1920,
                        hop_length=960, transformer_layers=2, target_frame_rate=12.5, causal=False),
    quantizer_config=dict(dim=512, codebook_size=1024, num_quantizers=16, decay=0.99, kmeans_init=True,
                          kmeans_iters=50, quantize_dropout=False),
    semantic_encoder_config=dict(input_channels=768, encode_channels=1536, out_channels=512,
                                 channel_ratios=[1, 1, 1], strides=[2, 1, 2]),
    semantic_decoder_config=dict(code_dim=512, output_channels=768, decode_channels=1536,
                                 channel_ratios=[1, 1, 1], strides=[2, 1, 2]),
)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def random_init_(model, seed: int):
    """Seeded random weights of the shipped architecture, generated on the module's device."""
    dev = next(model.parameters()).device
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "rnn." in name:
                H = p.shape[-1] if p.dim() == 2 else p.shape[0] // 4
                p.copy_((torch.rand(p.shape, generator=g, device=dev) * 2 - 1) / H ** 0.5)
            elif name.endswith("layer_scale_1.scale") or name.endswith("layer_scale_2.scale"):     # H-Codec-1.5 mimi LayerScale
                p.copy_(0.35 * (1 + 0.2 * torch.randn(p.shape, generator=g, device=dev)))
            elif name.endswith("weight_g"):
                p.copy_(1 + 0.2 * torch.rand(p.shape, generator=g, device=dev))
            elif name.endswith("gamma"):
                n_layers = 24 if name.startswith("encoder.") else 32
                p.copy_((1.0 / n_layers) * (1 + 0.2 * torch.randn(p.shape, generator=g, device=dev)))
            elif p.dim() >= 2:
                fan = p[0].numel()
                p.copy_(torch.randn(p.shape, generator=g, device=dev) * fan ** -0.5)
            elif "norm" in name and name.endswith("weight") or name.endswith("prior_net.7.weight"):
                p.copy_(1 + 0.1 * torch.randn(p.shape, generator=g, device=dev))
            else:
                p.copy_(0.05 * torch.randn(p.shape, generator=g, device=dev))
        for q in (model.quantizer, model.semantic_quantizer):
            cb = torch.stack([torch.randn(q.codebook_size, q.dim, generator=g, device=dev) * 0.35 * 0.85 ** i
                              for i in range(q.num_quantizers)], 0)
            q.set_codebooks(cb)
    model._w = None
    model._engine = None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


LM_CFG = dict(num_tasks=3, task_map=dict(se=0, tse=1, rtse=2), feats_dim=768,
              llm_base_config=dict(cond_dim=80, global_size=4096, semantic_size=8192, hidden_size=512, num_layers=12,
                                   num_attention_heads=8, dropout_p=0.1, max_position_embeddings=4096, label_smoothing=0.1))
REF_THREADS = 32        # pinned host thread count of every CPU leg (VERDICT r01 weak item 14: no per-run calibration)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_threads():
    n = min(REF_THREADS, host_cores())
    torch.set_num_threads(n)
    return n


class Ctx:
    """One process per GPU (torchrun env); NCCL only for the barrier, the max-over-ranks timing and the token gather."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dist = None
        self.t0 = time.perf_counter()
        # wall-clock budget for the optional legs (the driver's per-N limit in the scaling run is 870 s): a leg that would start
        # after the budget is recorded as skipped instead of endangering the headline line
        self.budget_s = float(os.environ.get("QB_BENCH_BUDGET_S", "540"))
        if self.world > 1:
            import torch.distributed as dist_
            if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
                os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the single JSON line
            dist_.init_process_group("nccl", device_id=self.dev)
            self.dist = dist_

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        """K steps bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks -> ms / step"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.dist is not None:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps

    def over_budget(self):
        """True once the invocation has used its wall-clock budget; rank 0 decides for every rank (the legs contain barriers)."""
        over = time.perf_counter() - self.t0 > self.budget_s
        if self.dist is not None:
            t = torch.tensor([1 if over else 0], device=self.dev, dtype=torch.int32)
            self.dist.broadcast(t, src=0)
            over = bool(int(t))
        return over

    def elapsed_s(self):
        return time.perf_counter() - self.t0

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


DUMP_BUDGET_BYTES = 64 * 10 ** 6
NPY_HEADER_BYTES = 256          # allowance per file for the .npy header (numpy writes 128 bytes for these shapes)


def dump_outputs(out_dir, arrays, budget=DUMP_BUDGET_BYTES, seed=0):
    """Write each named tensor as <out_dir>/<name>.npy in float32 (the integer codes are < 2^24, exact in float32), at most
    `budget` bytes in all, so that two builds run with the same arguments can be compared output for output.  The smallest
    tensors are written whole; one that does not fit what is left is replaced by a seeded, sorted sample of its rows
    (first dimension), with the sampled row indices beside it as <name>_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = budget
    for name, t in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        a = t.detach().float().cpu()
        rows_path = os.path.join(out_dir, f"{name}_rows.npy")
        if os.path.exists(rows_path):           # from an earlier dump into the same directory
            os.remove(rows_path)
        if a.numel() * 4 + NPY_HEADER_BYTES > left:
            n, row_bytes = a.shape[0], a[0].numel() * 4
            k = (left - 2 * NPY_HEADER_BYTES) // (row_bytes + 8)
            if k < 1:
                raise ValueError(f"dump_outputs: no row of {name} {tuple(a.shape)} fits the {budget} byte budget")
            rows = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values
            a = a[rows]
            np.save(rows_path, rows.double().numpy())
            left -= rows.numel() * 8 + NPY_HEADER_BYTES
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())
        left -= a.numel() * 4 + NPY_HEADER_BYTES


def run_leg(ctx, sec, name, fn):
    """One optional leg of the bench line: never takes the headline down, never starts after the wall-clock budget."""
    if ctx.over_budget():
        sec[name] = dict(skipped=f"wall-clock budget of {ctx.budget_s:.0f} s reached after {ctx.elapsed_s():.0f} s (QB_BENCH_BUDGET_S)")
        return
    t0 = time.perf_counter()
    try:
        sec[name] = fn()
    except Exception as e:
        sec[name] = dict(error=repr(e))
        if torch.cuda.is_available():
            torch.cuda.synchronize()
    if isinstance(sec[name], dict):
        sec[name]["leg_wall_s"] = round(time.perf_counter() - t0, 1)


# ------------------------------------------------------------------------------------------------ CPU legs (oracle port)
def cpu_codec(sd_cpu, cfg, wav, feat, want_codes=False):
    """The reference's own PyTorch CPU path (oracle port, pinned bit-exact against the reference modules) on this box's
    host cores: encode + RVQ + decode of the given clips.  -> (samples/s, seconds, taps, codes)"""
    from oracle import hcodec2
    cpu_threads()
    taps = {} if want_codes else None
    t0 = time.perf_counter()
    ac, sc = hcodec2.codec_encode(sd_cpu, cfg, wav, feat, taps=taps)
    hcodec2.codec_decode(sd_cpu, cfg, ac, sc)
    dt = time.perf_counter() - t0
    return wav.numel() / dt, dt, taps, (ac, sc)


def cpu_lm_generate(task, Bc=4, T=250):
    """oracle port of LLM_SFT.generate (greedy) on the host: Bc sequences, the benchmarked prefix + 283 cached steps"""
    from oracle import llama
    n = cpu_threads()
    sd = llama.make_lm_state_dict(LM_CFG, 7, 2.0)
    g = torch.Generator().manual_seed(9)
    mix = torch.randn(Bc, T, 768, generator=g)
    enr = torch.randn(Bc, T, 768, generator=g) if task == "tse" else None
    t0 = time.perf_counter()
    llama.sft_generate(sd, LM_CFG, task, enr, mix, T)
    dt = time.perf_counter() - t0
    return dict(value=Bc * 283 / dt, unit="tokens/s", cores=n, host_cores=host_cores(), kind="port",
                sample=f"{Bc} sequences x 283 tokens (prefix {503 if task == 'tse' else 252}, {dt:.1f} s), oracle port pinned against "
                       "transformers.LlamaModel, torch CPU fp32")


def run_reference(args, cfg):
    """--impl reference: the reference's CPU path alone (oracle port), same metric / config, rank 0 only; the LM legs ride
    in `secondary` like on the GPU arm."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import weights
    sd = weights.make_h2_state_dict(cfg, 0)
    clips = args.ref_clips
    T = int(args.seconds * cfg["sampling_rate"])
    T -= T % 3840
    g = torch.Generator().manual_seed(7)
    wav = 0.1 * torch.randn(clips, T, generator=g)
    f = torch.randn(clips, 768, T // 960, generator=g)
    feat = torch.sign(f) * f.abs() ** 0.3
    times = []
    for i in range(args.warmup + args.steps):
        _, dt, _, _ = cpu_codec(sd, cfg, wav, feat)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = clips * T / (ms / 1e3)
    n = cpu_threads()
    sample = (f"{clips} clip(s) x {args.seconds:g} s per step, oracle port of the reference (pinned bit-exact against the "
              f"reference modules), torch CPU fp32, {n} threads of {host_cores()} host cores")
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=f"HCodec-2.0 (48 kHz shipped config) {args.seconds:g} s clips, encode+RVQ+decode",
                            batch_per_step=clips, samples_per_clip=T, cpu_threads=n, host_cores=host_cores()),
                cpu_baseline=dict(value=value, unit=UNIT, cores=n, host_cores=host_cores(), kind="port", sample=sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    if args.workload == "all":
        sec = {}
        for name, task in (("lm_sr", "se"), ("lm_tse", "tse")):
            c = cpu_lm_generate(task)
            sec[name] = dict(metric=f"unise_{'sr' if task == 'se' else 'tse'}_arlm_generate_tokens_per_s", value=c["value"],
                             unit="tokens/s", impl="reference", cpu_baseline=c)
        line["secondary"] = sec
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ UniSE AR-LM
def build_lm(dev):
    from unified_audio_b200.llm import LLM_SFT
    m = LLM_SFT(num_tasks=3, task_map=LM_CFG["task_map"], feats_dim=768, llm_base_config=LM_CFG["llm_base_config"]).to(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    with torch.no_grad():       # x2-gain weights so the logits are not near-uniform (SURVEY 8d)
        for n, p in m.named_parameters():
            if p.dim() >= 2 and "embedding" not in n:
                p.copy_(torch.randn(p.shape, generator=g, device=dev) * (2.0 / p.shape[-1] ** 0.5))
            elif p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, device=dev))
            else:
                p.copy_(1 + 0.1 * torch.randn(p.shape, generator=g, device=dev))
    m._w = None
    return m


def lm_decode_bytes(B, P, world, chunks=None):
    """SURVEY 8(d) algorithmic bytes of one generation: per decode step the fp32-equivalent layer weights (4 B / parameter:
    the packed fp16 hi/lo groups are the same size) + the active head slice + the fp32 KV read / write of every sequence."""
    w_layers = 12 * (4 * 512 * 512 + 3 * 512 * 2048) * 4
    head = 33 * 4096 * 512 * 4 + 250 * 8192 * 512 * 4
    kv = sum(B * 2 * 12 * 512 * 4 * (P + i + 1) for i in range(283))
    # B is the whole-job batch; the weights are streamed once per generation chunk (<= 32 sequences) on every rank
    return (chunks if chunks is not None else world) * (283 * w_layers + head) + kv


def bench_lm_generate(args, ctx, m, task, B_local, total_batch=None, with_cpu=False, steps=None):
    """UniSE AR-LM greedy generate (llm_sft.py:93-195): prefill (252 SR / 503 TSE positions) + 33 + 250 cached steps.
    tokens/s counts generated tokens (283 per sequence, SURVEY 8d).  `total_batch` (strong scaling): the job's batch is
    fixed and split over the ranks; generate() walks it in chunks of <= 32 sequences."""
    from unified_audio_b200 import ops
    from unified_audio_b200.parallel import gather_tokens
    T = 250
    steps = steps or args.steps
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    if total_batch is not None:
        from unified_audio_b200.parallel import shard_range
        lo, hi = shard_range(total_batch, rank, world)
        B_local = hi - lo
    B_all = total_batch if total_batch is not None else B_local * world
    g = torch.Generator().manual_seed(3000 + rank if task == "se" else 4001 + rank)
    mix_h = torch.randn(B_local, T, 768, generator=g).pin_memory()
    enr_h = torch.randn(B_local, T, 768, generator=g).pin_memory() if task == "tse" else None
    mix = mix_h.to(dev)
    enr = enr_h.to(dev) if enr_h is not None else None
    gather_buf = {}

    def step(src, esrc):
        gi, si = m.generate(task, esrc, esrc, src, src, do_sample=False)
        if ctx.dist is not None:
            gather_tokens(torch.cat([gi, si], 1), B_all, buffers=gather_buf)
        return gi, si

    for _ in range(max(args.warmup, 2) if steps == args.steps else 1):
        step(mix, enr)
    ops.launch_count_reset()
    ms = ctx.timed(lambda: step(mix, enr), steps)
    launches = ops.launch_count() // steps
    ids_h = torch.empty(B_local, 32 + T, dtype=torch.int64).pin_memory()

    def e2e_step():
        gi, si = step(mix_h.to(dev, non_blocking=True), enr_h.to(dev, non_blocking=True) if enr_h is not None else None)
        ids_h[:, :32].copy_(gi, non_blocking=True)
        ids_h[:, 32:].copy_(si, non_blocking=True)
    ms_e2e = ctx.timed(e2e_step, steps)
    P = 503 if task == "tse" else 252
    peaks = load_peaks()
    chunks_local = -(-B_local // 32)
    if ctx.dist is not None:
        tch = torch.tensor([chunks_local], device=dev)
        ctx.dist.all_reduce(tch)
        chunks_all = int(tch)
    else:
        chunks_all = chunks_local
    gbs = lm_decode_bytes(B_all, P, world, chunks_all) / (ms * 1e-3) / 1e9
    name = "sr" if task == "se" else "tse"
    out = dict(metric=f"unise_{name}_arlm_generate_tokens_per_s", value=B_all * 283 / (ms * 1e-3), unit="tokens/s", n_gpus=world,
               steps=steps, ms_per_step=ms, higher_is_better=True, scaling="strong" if total_batch is not None else "weak",
               dtype="f16x3 split tensor-core (fp32-grade), f32 accumulate / f32 KV cache", data="synthetic",
               config=dict(workload=f"UniSE {'SR' if task == 'se' else 'TSE (enrollment prefix)'} AR-LM greedy generate: prefill {P} + 33 + 250 cached "
                                    f"steps, KV <= {P + 283}", batch=B_all, batch_per_gpu=B_local, semantic_length=T,
                           parallelism=f"dp{world} (sequences sharded, one NCCL all_gather of ids)",
                           chunks=f"{chunks_local} chunk(s) of <= {m.chunk} sequences per GPU on {min(m.lanes, chunks_local)} concurrent lane(s) "
                                  "(own stream / KV cache / captured graphs each; profiles/r02_lm_lanes_ab.md)",
                           launches="decode steps replay captured CUDA graphs (8 steps x 62 kernels each); gpu_launches counts the eager launches "
                                    "(prefill, adapter) per generation"),
               e2e=dict(value=B_all * 283 / (ms_e2e * 1e-3), unit="tokens/s", ms_per_step=ms_e2e,
                        h2d_bytes_per_step=int(mix_h.numel() * 4 * (2 if task == "tse" else 1)) * world, d2h_bytes_per_step=B_all * 282 * 8),
               gpu_launches=int(launches),
               roofline=dict(bound="hbm", achieved=gbs, peak=peaks["hbm"] * world, unit="GB/s", frac=gbs / (peaks["hbm"] * world), traffic=None,
                             kernel="decode step (lm_skinny<QKV|RESID|GATEUP|HEAD> + lm_decode_attn2): algorithmic bytes = 4 B/param layer weights + head "
                                    "slice + fp32 KV read/write per step (SURVEY 8d), over the whole generate incl. prefill",
                             peak_source=f"{peaks['src']} HBM copy bandwidth x {world} GPU(s)"))
    if with_cpu and rank == 0:
        out["cpu_baseline"] = cpu_lm_generate(task)
    return out


def bench_lm_forward(args, ctx, m):
    """teacher-forced UniSE LM forward (llm_sft.py:37-89): prefix 252 + 284 code tokens per sequence, logits over the
    12291-entry vocabulary, loss + accuracy - the "AR-LM forward" of north_star.  Tensor-bound; every GEMM is a 3-term split."""
    from unified_audio_b200 import ops
    B, T = 32, 250
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    mix_h = torch.randn(B, T, 768, generator=torch.Generator().manual_seed(100 + rank)).pin_memory()
    mix = mix_h.to(dev)
    gt = torch.Generator().manual_seed(7 + rank)
    gids_h = torch.randint(0, 4096, (B, 32), generator=gt).pin_memory()
    sids_h = torch.randint(0, 8192, (B, T), generator=gt).pin_memory()
    gids, sids = gids_h.to(dev), sids_h.to(dev)
    L = 2 + T + 32 + 1 + T + 1            # task + mix_sos + feats, then sos/global/sos/semantic (+ eos target)
    fwd = lambda a, b_, c_: m("se", None, None, a, a, b_, c_)
    for _ in range(max(args.warmup, 3)):
        fwd(mix, gids, sids)
    ops.launch_count_reset()
    ms = ctx.timed(lambda: fwd(mix, gids, sids), args.steps)
    launches = ops.launch_count() // args.steps

    def e2e_fwd():
        loss, acc = fwd(mix_h.to(dev, non_blocking=True), gids_h.to(dev, non_blocking=True), sids_h.to(dev, non_blocking=True))
        loss.cpu(); acc.cpu()
    ms_e2e = ctx.timed(e2e_fwd, args.steps)
    peaks = load_peaks()
    per_tok = 12 * 2 * (4 * 512 * 512 + 3 * 512 * 2048)
    flops = world * B * (L * per_tok + 12 * 4 * 512 * L * L / 2 + 2 * 768 * 512 * T + (T + 34) * 2 * 512 * 12291)
    tf = flops / (ms * 1e-3) / 1e12
    return dict(
        metric="unise_lm_forward_tokens_per_s", value=world * B * L / (ms * 1e-3), unit="tokens/s", n_gpus=world,
        steps=args.steps, ms_per_step=ms, higher_is_better=True, scaling="weak",
        dtype="f16x3 split tensor-core (fp32-grade), f32 accumulate", data="synthetic",
        config=dict(workload=f"UniSE LM teacher-forced forward, {B} sequences x {L} positions per GPU, logits + loss", batch=B * world,
                    positions=L, parallelism=f"dp{world}"),
        e2e=dict(value=world * B * L / (ms_e2e * 1e-3), unit="tokens/s", ms_per_step=ms_e2e,
                 h2d_bytes_per_step=int(mix_h.numel() * 4 + gids_h.numel() * 8 + sids_h.numel() * 8) * world, d2h_bytes_per_step=8 * world),
        gpu_launches=int(launches),
        roofline=dict(bound="tensor", achieved=tf, peak=peaks["tf_sus"] * world, unit="TFLOP/s", frac=tf / (peaks["tf_sus"] * world),
                      traffic=None, kernel="whole forward, algorithmic FLOPs (every GEMM and the attention issued 3x: ceiling 1/3)"))


# ------------------------------------------------------------------------------------------------ H-Codec-2.0
def build_codec(cfg, dev, precision):
    from unified_audio_b200.codec import Codec
    model = Codec(cfg["encoder_config"], cfg["decoder_config"], cfg["quantizer_config"],
                  cfg["semantic_encoder_config"], cfg["semantic_decoder_config"], precision=precision).to(dev)
    random_init_(model, 1234)
    return model


def synth_batch(cfg, B, seconds, seed):
    T = int(seconds * cfg["sampling_rate"])
    T -= T % 3840
    g = torch.Generator().manual_seed(seed)
    wav_h = (0.1 * torch.randn(B, T, generator=g)).pin_memory()
    f = torch.randn(B, 768, T // 960, generator=g)
    feat_h = (torch.sign(f) * f.abs() ** 0.3).pin_memory()
    return wav_h, feat_h, T


def bench_codec_strong(args, ctx, model, cfg, total):
    """BASELINE configs[4] as written: `total` clips sharded over the ranks (strong scaling); each rank walks its shard in chunks
    of <= 64 clips through the captured round trip; one token all-gather per step."""
    from unified_audio_b200.parallel import gather_tokens, shard_range
    lo, hi = shard_range(total, ctx.rank, ctx.world)
    n_local = hi - lo
    chunk = min(64, n_local)
    wav_h, feat_h, T = synth_batch(cfg, chunk, args.seconds, 5000 + ctx.rank)
    wav_d, feat_d = wav_h.to(ctx.dev), feat_h.to(ctx.dev)
    graphed = model.graphed("roundtrip", wav_d, feat_d)
    n_chunks = -(-n_local // chunk)
    toks = torch.zeros(n_local, 2, 16, T // 3840, dtype=torch.int64, device=ctx.dev)
    gbuf = {}

    def step():
        for c in range(n_chunks):
            ac, sc, rec = graphed()
            n = min(chunk, n_local - c * chunk)
            toks[c * chunk:c * chunk + n, 0].copy_(ac[:n])
            toks[c * chunk:c * chunk + n, 1].copy_(sc[:n])
        if ctx.dist is not None:
            gather_tokens(toks, total, buffers=gbuf)
    step()
    ms = ctx.timed(step, max(2, min(args.steps, 3)))
    return dict(metric=METRIC, value=total * T / (ms * 1e-3), unit=UNIT, n_gpus=ctx.world, ms_per_step=ms, scaling="strong",
                config=dict(workload=f"HCodec-2.0 batch={total} x {args.seconds:g} s (BASELINE configs[4]) sharded over {ctx.world} GPU(s)",
                            clips_per_gpu=n_local, chunk=chunk, chunks_per_step=n_chunks),
                note="last chunk of a shard that is not a multiple of the chunk size is computed in full and trimmed" if n_local % chunk else None)


def init_ssl_(fe, dev, seed):
    """random-init weights of an SSL front end (HuBERT-base / WavLM-base-plus architecture; no checkpoints offline)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    with torch.no_grad():
        for n, p in fe.named_parameters():
            if n.endswith("original0"):
                continue
            if p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, device=dev) * (1.5 / p[0].numel()) ** 0.5)
            elif "norm" in n and n.endswith("weight"):
                p.copy_(1 + 0.1 * torch.randn(p.shape, generator=g, device=dev))
            else:
                p.copy_(0.05 * torch.randn(p.shape, generator=g, device=dev))
        v = fe.encoder.pos_conv_embed.conv.parametrizations.weight.original1
        fe.encoder.pos_conv_embed.conv.parametrizations.weight.original0.copy_(v.pow(2).sum((0, 1), keepdim=True).sqrt() * 0.5)
    fe._w = None
    return g


def bench_tokenize(args, ctx, model, cfg):
    """HCodecTokenizer.tokenize-shaped leg (audio_tokenizer.py:68-74): raw 48 kHz waveform -> pad_wav -> Resample + HuBERT-base (mean of
    13 hidden states, |x|^0.3) -> Codec.encode -> codes, everything on the device (SURVEY 8f.2 / 8f.3)."""
    from unified_audio_b200 import ops
    from unified_audio_b200.ssl import HCodecTokenizer, HUBERT_BASE, SSLFrontEnd
    dev = ctx.dev
    fe = SSLFrontEnd(HUBERT_BASE, in_rate=48000, compress=True).to(dev)
    g = init_ssl_(fe, dev, 99)
    tok = HCodecTokenizer(model, fe, cfg["sampling_rate"], cfg["encoder_config"]["target_frame_rate"])
    B = args.batch
    T = int(args.seconds * cfg["sampling_rate"]) - 700               # not a multiple of the hop: pad_wav has work to do
    wav = 0.1 * torch.randn(B, T, device=dev, generator=g)
    for _ in range(2):
        tok.tokenize(wav)
    ops.launch_count_reset()
    ms = ctx.timed(lambda: tok.tokenize(wav), 3)
    launches = ops.launch_count() // 3
    # SSL front end algorithmic FLOPs per 16 kHz second: conv stack 4.9 G + 50 frames x (12 layers x 14.2 M + pos conv 9.4 M + proj 0.8 M) x 2
    frames = B * (T + 700) // 960
    ssl_flops = B * (T + 700) / 48000 * (4.9e9 + 50 * 2 * (12 * 7.08e6 + 4.7e6 + 0.4e6))
    enc_flops = frames * (896.1e6 + 105.0e6 + 8.4e6)
    tf = ctx.world * (ssl_flops + enc_flops) / (ms * 1e-3) / 1e12
    peaks = load_peaks()
    del tok, fe
    return dict(metric="hcodec2_tokenize_samples_per_s", value=ctx.world * B * T / (ms * 1e-3), unit=UNIT, ms_per_step=ms, n_gpus=ctx.world,
                config=dict(workload=f"HCodecTokenizer.tokenize: {B} clips x {T} samples @ 48 kHz -> pad_wav -> Resample + HuBERT-base features -> "
                                     "Codec.encode (wav in, codes out)", precision_policy=f"codec {args.precision}; SSL front end 3-term split"),
                gpu_launches=int(launches),
                roofline=dict(bound="tensor", achieved=tf, peak=peaks["tf_sus"] * ctx.world, unit="TFLOP/s", frac=tf / (peaks["tf_sus"] * ctx.world),
                              kernel="whole tokenize path, algorithmic FLOPs (SSL conv stack + 12 encoder layers + codec encoder / semantic encoder / RVQ)"))


def bench_unise_sr(args, ctx, lm):
    """BASELINE configs[2] as written - "UniSE SR: WavLM feats + AR-LM decode + codec decode, batch=32" - through the reference's
    caller surface (unise.Model.enhance == the body of test_step, U/model/model.py:174-193): one utterance of 32 x 5 s @ 16 kHz per GPU ->
    wrap-pad + segmenting -> WavLM-base-plus mean hidden state -> LLM_SFT.generate (greedy, 33 + 250 steps) -> BiCodec.detokenize ->
    waveform, everything on the device.  The decoder is BiCodec, the codec UniSE actually feeds (SURVEY 8f.1).  Stage split by CUDA events."""
    from unified_audio_b200 import ops
    from unified_audio_b200.bicodec import BICODEC_CONFIG, BiCodec
    from unified_audio_b200.ssl import SSLFrontEnd, WAVLM_BASE_PLUS
    from unified_audio_b200.unise import SEG_LEN, BiCodecTokenizer, Model
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    wavlm = SSLFrontEnd(WAVLM_BASE_PLUS, in_rate=16000, compress=False).to(dev)
    init_ssl_(wavlm, dev, 98)
    codec = BiCodec(BICODEC_CONFIG).to(dev)
    init_bicodec_(codec, dev)
    model = Model(None, tokenizer=BiCodecTokenizer(codec), dnn=lm, semantic_model=wavlm)
    B = 32
    T = B * SEG_LEN - 1234                                   # the last segment is wrap-padded
    g = torch.Generator().manual_seed(3200 + rank)
    src_h = (0.1 * torch.randn(1, T, generator=g)).pin_memory()
    src = src_h.to(dev)
    out_h = torch.empty(T).pin_memory()
    for _ in range(2):
        model.enhance("se", None, src)
    steps = min(args.steps, 5)
    ops.launch_count_reset()
    ms = ctx.timed(lambda: model.enhance("se", None, src), steps)
    launches = ops.launch_count() // steps

    def e2e_step():
        out_h.copy_(model.enhance("se", None, src_h.to(dev, non_blocking=True)), non_blocking=True)
    ms_e2e = ctx.timed(e2e_step, steps)
    # stage split (one more step, events between the stages)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    ev[0].record()
    seg = model._segments(src)
    seg = seg / src.abs().max(dim=-1, keepdim=True)[0]
    feats = model.extract_semantic_features(seg)
    ev[1].record()
    gids, sids = lm.generate("se", None, None, model.mel_like(seg), feats, do_sample=False)
    ev[2].record()
    model._detok(gids, sids, T)
    ev[3].record()
    torch.cuda.synchronize()
    split = dict(wavlm_ms=ev[0].elapsed_time(ev[1]), lm_generate_ms=ev[1].elapsed_time(ev[2]), bicodec_ms=ev[2].elapsed_time(ev[3]))
    del model, codec, wavlm
    return dict(metric="unise_sr_pipeline_samples_per_s", value=world * T / (ms * 1e-3), unit="samples/s (16 kHz)", n_gpus=world, steps=steps,
                ms_per_step=ms, higher_is_better=True, scaling="weak", data="synthetic", tokens_per_s=world * B * 283 / (ms * 1e-3),
                config=dict(workload=f"UniSE SR test_step: 1 utterance of {T} samples ({B} x 5 s segments) per GPU: wrap-pad -> WavLM-base-plus "
                                     "features -> AR-LM greedy generate (252 prefix + 283 steps) -> BiCodec detokenize -> waveform",
                            batch_per_gpu=B, precision="WavLM / LM / BiCodec: 3-term split (fp32-grade)"),
                stage_split=split, gpu_launches=int(launches),
                e2e=dict(value=world * T / (ms_e2e * 1e-3), unit="samples/s (16 kHz)", ms_per_step=ms_e2e, h2d_bytes_per_step=T * 4 * world,
                         d2h_bytes_per_step=T * 4 * world))


def bench_h15(args, ctx):
    """SURVEY 8f.4: H-Codec-1.5 adaptive frame-rate codec, shipped config (conf/config_adaptive_v3.yaml), `batch` clips x `seconds` s at
    16 kHz: encode (SEANet + semantic encoder + similarity alignment + 2 x 32-layer query-token aggregators + RVQ + length packing)
    -> decode (unpack + de-aggregate + 32-layer bottleneck transformer + decoder).  Launched kernel by kernel: the sequence lengths
    T + G depend on the batch's largest group count (one host read per encode / decode, as in the reference)."""
    from unified_audio_b200 import ops
    from unified_audio_b200.codec_h15 import CodecH15, H15
    dev = ctx.dev
    model = CodecH15(precision=args.precision if args.precision in ("mixed", "accurate", "mixed_dec16", "fast") else "mixed", _cfg=dict(H15)).to(dev)
    random_init_(model, 4321)
    B, T50 = args.batch, int(args.seconds * 50)
    T50 -= T50 % 2
    g = torch.Generator(device=dev).manual_seed(1500 + ctx.rank)
    wav = 0.1 * torch.randn(B, 1, T50 * 320, generator=g, device=dev)
    # semantic features in runs (mean 7.7 frames) + noise (so that tokens of 1..8 frames occur), compressed like the SSL front end's output
    ids = torch.cumsum((torch.rand(B, T50, generator=g, device=dev) < 0.13).long(), 1)                     # frame -> run index
    base = torch.randn(B, T50 + 1, 1024, generator=g, device=dev)
    f = torch.gather(base, 1, ids[..., None].expand(-1, -1, 1024)).transpose(1, 2) + 0.25 * torch.randn(B, 1024, T50, generator=g, device=dev)
    feat = (torch.sign(f) * f.abs() ** 0.3).contiguous()
    del base, f

    def step():
        out = model.encode(wav, feat)
        return out, model.decode(out["acoustic_codes"], out["semantic_codes"])
    # one counted step: GEMM FLOPs as the algorithm states them (2 M N K, one pass) + attention (4 L^2 C per layer and item)
    flops = [0.0]
    real_gemm, real_att, real_att_tc, real_att5 = ops.gemm, ops.attention_hd, ops.attention_tc, ops.attention_umma

    def count_gemm(a, w, n, **kw):
        flops[0] += 2.0 * kw["a_batch"] * kw["m_per_batch"] * n * kw.get("taps", 1) * (kw.get("a_cols") or kw["a_ld"])
        return real_gemm(a, w, n, **kw)

    def count_att(qkv, B_, T_, heads, hd, *a):
        flops[0] += 4.0 * B_ * T_ * T_ * heads * hd
        return real_att(qkv, B_, T_, heads, hd, *a)

    def count_att_tc(qkv, B_, T_, heads, *a):
        flops[0] += 4.0 * B_ * T_ * T_ * heads * 64
        return real_att_tc(qkv, B_, T_, heads, *a)
    def count_att5(qkv, B_, T_, heads, hd, *a, **kw):
        flops[0] += 4.0 * B_ * T_ * T_ * heads * hd
        return real_att5(qkv, B_, T_, heads, hd, *a, **kw)
    ops.gemm, ops.attention_hd, ops.attention_tc, ops.attention_umma = count_gemm, count_att, count_att_tc, count_att5
    try:
        out, rec = step()
    finally:
        ops.gemm, ops.attention_hd, ops.attention_tc, ops.attention_umma = real_gemm, real_att, real_att_tc, real_att5
    torch.cuda.synchronize()
    from unified_audio_b200 import adaptive
    _, lens = adaptive.extract_lengths(out["acoustic_codes"], model.codebook_size)
    n_tok = (lens > 0).sum(1).float()
    step()
    step()
    ops.launch_count_reset()
    k15 = max(2, min(args.steps, 3))
    ms_a = ctx.timed(step, k15)
    launches = ops.launch_count() // k15
    ms_b = ctx.timed(step, k15)                 # ~960 eager launches + two host reads per step: the first timed pass still grows the allocator
    ms = min(ms_a, ms_b)
    peaks = load_peaks()
    tf = ctx.world * flops[0] / (ms * 1e-3) / 1e12
    n_samples = B * T50 * 320
    # e2e: inputs from pinned host memory, length-packed codes + waveform read back, every step
    wav_h, feat_h = wav.cpu().pin_memory(), feat.cpu().pin_memory()
    out_h = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in (out["acoustic_codes"], out["semantic_codes"], rec)]

    def e2e_step():
        o, r = None, None
        w, f = wav_h.to(dev, non_blocking=True), feat_h.to(dev, non_blocking=True)
        o = model.encode(w, f)
        r = model.decode(o["acoustic_codes"], o["semantic_codes"])
        for dst, src in zip(out_h, (o["acoustic_codes"], o["semantic_codes"], r)):
            if dst.shape == src.shape:
                dst.copy_(src, non_blocking=True)
            else:                                   # the group count G of a batch is data dependent: same batch, same G
                dst.resize_(src.shape).copy_(src, non_blocking=True)
    e2e_step()
    ms_e2e = ctx.timed(e2e_step, 2)
    extra = {}
    if ctx.world == 1 and not args.no_cpu_baseline:
        # the oracle (CPU restatement of the reference, same weights) on clip 0 alone; the GPU path re-run on that clip alone (the T + G padding of a
        # batch depends on its largest group count, so a clip is only comparable with itself at batch 1)
        from oracle import adaptive as oad
        from oracle import hcodec15 as o15
        from oracle.parity import audit_codes
        sd_cpu = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in model.state_dict().items()}
        c = dict(o15.H15)
        n = cpu_threads()
        torch.set_num_threads(n)
        w1, f1 = wav[:1].cpu(), feat[:1].cpu()
        t0 = time.perf_counter()
        otaps = {}
        oa, os_ = o15.codec_encode(sd_cpu, c, w1, f1, otaps)
        ref = o15.codec_decode(sd_cpu, c, oa, os_)
        dt = time.perf_counter() - t0
        gtaps = {}
        go = model.encode(wav[:1], feat[:1], taps=gtaps)
        grec = model.decode(oa.to(dev), os_.to(dev))
        relf = lambda a, b: float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
        G1 = oa.shape[-1]
        rows = lambda t: t.double().cpu().transpose(1, 2).reshape(G1, -1)
        par = dict(sample="clip 0 of the timed batch, alone, vs the oracle (same weights)", grouping_identical=bool(torch.equal(gtaps["seg"].cpu().long(), otaps["align"].argmax(1))),
                   sem_tok_rel=relf(gtaps["sem_agg.out"], otaps["sem_agg.out"]), ac_tok_rel=relf(gtaps["ac_agg.out"], otaps["ac_agg.out"]), wav_rel=relf(grec, ref))
        K = model.codebook_size
        for tag, got, want, key, q in (("acoustic", go["acoustic_codes"], oa, "ac_agg.out", "quantizer"), ("semantic", go["semantic_codes"], os_, "sem_agg.out", "semantic_quantizer")):
            gp, gl = oad.extract_lengths(got.cpu(), K)
            wp, wl = oad.extract_lengths(want, K)
            cb = torch.stack([sd_cpu[f"{q}.layers.{i}._codebook.embed"][0] for i in range(c["nq"])], 0)
            a = audit_codes(gp, wp, rows(gtaps[key]), rows(otaps[key]), cb) if torch.equal(gl, wl) else dict(explained=False)
            par[tag] = {k: a.get(k) for k in ("tokens", "tokens_differing", "index_match_rate", "worst_gap", "worst_reach", "explained")}
        par["ok"] = bool(par["grouping_identical"] and par["sem_tok_rel"] < 1e-3 and par["ac_tok_rel"] < 1e-3 and par["wav_rel"] < 1e-3
                         and par["acoustic"]["explained"] and par["semantic"]["explained"])
        extra = dict(parity=par, cpu_baseline=dict(value=T50 * 320 / dt, unit=UNIT, cores=n, host_cores=host_cores(), kind="port",
                                                   sample=f"1 clip x {T50 / 50:g} s encode + decode ({dt:.1f} s), oracle port of the reference's PyTorch CPU path, same weights, {n} threads"))
    h2d = wav_h.numel() * 4 + feat_h.numel() * 4
    d2h = sum(o.numel() * o.element_size() for o in out_h)
    del model
    torch.cuda.empty_cache()
    return dict(e2e=dict(value=ctx.world * n_samples / (ms_e2e * 1e-3), unit=UNIT, ms_per_step=ms_e2e, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h), **extra,
                metric="hcodec15_adaptive_encode_decode_samples_per_s", value=ctx.world * n_samples / (ms * 1e-3), unit=UNIT, ms_per_step=ms,
                timed_passes_ms=[ms_a, ms_b], n_gpus=ctx.world, scaling="weak",
                config=dict(workload=f"HCodec-1.5 adaptive (config_adaptive_v3) batch={B} x {T50 / 50:g} s @16 kHz encode + decode, threshold 0.6",
                            batch_per_gpu=B, frames_25hz=T50 // 2, tokens_per_clip_mean=float(n_tok.mean()), tokens_per_clip_max=int(n_tok.max()),
                            precision_policy=args.precision, launch="kernel by kernel (data-dependent sequence lengths)"),
                gpu_launches=int(launches),
                roofline=dict(bound="tensor", achieved=tf, peak=peaks["tf_sus"] * ctx.world, unit="TFLOP/s", frac=tf / (peaks["tf_sus"] * ctx.world),
                              kernel="whole encode + decode, algorithmic FLOPs (every GEMM 2MNK once + attention 4 L^2 C)",
                              flops_per_step=flops[0]))


def run_codec(args, cfg, ctx, collect_secondary, first_legs=None):
    from unified_audio_b200 import ops
    from unified_audio_b200.parallel import gather_tokens
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    peaks = load_peaks()
    model = build_codec(cfg, dev, args.precision)
    B = args.batch
    wav_h, feat_h, T = synth_batch(cfg, B, args.seconds, 2000 + rank)
    F_ = T // 960
    wav_d, feat_d = wav_h.to(dev), feat_h.to(dev)

    # the public fixed-shape entry point: encode -> decode captured once in a CUDA graph (Codec.graphed), replayed per step
    graphed = None
    if not args.no_graph:
        try:
            graphed = model.graphed("roundtrip", wav_d, feat_d)
        except Exception as e:      # same kernels either way: fall back to launching them one by one
            print(f"[bench] CUDA-graph capture failed ({e!r}); launching kernel by kernel", file=sys.stderr)
            torch.cuda.synchronize()
    gbuf = {}
    tok_stack = torch.zeros(B, 2, 16, T // 3840, dtype=torch.int64, device=dev)
    last = []                   # outputs of the latest step (the graph's static buffers: read before the next replay)

    def step_device():
        if graphed is not None:
            ac, sc, rec = graphed()                      # static inputs already hold this rank's batch (HBM-resident)
        else:
            ac, sc = model.encode(wav_d, feat_d)
            rec = model.decode(ac, sc)
        if ctx.dist is not None:   # the path's single exchange: gather the int64 tokens (SURVEY 8e)
            tok_stack[:, 0].copy_(ac)
            tok_stack[:, 1].copy_(sc)
            gather_tokens(tok_stack, world * B, buffers=gbuf)
        last[:] = (ac, sc, rec)
        return ac, sc, rec

    def dump_last_step():
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dict(zip(("acoustic_codes", "semantic_codes", "wav_rec"), last)))

    codes_h = torch.empty(2, B, 16, T // 3840, dtype=torch.int64).pin_memory()
    rec_h = torch.empty(B, T).pin_memory()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def step_e2e(split=False):
        if split:
            ev[0].record()
        if graphed is not None:
            for dst, src in zip(graphed.inputs, (wav_h, feat_h)):      # pinned host -> static device inputs (H2D inside the timed region)
                dst.copy_(src, non_blocking=True)
            if split:
                ev[1].record()
            ac, sc, rec = graphed()
        else:
            w = wav_h.to(dev, non_blocking=True)
            ft = feat_h.to(dev, non_blocking=True)
            if split:
                ev[1].record()
            ac, sc = model.encode(w, ft)
            rec = model.decode(ac, sc)
        if split:
            ev[2].record()
        codes_h[0].copy_(ac, non_blocking=True)
        codes_h[1].copy_(sc, non_blocking=True)
        rec_h.copy_(rec, non_blocking=True)
        if split:
            ev[3].record()
        return rec

    if args.quick:
        for _ in range(args.warmup):
            step_device()
        ms = ctx.timed(step_device, args.steps)
        dump_last_step()
        if rank == 0:
            print(json.dumps(dict(quick=True, ms_per_step=ms, value=world * B * T / (ms * 1e-3))))
        return None
    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
    ops.launch_count_reset()
    ms = ctx.timed(step_device, args.steps)
    launches = ops.launch_count() + (graphed.launches_per_replay * args.steps if graphed is not None else 0)
    clocks = sampler.stop() if rank == 0 else None
    dump_last_step()
    for _ in range(2):
        step_e2e()
    ms_e2e_serial = ctx.timed(step_e2e, args.steps)
    ms_e2e = ms_e2e_serial
    if graphed is not None:
        # the public streaming entry point (GraphedCall.stream): every step still copies its inputs from pinned host memory and its codes +
        # waveform back, on a copy stream, overlapped with the neighbouring steps' compute
        outs_h = (codes_h[0], codes_h[1], rec_h)

        def step_e2e_stream():
            graphed.stream((wav_h, feat_h), outs_h)
        for _ in range(2):
            step_e2e_stream()
        graphed.finish()

        calls = [0]

        def run_stream_step():          # the launching stream joins the copy stream after the LAST step, inside the timed region
            step_e2e_stream()
            calls[0] += 1
            if calls[0] == args.steps:
                graphed.finish()
        ms_e2e = ctx.timed(run_stream_step, args.steps)
    torch.cuda.synchronize()
    step_e2e(split=True)
    torch.cuda.synchronize()
    e2e_split = dict(h2d_ms=ev[0].elapsed_time(ev[1]), compute_ms=ev[1].elapsed_time(ev[2]), d2h_ms=ev[2].elapsed_time(ev[3]),
                     note="one extra step, serial on the launching stream (no overlap between copies and kernels)")

    # ---- roofline of the dominant kernel: the ConvNeXt pointwise GEMM (tcgen05), timed alone on operands of the step's shapes
    M, C, I = B * F_, 1536, 4608
    sd_ = model.state_dict()
    w1 = ops.Planes.from_f32(sd_["encoder.prior_net.0.pwconv1.linear.weight"], False)
    b1 = sd_["encoder.prior_net.0.pwconv1.linear.bias"].float().contiguous()
    t1 = ops.Planes(torch.randn(M, C, device=dev).half(), None)
    hid = ops.Planes.zeros((M, I), False, dev)
    reps = 10
    run1 = lambda: ops.gemm(t1, w1, I, a_batch=1, a_rows_per_batch=M, a_ld=C, m_per_batch=M, bias=b1, act=ops.ACT_GELU,
                            out_planes=hid, out_planes_map=(I, M, 0))
    for _ in range(3):
        run1()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        run1()
    e1.record()
    torch.cuda.synchronize()
    gemm_ms = e0.elapsed_time(e1) / reps
    gemm_tf = 2.0 * M * I * C / (gemm_ms * 1e-3) / 1e12
    del t1, hid, w1

    samples = world * B * T
    value = samples / (ms * 1e-3)
    path_tf = world * B * F_ * FLOP_PER_FRAME / (ms * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    line = dict(
        metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
        ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f16x3/f16 tensor-core, f32 accumulate",
        data="synthetic",
        config=dict(workload=f"HCodec-2.0 batch={B} x {args.seconds:g} s (48 kHz shipped config, {T} samples/clip) encode+RVQ+decode",
                    batch_per_gpu=B, samples_per_clip=T, tokens_per_stream=T // 3840, precision_policy=args.precision,
                    l2="working set per step (~3 GB activations + 4.6 GB weights) exceeds the 126 MB L2; no flush needed",
                    parallelism=f"dp{world} (clips sharded, one NCCL all_gather_into_tensor of tokens)",
                    launch="one CUDA graph replay per step (Codec.graphed('roundtrip')); gpu_launches = library kernels in the "
                           "graph x steps" if graphed is not None else "kernel by kernel"),
        e2e=dict(value=samples / (ms_e2e * 1e-3), unit=UNIT, ms_per_step=ms_e2e,
                 h2d_bytes_per_step=int(wav_h.numel() * 4 + feat_h.numel() * 4) * world,
                 d2h_bytes_per_step=int(codes_h.numel() * 8 + rec_h.numel() * 4) * world, split=e2e_split,
                 mode=("Codec.graphed('roundtrip').stream(...): per-step H2D / D2H on a copy stream, overlapped with the neighbouring steps' compute"
                       if graphed is not None else "serial"), serial_ms_per_step=ms_e2e_serial),
        gpu_launches=int(launches),
        clocks=clocks,
        roofline=dict(bound="tensor", achieved=gemm_tf, peak=peaks["tf_burst"], unit="TFLOP/s", frac=gemm_tf / peaks["tf_burst"],
                      traffic=traffic, kernel=f"{ops.gemm_kernel_name(M, I, False)} ConvNeXt pwconv1 [{M}x{I}x{C}] fp16 + GELU epilogue, timed alone on rank 0",
                      peak_source=f"{peaks['src']} dense bf16 burst (fp16 shares the pipe), one GPU",
                      path_algorithmic_tflops=path_tf, path_algorithmic_tflops_per_gpu=path_tf / world,
                      path_frac_of_sustained=path_tf / (peaks["tf_sus"] * world)),
    )
    line["cpu_baseline"] = None                  # timed on rank 0 at N = 1 only (the N > 1 lines carry the key, empty)
    line["parity"] = None
    if not args.no_cpu_baseline and world == 1:
        # clip 0 of the timed batch on the reference's CPU path: the CPU baseline AND the parity check of this very run
        from oracle import hcodec2
        from oracle.parity import audit_codes
        sd_cpu = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        v, dt, otaps, (oa, os_) = cpu_codec(sd_cpu, cfg, wav_h[:1].clone(), feat_h[:1].clone(), want_codes=True)
        n = cpu_threads()
        line["cpu_baseline"] = dict(value=v, unit=UNIT, cores=n, host_cores=host_cores(), kind="port",
                                    sample=f"1 clip x {args.seconds:g} s encode+RVQ+decode ({dt:.1f} s), oracle port of "
                                           f"the reference's PyTorch CPU path, same weights, {n} threads")
        gtaps = {}
        ac, sc = model.encode(wav_d, feat_d, taps=gtaps)
        rec = model.decode(oa.to(dev), os_.to(dev))
        ref = hcodec2.codec_decode(sd_cpu, cfg, oa, os_)
        rows = lambda t: t[:1].float().cpu().transpose(1, 2).reshape(-1, t.shape[1])
        relf = lambda a, b: float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
        par = dict(sample="clip 0 of the timed batch vs the oracle (same weights, same run)",
                   emb_rel=relf(gtaps["enc.out"][:1], otaps["enc.out"]), sem_rel=relf(gtaps["sem.out"][:1], otaps["sem.out"]),
                   wav_rel=relf(rec, ref))
        for tag, got, want, key, q in (("acoustic", ac[:1], oa, "enc.out", "quantizer"), ("semantic", sc[:1], os_, "sem.out", "semantic_quantizer")):
            a = audit_codes(got, want, rows(gtaps[key]), rows(otaps[key]), hcodec2._codebooks(sd_cpu, q))
            par[tag] = {k: a[k] for k in ("tokens", "tokens_differing", "index_match_rate", "worst_gap", "worst_reach", "explained")}
        par["ok"] = bool(par["emb_rel"] < 1e-3 and par["sem_rel"] < 1e-3 and par["wav_rel"] < 1e-3 and par["acoustic"]["explained"]
                         and par["semantic"]["explained"])
        line["parity"] = par
    sec = None
    if collect_secondary:
        sec = {}
        if first_legs is not None:      # the AR-LM half of the metric goes before the codec's extra shapes
            first_legs(sec)

        def leg_strong():
            return bench_codec_strong(args, ctx, model, cfg, 256)

        def leg_240k():     # SURVEY 8(d) "24 kHz sample-count" reporting shape: 240 000 samples -> pad_wav -> 241 920 (63 tokens, 252 frames)
            from unified_audio_b200.ssl import pad_wav
            g24 = torch.Generator().manual_seed(2400 + rank)
            w24 = pad_wav((0.1 * torch.randn(B, 240000, generator=g24)).to(dev), 3840)
            f24 = torch.randn(B, 768, w24.shape[1] // 960, generator=g24)
            f24 = (torch.sign(f24) * f24.abs() ** 0.3).to(dev)
            g24c = model.graphed("roundtrip", w24, f24)
            g24c()
            ms24 = ctx.timed(lambda: g24c(), 3)
            return dict(metric=METRIC, value=world * B * 240000 / (ms24 * 1e-3), unit=UNIT, ms_per_step=ms24,
                        config=dict(workload=f"HCodec-2.0 batch={B} x 240 000 samples (padded to {w24.shape[1]}: 63 tokens, "
                                             "252 frames) encode+RVQ+decode", batch_per_gpu=B),
                        path_algorithmic_tflops=world * B * (w24.shape[1] // 960) * FLOP_PER_FRAME / (ms24 * 1e-3) / 1e12)

        def leg_tokenize():
            return bench_tokenize(args, ctx, model, cfg)

        def leg_accurate():     # fp32-grade policy (every GEMM a 3-term split) beside the default
            nonlocal graphed
            graphed = None
            model._ws, model._engine = {}, None
            torch.cuda.empty_cache()
            macc = build_codec(cfg, dev, "accurate")
            gacc = macc.graphed("roundtrip", wav_d, feat_d)
            gacc()
            ms_acc = ctx.timed(lambda: gacc(), 3)
            return dict(metric=METRIC, value=B * T / (ms_acc * 1e-3), unit=UNIT, ms_per_step=ms_acc,
                        config=dict(precision_policy="accurate", batch_per_gpu=B))

        legs = [("codec_b256_strong", leg_strong), ("codec_240k_samples_shape", leg_240k), ("tokenize_wav_to_codes", leg_tokenize)]
        if world == 1 and args.precision != "accurate":
            legs.append(("codec_accurate_policy", leg_accurate))
        for name, fn in legs:
            run_leg(ctx, sec, name, fn)
    del model
    torch.cuda.empty_cache()
    return line, sec


def bicodec_flops_per_clip(cfg, T):
    """algorithmic FLOPs of BiCodec.detokenize for one clip of T tokens (2 x MACs, true channel counts and taps)"""
    p, d = cfg["prenet"], cfg["decoder"]
    dim, inter = p["vocos_dim"], p["vocos_intermediate_dim"]
    blocks = 2 * len(p["sample_ratios"]) + p["vocos_num_layers"]
    backbones = len(p["sample_ratios"]) + 1
    f = 2.0 * T * (p["input_channels"] * dim + backbones * dim * dim * 7 + blocks * 2 * dim * inter + dim * p["out_channels"])
    ch = d["channels"]
    f += 2.0 * T * d["input_channel"] * ch * 7
    Tc = T
    for i, (k, r) in enumerate(zip(d["kernel_sizes"], d["rates"])):
        cin, cout = ch // 2 ** i, ch // 2 ** (i + 1)
        f += 2.0 * Tc * cin * cout * k                     # transposed conv: k taps per INPUT frame
        Tc *= r
        f += 3 * 2.0 * Tc * cout * cout * 8                # 3 residual units: dilated k7 + 1x1
    f += 2.0 * Tc * (ch // 2 ** len(d["rates"])) * 7
    return f


def init_bicodec_(m, dev):
    """random-init weights of the BiCodec detokenize path (weight-norm gains ~ ||v||, residual branches damped, as oracle.bicodec.make_state_dict)"""
    g = torch.Generator(device=dev).manual_seed(5)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("alpha"):
                p.copy_(1 + 0.3 * torch.rand(p.shape, generator=g, device=dev))
            elif n.endswith(("weight_g",)):
                p.fill_(1.0)
            elif p.dim() >= 2:
                fan = p[0].numel() if "block.1.weight_v" not in n else 2 * p.shape[0]
                p.copy_(torch.randn(p.shape, generator=g, device=dev) / fan ** 0.5)
            elif n.endswith(("gamma",)):
                p.fill_(1.0 / 12)
            elif n.endswith(("norm.weight", "scale.bias", "final_layer_norm.weight")):
                p.fill_(1.0)
            else:
                p.copy_(0.02 * torch.randn(p.shape, generator=g, device=dev))
        sdm = m.state_dict()
        for n in list(sdm):
            if n.endswith("weight_g"):
                v = sdm[n[:-1] + "v"]
                gain = 0.3 if ".block.3." in n else (0.1 if n.startswith("decoder.model.6.") else 1.0)
                sdm[n].copy_(gain * v.reshape(v.shape[0], -1).norm(dim=1).reshape(sdm[n].shape))
    m._w = None


def run_bicodec(args):
    """Secondary line: BiCodec.detokenize, the decoder UniSE feeds its AR-LM tokens to (SURVEY 8f.1; configs[2] back half):
    B=32 clips x 250 semantic tokens + 32 global tokens -> 5 s @ 16 kHz each."""
    B, T = 32, 250
    if args.impl == "reference" and int(os.environ.get("RANK", "0")) != 0:
        return
    if args.impl == "reference":
        from oracle import bicodec as ob
        cfg = ob.BICODEC_FULL
        sd = ob.make_state_dict(cfg, 5)
        sem, glob = ob.synth_tokens(cfg, 1, T, 9)
        torch.set_num_threads(min(16, os.cpu_count() or 1))
        ob.detokenize(sd, cfg, sem[:, :25], glob)
        t0 = time.perf_counter()
        ob.detokenize(sd, cfg, sem, glob)
        dt = time.perf_counter() - t0
        v = T * 320 / dt
        print(json.dumps(dict(metric="bicodec_detokenize_samples_per_s", value=v, unit="samples/s", n_gpus=args.gpus, steps=1,
                              warmup=1, ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                              dtype="f32", data="synthetic", impl="reference",
                              config=dict(workload="BiCodec detokenize, 1 clip x 250 tokens -> 5 s @ 16 kHz", batch=1),
                              cpu_baseline=dict(value=v, unit="samples/s", cores=torch.get_num_threads(), kind="port",
                                                sample="1 clip x 5 s, oracle port pinned against the reference's BiCodec classes"),
                              e2e=dict(value=v, unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)))
        return
    from unified_audio_b200 import ops
    from unified_audio_b200.bicodec import BICODEC_CONFIG, BiCodec
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:       # clips are independent: B per rank, no data-path collective (the waveforms stay on their rank)
        import torch.distributed as dist_
        dist = dist_
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    cfg = BICODEC_CONFIG
    m = BiCodec(cfg).to(dev)
    init_bicodec_(m, dev)
    gt = torch.Generator().manual_seed(50 + rank)
    sem_h = torch.randint(0, cfg["quantizer"]["codebook_size"], (B, T), generator=gt).pin_memory()
    glob_h = torch.randint(0, 4096, (B, 1, 32), generator=gt).pin_memory()
    sem, glob = sem_h.to(dev), glob_h.to(dev)
    wav_h = torch.empty(B, 1, T * 320).pin_memory()

    def timed(fn):
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(args.steps):
            fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    for _ in range(max(args.warmup, 3)):
        m.detokenize(sem, glob)
    if args.quick:
        ms = timed(lambda: m.detokenize(sem, glob))
        if rank == 0:
            print(json.dumps(dict(quick=True, ms_per_step=ms)))
        return
    ops.launch_count_reset()
    ms = timed(lambda: m.detokenize(sem, glob))
    launches = ops.launch_count()

    def e2e_step():
        w = m.detokenize(sem_h.to(dev, non_blocking=True), glob_h.to(dev, non_blocking=True))
        wav_h.copy_(w, non_blocking=True)
    ms_e2e = timed(e2e_step)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    samples = world * B * T * 320
    tf = world * B * bicodec_flops_per_clip(cfg, T) / (ms * 1e-3) / 1e12
    cpu = None
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", "bicodec", "--impl", "reference"],
                           capture_output=True, text=True, timeout=600)
        cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as e:      # the baseline is reported, never required for the GPU line
        cpu = dict(value=None, unit="samples/s", cores=0, kind="port", sample=f"failed: {e}")
    print(json.dumps(dict(
        metric="bicodec_detokenize_samples_per_s", value=samples / (ms * 1e-3), unit="samples/s", n_gpus=world, steps=args.steps,
        warmup=max(args.warmup, 3), ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype="f16x3 split tensor-core (fp32-grade), f32 accumulate", data="synthetic",
        config=dict(workload="BiCodec detokenize (UniSE's decoder): 32 clips x 250 semantic + 32 global tokens -> 5 s @ 16 kHz",
                    batch_per_gpu=B, tokens=T, precision_policy="accurate",
                    l2="activations per step (~10 GB) exceed the 126 MB L2; no flush needed",
                    parallelism=f"dp{world} (clips sharded, no collective)"),
        e2e=dict(value=samples / (ms_e2e * 1e-3), unit="samples/s", ms_per_step=ms_e2e,
                 h2d_bytes_per_step=int(sem_h.numel() * 8 + glob_h.numel() * 8) * world,
                 d2h_bytes_per_step=int(wav_h.numel() * 4) * world),
        gpu_launches=int(launches),
        roofline=dict(bound="tensor", achieved=tf, peak=peaks["tf_sus"] * world, unit="TFLOP/s", frac=tf / (peaks["tf_sus"] * world),
                      traffic=None, kernel="whole detokenize path, algorithmic FLOPs (true channels / taps; every GEMM issued 3x in the "
                      "`accurate` policy) against the sustained bf16 peak"),
        cpu_baseline=cpu)))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--no-graph", action="store_true", help="launch the step kernel by kernel instead of replaying the CUDA graph")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="clips per GPU per step")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--precision", default="mixed")
    ap.add_argument("--ref-clips", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="all", choices=["all", "codec", "lm", "lm_tse", "lm_forward", "bicodec", "h15"],
                    help="all (default, the driver's line) = the codec line (BASELINE configs[1]) with the UniSE AR-LM legs (configs[2], [3], "
                         "[4]) under `secondary`; codec / lm / lm_tse / lm_forward / bicodec = that line alone")
    ap.add_argument("--quick", action="store_true", help="profiling aid: W warm-up + K steps only, no e2e/roofline/cpu legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed H-Codec-2.0 step returned (acoustic / semantic codes, "
                         "waveform; rank 0) as DIR/<name>.npy in float32, at most 64 MB: a seeded sample of the waveform's clips if larger")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("all", "codec")):
        ap.error("--dump-outputs writes the outputs of the H-Codec-2.0 step: --impl ours with --workload all or codec")
    args.warmup = max(args.warmup, 0)
    cfg = H2_FULL
    if args.workload == "bicodec":
        return run_bicodec(args)
    if args.impl == "reference":
        if args.workload in ("lm", "lm_tse"):
            if int(os.environ.get("RANK", "0")) == 0:
                c = cpu_lm_generate("tse" if args.workload == "lm_tse" else "se")
                print(json.dumps(dict(metric="unise_arlm_generate_tokens_per_s", value=c["value"], unit="tokens/s", impl="reference",
                                      n_gpus=args.gpus, higher_is_better=True, cpu_baseline=c,
                                      e2e=dict(value=c["value"], unit="tokens/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
            return
        return run_reference(args, cfg)
    ctx = Ctx()
    if args.workload == "h15":
        out = bench_h15(args, ctx)
        if ctx.rank == 0:
            print(json.dumps(out))
        ctx.close()
        return
    if args.workload in ("lm", "lm_tse", "lm_forward"):
        m = build_lm(ctx.dev)
        if args.workload == "lm_forward":
            out = bench_lm_forward(args, ctx, m)
        else:
            task = "tse" if args.workload == "lm_tse" else "se"
            out = bench_lm_generate(args, ctx, m, task, 16 if task == "tse" else 32, with_cpu=ctx.world == 1 and not args.no_cpu_baseline)
        out.update(warmup=max(args.warmup, 2), vs_baseline=None)
        if ctx.rank == 0:
            print(json.dumps(out))
        ctx.close()
        return
    lm_box = {}

    def lm_first(sec):
        # the AR-LM half of BASELINE.json's metric in the same invocation: SR B=32 (configs[2]) and TSE B=16 (configs[3]) per GPU
        lm_box["m"] = m = build_lm(ctx.dev)
        with_cpu = ctx.world == 1 and not args.no_cpu_baseline
        run_leg(ctx, sec, "lm_sr", lambda: bench_lm_generate(args, ctx, m, "se", 32, with_cpu=with_cpu))
        run_leg(ctx, sec, "lm_tse", lambda: bench_lm_generate(args, ctx, m, "tse", 16, with_cpu=with_cpu))

    full = args.workload == "all" and not args.quick
    res = run_codec(args, cfg, ctx, collect_secondary=full, first_legs=lm_first if full else None)
    if res is None:
        ctx.close()
        return
    line, sec = res
    if full:
        # the batch-256 sweep (configs[4]), the teacher-forced forward, the adaptive codec
        m = lm_box["m"]
        for name, fn in (("lm_sr_b256_strong", lambda: bench_lm_generate(args, ctx, m, "se", None, total_batch=256, steps=2)),
                         ("unise_sr_pipeline", lambda: bench_unise_sr(args, ctx, m)),
                         ("lm_forward", lambda: bench_lm_forward(args, ctx, m)),
                         ("hcodec15_adaptive", lambda: bench_h15(args, ctx))):
            run_leg(ctx, sec, name, fn)
        line["secondary"] = sec
        line["bench_wall_s"] = round(ctx.elapsed_s(), 1)
    if ctx.rank == 0:
        print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    main()
