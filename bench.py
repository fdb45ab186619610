#!/usr/bin/env python
"""Benchmark of the per-frame hot path (BASELINE.json metric: streaming frames/sec/GPU, 10 tok/frame,
~12k-token KV) — driver contract in the task statement.

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA engine), one rank per GPU under torchrun
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU (oracle port)

One *step* = one frame of one video stream through the whole path: SigLIP-L/16-384 ViT -> CLS + 3x3 pooled
tokens -> connector -> Llama-3-8B KV-append forward over [interval token | 10 frame tokens] on a >=12k-token
KV cache -> on-device speak/silent decision.  Workload = BASELINE.json configs[1] (1 stream per GPU, 10-min
video position: kv 12 000 -> 12 000 + 11*steps), synthetic frames and seeded random weights of the
full-size architecture (no checkpoint/network available).  N GPUs run N independent streams (weights
broadcast once over NCCL at init, no hot-path collective): "scaling": "weak".
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (which may be read-only)

METRIC = "streaming frames/sec (10 tok/frame, 12k-ctx KV), all GPUs"
UNIT = "frames/s"
KV_START = 12000
WORKLOAD = ("configs[1]: 1 stream/GPU, SigLIP-L/16-384 + Llama-3-8B, frame step of 11 tokens at kv>=12000 "
            "(10-min video @2FPS position), synthetic 384x384 frames, seeded random weights")


def static_config(world: int) -> dict:
    """The `config` object of the JSON line: identical for the engine arm and the --impl reference arm (the driver
    compares them); everything measured or run-dependent goes under "run"."""
    return {"workload": WORKLOAD, "streams_per_gpu": 1, "kv_tokens_start": KV_START, "tokens_per_step": 11,
            "vit_dtype": "fp16 operands / fp32 accumulate",
            "parallelism": f"replicas x{world} (weights broadcast at init, no hot-path collective)",
            "l2": "inputs larger than L2: every step streams 15.0 GB of weights + 1.6 GB of KV (L2 = 126 MB)",
            "pipelining": "ViT+connector of the NEXT frames on a side CUDA stream during the decoder steps of the current ones "
                          "(same work per frame; --encode-ahead frames per ViT pass, default 1: the next frame, as a live "
                          "camera delivers it)"}


# ----------------------------------------------------------------------------- helpers
def _ncu_traffic(kernel_key):
    """(dram__bytes_read.sum + dram__bytes_write.sum per launch, commit of the capture) from the committed ncu --set full
    summaries (profiles/ncu_traffic.json, written by tools/profile_summary.py from the .ncu-rep files), or (None, None)."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    if not p.exists():
        return None, None
    try:
        d = json.loads(p.read_text())
        return d.get(kernel_key, {}).get("dram_bytes_per_launch"), d.get(kernel_key, {}).get("commit", d.get("commit"))
    except Exception:
        return None, None


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1468.8))), "measured"
    return 6650.0, 1400.0, "fallback"


def dump_outputs(out_dir, frame_embeds, logits, decisions):
    """--dump-outputs: what the last timed frame step handed its caller, as .npy files: frame_embeds.npy (float32
    [10, hidden], the ViT + connector output the step consumed), logits.npy (float32 [1, vocab], last position) and one
    float64 decision_<field>.npy per field of the on-device speak/silent decision."""
    import numpy as np
    import torch
    from videollm_online_b200.engine import Decision
    row = decisions[0].cpu()
    dec = Decision(row, row.view(torch.float32))
    arrays = {"frame_embeds": frame_embeds.float().cpu().numpy(), "logits": logits.float().cpu().numpy()}
    arrays.update({"decision_" + f: np.array([getattr(dec, f)], dtype=np.float64) for f in Decision.__slots__})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "10",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU (reference algorithm) arm
def cpu_reference_times(n_steps: int, n_warm: int, dec_layers: int = 0, vit_layers: int = 0, budget_s: float = 200.0):
    """Times the oracle (CPU port of the reference forward, oracle/vlo_oracle.py) on the host cores.

    A step is the FULL frame step (24 ViT blocks + connector, 32 decoder layers over a 12k-token cache, lm_head,
    decision) whenever (n_steps + n_warm) of them fit `budget_s` on this host (probed with one full step): then nothing
    is extrapolated and ms_per_step x steps is the run's wall time.  On a slower host the stacks are truncated
    (dec_layers / vit_layers > 0 force that) and the per-layer cost is scaled to the full depth; the line says so."""
    import torch
    # all the host threads it can use: torchrun exports OMP_NUM_THREADS=1 to every rank, which would time the CPU arm
    # on one core; use one thread per physical core (torch's own default outside torchrun)
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    torch.set_num_threads(max(1, avail // 2))   # pinned: one thread per physical core of the affinity mask
    sys.path.insert(0, str(ROOT / "oracle"))
    import vlo_bootstrap  # noqa: F401
    import vlo_oracle as O
    from videollm_online_b200 import llama3_8b_siglip_l
    import dataclasses
    cfg = llama3_8b_siglip_l()
    g = torch.Generator().manual_seed(0)
    H, I, V = cfg.hidden_size, cfg.intermediate_size, cfg.vocab_size
    nh, nkv, hd = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim

    def rnd(shape, std=0.02, dtype=torch.bfloat16):
        n = 1
        for s in shape:
            n *= s
        block = torch.randn(min(n, 1 << 22), generator=g) * std       # tile a 4M-element random block: fast fill
        reps = (n + block.numel() - 1) // block.numel()
        return block.repeat(reps)[:n].view(*shape).to(dtype).contiguous()

    # ---- decoder: ONE layer's random weights aliased for every sampled layer (436 MB >> L3, so no cache reuse)
    layer = {"self_attn.q_proj.weight": rnd((nh * hd, H)), "self_attn.k_proj.weight": rnd((nkv * hd, H)),
             "self_attn.v_proj.weight": rnd((nkv * hd, H)), "self_attn.o_proj.weight": rnd((H, nh * hd)),
             "mlp.gate_proj.weight": rnd((I, H)), "mlp.up_proj.weight": rnd((I, H)), "mlp.down_proj.weight": rnd((H, I)),
             "input_layernorm.weight": torch.ones(H, dtype=torch.bfloat16),
             "post_attention_layernorm.weight": torch.ones(H, dtype=torch.bfloat16)}
    sd = {"model.norm.weight": torch.ones(H, dtype=torch.bfloat16), "lm_head.weight": rnd((V, H)),
          "connector.0.weight": rnd((H, cfg.vision_hidden_size)), "connector.0.bias": rnd((H,)),
          "connector.2.weight": rnd((H, H)), "connector.2.bias": rnd((H,))}
    for i in range(cfg.num_hidden_layers):   # every layer aliases the same tensors: full depth costs no extra host memory
        for k, v in layer.items():
            sd[f"model.layers.{i}.{k}"] = v
    kv_block = rnd((1, nkv, KV_START, hd), 1.0)
    # ---- ViT: full-size SigLIP-L blocks (fp32, as on a CPU host); one block's weights aliased for all 24
    from videollm_online_b200 import weights as W
    one_blk = dataclasses.replace(cfg, vision_num_hidden_layers=1)
    vs = {k: v for k, v in W.synthetic_vision_state(one_blk, seed=1).items()}
    for i in range(1, cfg.vision_num_hidden_layers):
        for k in [k for k in vs if k.startswith("encoder.layers.0.")]:
            vs["encoder.layers.%d." % i + k[len("encoder.layers.0."):]] = vs[k]
    frames = torch.randint(0, 256, (1, 3, cfg.frame_resolution, cfg.frame_resolution), dtype=torch.uint8, generator=g)
    ids = torch.tensor([cfg.frame_token_interval_id])
    sd["model.embed_tokens.weight"] = rnd((1024, H), 1.0)  # only row `interval id` is read

    def one_step(nd, nv):
        dcfg = dataclasses.replace(cfg, num_hidden_layers=nd)
        vcfg = dataclasses.replace(cfg, vision_num_hidden_layers=nv)
        t0 = time.perf_counter()
        fe = O.visual_embed(sd, vs, vcfg, frames)
        t1 = time.perf_counter()
        cache = O.KVCache(nd)
        for i in range(nd):
            cache.k[i], cache.v[i] = kv_block, kv_block
        emb = torch.cat([O.embed_tokens(sd, ids), fe], 0)
        t2 = time.perf_counter()
        logits = O.llama_forward(sd, dcfg, emb, cache)
        O.decide(logits[-1], cfg.frame_token_interval_id, 0.725)
        t3 = time.perf_counter()
        return t1 - t0, t3 - t2

    with torch.no_grad():
        if dec_layers <= 0 or vit_layers <= 0:
            one_step(2, 2)                                       # page in MKL / the weights
            pv, pd = one_step(8, 6)                              # probe: a quarter of the stacks
            est_full = pv * cfg.vision_num_hidden_layers / 6 + pd * cfg.num_hidden_layers / 8
            frac = min(1.0, budget_s / (est_full * (n_steps + n_warm)))
            dec_layers = cfg.num_hidden_layers if frac >= 1.0 else max(4, int(cfg.num_hidden_layers * frac))
            vit_layers = cfg.vision_num_hidden_layers if frac >= 1.0 else max(3, int(cfg.vision_num_hidden_layers * frac))
        for _ in range(n_warm):
            one_step(dec_layers, vit_layers)
        tv, td = [], []
        for _ in range(n_steps):
            a, b = one_step(dec_layers, vit_layers)
            tv.append(a); td.append(b)
    full = dec_layers == cfg.num_hidden_layers and vit_layers == cfg.vision_num_hidden_layers
    # scale the truncated stacks to the full model (per-layer cost is uniform; embeddings/head/lm_head are
    # counted once at full size inside the sample and slightly over-weighted by the scaling -> conservative for us)
    vit_s = sum(tv) / len(tv) * (cfg.vision_num_hidden_layers / vit_layers)
    dec_s = sum(td) / len(td) * (cfg.num_hidden_layers / dec_layers)
    per_step = [a * (cfg.vision_num_hidden_layers / vit_layers) + b * (cfg.num_hidden_layers / dec_layers) for a, b in zip(tv, td)]
    return vit_s + dec_s, {"vit_s_per_frame": vit_s, "decoder_s_per_step": dec_s, "threads": torch.get_num_threads(),
                           "per_step_s": [round(x, 3) for x in per_step], "extrapolated": not full,
                           "rel_std": (round(float(torch.tensor(per_step).std() / torch.tensor(per_step).mean()), 4) if len(per_step) > 1 else None),
                           "sample": (f"{n_steps} FULL frame steps (+{n_warm} warm-up) of oracle/vlo_oracle.py: SigLIP-L 24 blocks + connector + "
                                      f"Llama-3-8B 32 layers at kv={KV_START} + lm_head + decision, nothing extrapolated" if full else
                                      f"{n_steps} frame steps (+{n_warm} warm-up) of oracle/vlo_oracle.py with the stacks truncated to "
                                      f"{vit_layers}/24 ViT blocks and {dec_layers}/32 decoder layers at kv={KV_START} (host too slow for full "
                                      "steps within the time budget), per-layer cost scaled to the full depth")
                                     + "; fp32 ViT / bf16 decoder as the reference runs on a CPU host"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    import torch
    t0 = time.perf_counter()
    per_step, info = cpu_reference_times(max(1, args.steps), max(0, args.warmup))
    fps = 1.0 / per_step
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": static_config(int(os.environ.get("WORLD_SIZE", "1"))),
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": info["threads"], "kind": "port", "sample": info["sample"],
                             "vit_s_per_frame": info["vit_s_per_frame"], "decoder_s_per_step": info["decoder_s_per_step"],
                             "host_cpus": os.cpu_count(), "per_step_s": info["per_step_s"], "extrapolated": info["extrapolated"],
                             "rel_std": info["rel_std"],
                             "note": "CPU port of the reference forward (oracle/), NOT the reference's GPU path: a reported baseline, not a speed-up claim"},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    return line


# ----------------------------------------------------------------------------- our arm
def run_engine_arm(args):
    import torch
    import vlo_bootstrap  # noqa: F401
    from videollm_online_b200 import llama3_8b_siglip_l, weights as W
    from videollm_online_b200.engine import Engine
    from videollm_online_b200.modeling_live import LiveLlamaForCausalLM
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    cfg = llama3_8b_siglip_l()
    K, Wm = args.steps, max(3, args.warmup)
    n_frames = K + Wm + 8
    cap = ((KV_START + 11 * (2 * n_frames + 8) + 63) // 64) * 64 + 128
    if args.extras:
        cap = max(cap, 13568)          # the literal configs[1] run ends at ~13.3k tokens
    n_extra = 8 if args.extras else 1   # streams for the multi-stream side measurements
    eng = Engine(cfg, dev, max_streams=n_extra, max_kv_tokens=cap, max_step_tokens=128, max_vit_batch=max(n_extra, args.encode_ahead))

    # ---- weights: rank 0 synthesises, everyone else receives them over NCCL/NVLink (init only)
    from videollm_online_b200.dist import broadcast_weights
    weights = W.synthetic_engine_weights(cfg, dev, cap, seed=0) if rank == 0 else None
    t_b0 = time.perf_counter()
    weights = broadcast_weights(cfg, weights, dev, cap, dist, release_source=True)
    torch.cuda.synchronize()
    bcast_s = time.perf_counter() - t_b0
    eng.load_weights(weights)
    model = LiveLlamaForCausalLM(cfg, eng)
    sid = eng.stream_open()
    g = torch.Generator().manual_seed(1234 + rank)
    S = cfg.frame_resolution
    frames_host = torch.randint(0, 256, (n_frames, 3, S, S), dtype=torch.uint8, generator=g).pin_memory()
    frames_dev = frames_host.to(dev)
    prefix = torch.tensor([cfg.frame_token_interval_id] + [-1] * 10, dtype=torch.int64, device=dev)
    packed = torch.zeros(11, cfg.hidden_size, dtype=torch.bfloat16, device=dev)
    stream = torch.cuda.current_stream(dev)

    def frame_step_resident(i):           # inputs already in HBM, no host sync
        fe = eng.vit_encode(frames_dev[i:i + 1])
        packed[1:] = fe
        eng.step([sid], [11], packed, row_ids=prefix, want_logits=True)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def reduce_max(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- pipelining across frames: the ViT + connector of frame i+1 run on a second CUDA stream while the decoder
    #      step of frame i runs on the main stream (a live stream delivers frame i+1 during step i anyway; with a
    #      loaded clip LiveInfer prefetches the next frame the same way).  Every timed step still does one full
    #      ViT + one full decoder step; n frames in the region = n ViTs + n steps.
    side = torch.cuda.Stream(dev)
    D = max(1, min(args.encode_ahead, eng.max_vit_batch))     # frames per encode-ahead ViT pass
    evs = [torch.cuda.Event(), torch.cuda.Event()]
    fes = [None, None]
    fbufs = [torch.empty(D, 3, S, S, dtype=torch.uint8, device=dev) for _ in range(2)]

    def encode_on_side(i, slot, from_host, after=None, count=1):
        """ViT + connector of frames [i, i+count) (indices modulo the synthetic clip) on the side stream"""
        if after is not None:
            side.wait_event(after)      # the frames arrive while the step launched just before `after` is running
        else:
            side.wait_stream(stream)
        idx = [(i + k) % n_frames for k in range(count)]
        contiguous = idx[-1] - idx[0] == count - 1
        with torch.cuda.stream(side):
            if from_host:   # e2e: these steps' inputs come from pinned host memory
                for k, j in enumerate(idx):
                    fbufs[slot][k:k + 1].copy_(frames_host[j:j + 1], non_blocking=True)
                fes[slot] = model.visual_embed(fbufs[slot][:count])
            else:
                fes[slot] = eng.vit_encode(frames_dev[idx[0]:idx[0] + count] if contiguous else frames_dev[idx])
            evs[slot].record(side)

    pre_evs = [torch.cuda.Event(), torch.cuda.Event()]

    def pipelined(n, base, from_host=False, read_back=False, step_fn=None):
        """n frame steps; the ViT runs D frames at a time on the side stream, one group ahead of the decoder.
        Returns what the last step's eng.step returned (without step_fn): its logits and decisions on the device."""
        n_groups = (n + D - 1) // D
        encode_on_side(base, 0, from_host, count=min(D, n))
        fe = res = None
        for i in range(n):
            g, j = divmod(i, D)
            if j == 0:
                stream.wait_event(evs[g & 1])
                fe = fes[g & 1]
                fe.record_stream(stream)
            if j == 0:
                pre_evs[g & 1].record(stream)
            # the decoder step is enqueued FIRST: after a decision read-back the host is the critical path, and the
            # launches of the next group's ViT must not sit in front of the step's
            if step_fn is not None:
                step_fn(i, fe[10 * j:10 * j + 10])
            else:
                packed[1:] = fe[10 * j:10 * j + 10]
                res = eng.step([sid], [11], packed, row_ids=prefix, want_logits=True)
            if j == 0 and g + 1 < n_groups:
                encode_on_side(base + (g + 1) * D, (g + 1) & 1, from_host, after=pre_evs[g & 1], count=min(D, n - (g + 1) * D))
            if read_back:
                eng.read_decisions(1)
        return res

    # ---- device-resident timing (value)
    eng.kv_fill_synthetic(sid, KV_START, seed=7 + rank)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()       # 10 ms period, running from the warm-up on: the timed region alone can be 0.1 s
    pipelined(Wm, 0)
    barrier()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    last_logits, last_dec = pipelined(K, Wm)
    e1.record(stream)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, packed[1:], last_logits, last_dec)
    ms_total = reduce_max(e0.elapsed_time(e1))
    launches = eng.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    kv_end = eng.kv_len(sid)

    # ---- end-to-end timing through the public API with host frames (e2e): pinned-host frame copied in and the
    #      32-byte decision read back (one sync) every step
    eng.kv_truncate(sid, KV_START)
    pipelined(Wm, 0, from_host=True, read_back=True)
    barrier()
    t0 = time.perf_counter()
    pipelined(K, Wm, from_host=True, read_back=True)
    torch.cuda.synchronize()
    e2e_s = reduce_max(time.perf_counter() - t0)
    barrier()

    # ---- the drop-in path: LiveInfer.input_video_stream + __call__ exactly as demo/cli.py:31-38 drives them (one frame per
    #      iteration, decision read back, encode-ahead of the next frame), frames in PINNED HOST memory copied in per step.
    #      Random weights never emit the protocol ids, so the documented test seam forces "silent" (the frame-step path;
    #      speak / AR bursts are measured by the configs[4] extra).
    from videollm_online_b200.config import LiveArguments, SYSTEM_PROMPT
    from videollm_online_b200.inference import LiveInfer
    from videollm_online_b200.tokenization_live import ByteTokenizer
    from videollm_online_b200.modeling_live import StreamKV
    eng.kv_truncate(sid, KV_START)
    li = LiveInfer(LiveArguments(frame_fps=2, system_prompt=SYSTEM_PROMPT), model=model, tokenizer=ByteTokenizer(cfg),
                   stream=StreamKV(eng, sid))
    def _silent(dec, call):
        dec.argmax_id = dec.argmax_prob_id = cfg.frame_token_interval_id
        dec.p_interval = 1.0
        return dec
    li.decision_hook = _silent
    li.load_video(frames_host[:Wm + K + 1], keep_on_host=True)
    eng.kv_fill_synthetic(sid, KV_START, seed=7 + rank)    # LiveInfer() reset the stream: back to the 10-minute position
    li.past_key_values = li._kv
    li.last_ids = torch.tensor([[cfg.frame_token_interval_id]])
    for i in range(Wm):
        li.input_video_stream(i / li.frame_fps)
        li()
    barrier()
    t0 = time.perf_counter()
    for i in range(Wm, Wm + K):
        li.input_video_stream(i / li.frame_fps)
        li()
    torch.cuda.synchronize()
    e2e_li_s = reduce_max(time.perf_counter() - t0)
    barrier()

    # ---- strictly sequential variant (ViT, then decoder step, one stream) for reference
    eng.kv_truncate(sid, KV_START)
    for i in range(Wm):
        frame_step_resident(i)
    torch.cuda.synchronize()
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    q0.record(stream)
    for i in range(K):
        frame_step_resident(Wm + i)
    q1.record(stream)
    torch.cuda.synchronize()
    seq_ms = q0.elapsed_time(q1) / K

    # ---- per-kernel-class roofline pass (CUDA events around every launch of the class, same workload)
    roof = None
    if rank == 0:
        eng.kv_truncate(sid, KV_START)
        eng.lib.vlo_profile_enable(1)
        P = min(K, 10)
        for i in range(P):
            frame_step_resident(Wm + i)
        ncls = 6
        ms, n, by = (C.c_double * ncls)(), (C.c_longlong * ncls)(), (C.c_double * ncls)()
        eng.lib.vlo_profile_read(ms, n, by, ncls)
        eng.lib.vlo_profile_enable(0)
        hbm_peak, tf_peak, which = _peaks()
        # kernel-class micro loops: one event pair around many back-to-back launches on the real buffers
        def micro(fn, iters):
            fn(1)
            torch.cuda.synchronize()
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0.record(stream); fn(iters); m1.record(stream)
            torch.cuda.synchronize()
            return m0.elapsed_time(m1) / iters
        ab, gb, gl = C.c_double(0), C.c_double(0), C.c_int(0)
        def attn_loop(sids_, skip):
            arr = (C.c_int32 * len(sids_))(*sids_)
            def f(it):
                rc = eng.lib.vlo_bench_attn(eng._h, len(sids_), arr, 11, it, skip, C.byref(ab), eng._stream()); assert rc == 0, eng.lib.vlo_last_error()
            return f
        run_attn = attn_loop([sid], 0)
        def run_gemm(it):
            rc = eng.lib.vlo_bench_gemm(eng._h, 11, it, C.byref(gb), C.byref(gl), eng._stream()); assert rc == 0, eng.lib.vlo_last_error()
        eng.kv_truncate(sid, KV_START + 11)
        attn_ms = micro(run_attn, 4) / cfg.num_hidden_layers          # per launch pair (main kernel + merge)
        attn_main_ms = micro(attn_loop([sid], 1), 4) / cfg.num_hidden_layers   # main kernel only
        gemm_ms_iter = micro(run_gemm, 4)
        micro_attn = {"us_per_launch_incl_merge": attn_ms * 1e3, "us_main_kernel_only": attn_main_ms * 1e3,
                      "algo_bytes_per_launch": ab.value, "achieved_gbs": ab.value / 1e9 / (attn_ms / 1e3),
                      "achieved_gbs_main_only": ab.value / 1e9 / (attn_main_ms / 1e3)}
        micro_gemm = {"us_per_launch": gemm_ms_iter * 1e3 / gl.value, "algo_bytes_per_launch": gb.value / gl.value,
                      "achieved_gbs": gb.value / 1e9 / (gemm_ms_iter / 1e3), "launches": gl.value}
        names = ["gemm_weight_stream", "attn_kvappend", "attn_merge", "gemm_vit", "vit_attn", "other"]
        cls = {}
        for j, nm in enumerate(names):
            if n[j]:
                cls[nm] = {"launches_per_step": n[j] / P, "ms_per_step": ms[j] / P, "avg_us_per_launch": 1e3 * ms[j] / n[j],
                           "algo_gb_per_step": by[j] / P / 1e9, "achieved_gbs": (by[j] / 1e9) / (ms[j] / 1e3) if ms[j] > 0 else None}
        gs, at = cls.get("gemm_weight_stream"), cls.get("attn_kvappend")
        roof = {"bound": "hbm", "kernel": "gemm_ws_kernel<bf16> / gemm_wsf_kernel (persistent stream-K weight streaming, same mainloop; 14.0 GB of the 16.6 GB/step; "
                          "the micro-loop runs the plain stream-K form of all four GEMMs of a layer, the step fuses the gate|up fix-up)",
                "achieved": micro_gemm["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": micro_gemm["achieved_gbs"] / hbm_peak,
                "peak_source": which, "traffic": _ncu_traffic("gemm_ws_decoder")[0], "traffic_commit": _ncu_traffic("gemm_ws_decoder")[1],
                "avg_us_per_launch": micro_gemm["us_per_launch"], "algo_bytes_per_launch": micro_gemm["algo_bytes_per_launch"],
                "method": "CUDA events around 4 back-to-back passes of the 128 decoder GEMM launches (q|k|v, o, gate|up, down of all 32 layers) on the engine's buffers, T=11",
                "in_step_event_bracketed": {"achieved": gs["achieved_gbs"], "avg_us_per_launch": gs["avg_us_per_launch"],
                                            "note": "per-launch event pairs inside the step (PDL off): includes ~3-5 us bracket overhead per launch"}}
        roof_attn = {"bound": "hbm", "kernel": "attn_tc_kernel + attn_merge_kernel (KV-append attention on tcgen05, one launch pair per layer; attn_tc2_kernel, P in TMEM + key-sliced softmax, takes over from 24k keys)",
                     "achieved": micro_attn["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": micro_attn["achieved_gbs"] / hbm_peak,
                     "peak_source": which, "traffic": _ncu_traffic("attn_tc")[0], "traffic_commit": _ncu_traffic("attn_tc")[1], "avg_us_per_launch": micro_attn["us_per_launch_incl_merge"],
                     "algo_bytes_per_launch": micro_attn["algo_bytes_per_launch"],
                     "method": "CUDA events around 4x32 back-to-back launch pairs over the 32 layers' caches (1.6 GB, > L2), q=11, kv=12011; merge kernel time included",
                     "main_kernel_only": {"achieved": micro_attn["achieved_gbs_main_only"], "frac": micro_attn["achieved_gbs_main_only"] / hbm_peak,
                                          "avg_us_per_launch": micro_attn["us_main_kernel_only"]},
                     "in_step_event_bracketed": {"achieved": at["achieved_gbs"], "avg_us_per_launch": at["avg_us_per_launch"]}}
        step_bytes = 15009316864 + (KV_START + 11 * (K // 2)) * 131072
        roof_step = {"bound": "hbm", "algo_bytes_per_step": step_bytes, "achieved": step_bytes / (ms_total / K / 1e3) / 1e9,
                     "peak": hbm_peak, "unit": "GB/s", "frac": step_bytes / (ms_total / K / 1e3) / 1e9 / hbm_peak}

    # ---- side measurements: the other BASELINE.json configs, every rank runs them and the line carries the aggregate
    #      (units summed over ranks / max time over ranks); reported as extras, not the headline
    extras = None
    if args.extras:
        extras = {}

        def agg_sum(x):
            if dist is None:
                return x
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            return float(t.item())

        def timed(fn):
            """barrier, run fn() (enqueues work on `stream`, may sync), device time via CUDA events, max over ranks"""
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0 = time.perf_counter()
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize()
            wall = time.perf_counter() - w0
            return reduce_max(a.elapsed_time(b) / 1e3), reduce_max(wall)

        # (a) AR response tokens at 12k context: q = 1 steps, id fed back on the device side of the ABI
        eng.kv_truncate(sid, KV_START)
        one = torch.zeros(1, cfg.hidden_size, dtype=torch.bfloat16, device=dev)
        tid = torch.tensor([1234], dtype=torch.int64, device=dev)
        for _ in range(5):
            eng.step([sid], [1], one, row_ids=tid)
        n_ar = 64
        def ar_loop():
            for _ in range(n_ar):
                eng.step([sid], [1], one, row_ids=tid)
        t_dev, _ = timed(ar_loop)
        extras["ar_decode"] = {"tokens_per_s": world * n_ar / t_dev, "ms_per_token": 1e3 * t_dev / n_ar, "kv_tokens": KV_START,
                               "hbm_frac": (15009316864 + KV_START * 131072) / (t_dev / n_ar) / 1e9 / _peaks()[0],
                               "note": "greedy AR step (q=1) of one stream per GPU, device-timed, ids resident"}

        # (b) configs[1] literal: one stream from an EMPTY cache to 1200 frames (10 min @ 2 FPS) through real appends:
        #     first frame = system prompt + frame, then 1199 steady frame steps; KV grows 0 -> ~13.2k
        eng.stream_reset(sid)
        n_lit = 1200 if not args.quick_extras else 120
        start_ids = ByteTokenizer(cfg).apply_chat_template([{'role': 'system', 'content': SYSTEM_PROMPT}], add_stream_prompt=True)
        first_rows = torch.tensor(list(start_ids) + [-1] * 10, dtype=torch.int64, device=dev)
        first_packed = torch.zeros(len(start_ids) + 10, cfg.hidden_size, dtype=torch.bfloat16, device=dev)
        marks = {}
        def literal_step(i, fe):
            if i == 0:
                first_packed[len(start_ids):] = fe
                eng.step([sid], [first_packed.shape[0]], first_packed, row_ids=first_rows, want_logits=True)
            else:
                packed[1:] = fe
                eng.step([sid], [11], packed, row_ids=prefix, want_logits=True)
            if i == n_lit - 101:
                marks["ev"] = torch.cuda.Event(enable_timing=True)
                marks["ev"].record(stream)
                marks["kv"] = eng.kv_len(sid)

        def literal_run():
            pipelined(n_lit, 0, step_fn=literal_step)
            marks["end"] = torch.cuda.Event(enable_timing=True)
            marks["end"].record(stream)
        t_dev, _ = timed(literal_run)
        last100_s = reduce_max(marks["ev"].elapsed_time(marks["end"]) / 1e3)
        extras["config1_literal"] = {"frames": n_lit, "frames_per_s_avg": world * n_lit / t_dev, "frames_per_s_last100": world * 100 / last100_s,
                                     "kv_tokens_end": eng.kv_len(sid), "kv_tokens_at_last100_start": marks["kv"], "seconds": t_dev,
                                     "note": "BASELINE configs[1] run literally: empty cache -> 1200 frames via real KV appends (pipelined ViT), device-timed"}

        # (c) configs[2]: 8 concurrent streams on one GPU (5-min clips -> kv ~6000), ViT batched over the streams,
        #     one ragged decoder step of 8 x 11 tokens per tick
        S8 = n_extra
        eng.stream_reset(sid)
        sids = [sid] + [eng.stream_open() for _ in range(S8 - 1)]
        for i, s_ in enumerate(sids):
            eng.kv_fill_synthetic(s_, 6000, seed=100 + i)
        packed8 = torch.zeros(11 * S8, cfg.hidden_size, dtype=torch.bfloat16, device=dev)
        rid8 = prefix.repeat(S8)
        def tick8(i):
            fe = eng.vit_encode(frames_dev[i:i + S8])
            packed8.view(S8, 11, -1)[:, 1:] = fe.view(S8, 10, -1)
            eng.step(sids, [11] * S8, packed8, row_ids=rid8, want_logits=False)
        for i in range(3):
            tick8(i)
        n_t = min(10, n_frames - S8)
        t_seq, _ = timed(lambda: [tick8(i) for i in range(n_t)])
        # pipelined like the single-stream path: the batch-8 ViT of tick i+1 runs on the side stream during the decoder step
        # of tick i (the 8 cameras deliver their next frames meanwhile); n ticks = n ViT passes + n decoder steps
        fe8 = [None, None]
        ev8 = [torch.cuda.Event(), torch.cuda.Event()]
        def enc8(i, slot, after=None):
            if after is not None:
                side.wait_event(after)
            else:
                side.wait_stream(stream)
            with torch.cuda.stream(side):
                fe8[slot] = eng.vit_encode(frames_dev[i:i + S8])
                ev8[slot].record(side)
        def ticks8_pipelined(n):
            enc8(0, 0)
            for i in range(n):
                stream.wait_event(ev8[i & 1])
                fe = fe8[i & 1]
                fe.record_stream(stream)
                packed8.view(S8, 11, -1)[:, 1:] = fe.view(S8, 10, -1)
                pre_evs[i & 1].record(stream)
                eng.step(sids, [11] * S8, packed8, row_ids=rid8, want_logits=False)
                if i + 1 < n:
                    enc8(i + 1, (i + 1) & 1, after=pre_evs[i & 1])
        ticks8_pipelined(3)
        for s_ in sids:
            eng.kv_truncate(s_, 6000)
        t_dev, _ = timed(lambda: ticks8_pipelined(n_t))
        ab8 = C.c_double(0)
        arr8 = (C.c_int32 * S8)(*sids)
        def attn8(it):
            rc = eng.lib.vlo_bench_attn(eng._h, S8, arr8, 11, it, 0, C.byref(ab8), eng._stream()); assert rc == 0, eng.lib.vlo_last_error()
        attn8(1); torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream); attn8(3); c1.record(stream); torch.cuda.synchronize()
        ms8 = c0.elapsed_time(c1) / 3 / cfg.num_hidden_layers
        hbm_peak8 = _peaks()[0]
        extras["attn_kvappend_8streams"] = {"us_per_launch_incl_merge": ms8 * 1e3, "algo_bytes_per_launch": ab8.value,
                                            "achieved_gbs": ab8.value / 1e9 / (ms8 / 1e3), "frac_of_hbm_peak": ab8.value / 1e9 / (ms8 / 1e3) / hbm_peak8,
                                            "note": "same kernel, ragged batch of 8 streams x 11 query tokens at kv~6.1k each (configs[2] shape)"}
        extras["multistream8"] = {"frames_per_s": world * S8 * n_t / t_dev, "ms_per_tick": 1e3 * t_dev / n_t,
                                  "sequential_frames_per_s": world * S8 * n_t / t_seq, "sequential_ms_per_tick": 1e3 * t_seq / n_t,
                                  "streams": S8 * world, "kv_tokens_start": 6000,
                                  "note": "configs[2]: 8 concurrent streams/GPU, ViT batch 8 + one ragged 88-token decoder step per tick, "
                                          "ViT of tick i+1 on the side stream during the step of tick i (sequential variant beside it), device-timed"}

        # (d) configs[4]: 8 streams/GPU (64 on 8 GPUs), mixed speak/silent with AR bursts up to 128 tokens, through the
        #     multi-stream scheduler (one ragged step per tick carries frame steps, response prompts and AR tokens of
        #     different streams).  Scripted protocol (random weights never emit it): stream s speaks at every 5th frame
        #     (staggered by s), response lengths ~ seeded uniform{8..128}.
        import random
        from videollm_online_b200.multistream import StreamScheduler
        for s_ in sids:
            eng.stream_close(s_)
        sch = StreamScheduler(model, ByteTokenizer(cfg), S8, frame_fps=2, system_prompt=SYSTEM_PROMPT, max_new_tokens=128)
        rng = random.Random(1234 + rank)
        lens = [[rng.randint(8, 128) for _ in range(64)] for _ in range(S8)]
        n_resp, n_frames_seen = [0] * S8, [0] * S8
        I_, E_, END_, A_ = cfg.frame_token_interval_id, cfg.eos_token_id, cfg.stream_end_id, 300
        def mixed_hook(s_, d, n):
            sess = sch.sessions[s_]
            if sess._op[0] == "gen":
                want = lens[s_][n_resp[s_] % 64]
                tok = E_ if len(sess.resp) + 1 >= want else A_
                if tok == E_:
                    n_resp[s_] += 1
            else:
                k = n_frames_seen[s_]
                n_frames_seen[s_] += 1
                tok = END_ if (k > 0 and k % 5 == s_ % 5) else I_
            d.argmax_id = d.argmax_prob_id = tok
            d.p_interval = 1.0 if tok == I_ else 0.0
            if tok != I_:
                d.argmax_excl_id = tok
            return d
        sch.decision_hook = mixed_hook
        clip = frames_dev[:min(n_frames, 32)]
        for k, sess in enumerate(sch.sessions):
            sess.load_video(torch.roll(clip, k, 0).repeat(4, 1, 1, 1))
            eng.kv_fill_synthetic(sess.stream_id, 6000, seed=300 + k)
            sess.started, sess.last_ids = True, [I_]
        n_ticks = 24 if not args.quick_extras else 8
        def mixed_run():
            for i in range(n_ticks):
                for sess in sch.sessions:
                    sess.input_video_stream(i / 2)
                while any(sess.pending_frames for sess in sch.sessions):   # bursts keep running across frame arrivals
                    sch.tick()
            sch.run_until_idle()
        _, t_wall = timed(mixed_run)
        toks = sum(len(ev[2]) for sess in sch.sessions for ev in sess.events if ev[0] == "response")
        extras["config4_mixed"] = {"streams": S8 * world, "frames_per_s": agg_sum(sch.frames_done) / t_wall, "response_tokens_per_s": agg_sum(toks) / t_wall,
                                   "responses": agg_sum(sum(n_resp)), "ticks": agg_sum(sch.ticks) / world, "seconds": t_wall, "max_new_tokens": 128,
                                   "note": "configs[4]: 8 streams/GPU through StreamScheduler, scripted speak every 5th frame (staggered), response "
                                           "lengths uniform{8..128}; wall time incl. the per-tick decision read-back (end to end)"}
        for sess in sch.sessions:
            eng.stream_close(sess.stream_id)

        # (e) configs[3]: 1 stream/GPU at 10 FPS x 10 min = 66k-token cache (second engine on the SAME weight tensors, 8.7 GB of KV)
        KV66 = 66000
        w66 = dict(weights)
        w66["rope.cos"], w66["rope.sin"] = W.rope_tables(cfg, KV66 + 512, dev)
        eng66 = Engine(cfg, dev, max_streams=1, max_kv_tokens=KV66 + 512, max_step_tokens=128, max_vit_batch=1)
        eng66.load_weights(w66)
        s66 = eng66.stream_open()
        eng66.kv_fill_synthetic(s66, KV66, seed=66 + rank)
        def step66(i):
            fe = eng.vit_encode(frames_dev[i:i + 1])
            packed[1:] = fe
            eng66.step([s66], [11], packed, row_ids=prefix, want_logits=True)
        for i in range(3):
            step66(i)
        n66 = 10
        t_dev, _ = timed(lambda: [step66(i) for i in range(n66)])
        b66 = 15009316864 + (KV66 + 11 * 8) * 131072
        extras["config3_66k"] = {"frames_per_s": world * n66 / t_dev, "ms_per_step": 1e3 * t_dev / n66, "kv_tokens": KV66,
                                 "algo_bytes_per_step": b66, "hbm_frac": b66 / (t_dev / n66) / 1e9 / _peaks()[0],
                                 "meets_10fps_per_stream": (n66 / t_dev) >= 10.0,
                                 "note": "configs[3]: 1 stream/GPU at the 10 FPS x 10 min position (66k-token KV), sequential ViT + frame step, device-timed"}
        eng66.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return None
    fps = world * K / (ms_total / 1e3)
    e2e_fps = world * K / e2e_s
    line = {"metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": static_config(world),
            "run": {"kv_tokens_end": kv_end, "sequential_ms_per_step": seq_ms, "sequential_frames_per_s": world * 1e3 / seq_ms,
                    "weight_broadcast_s": bcast_s},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_fps, "unit": UNIT, "h2d_bytes_per_step": int(3 * S * S + 11 * 4 * 2 + 8), "d2h_bytes_per_step": 32,
                    "ms_per_step": 1e3 * e2e_s / K, "api": "LiveLlamaForCausalLM.visual_embed + Engine.step (vlo_vit_encode / vlo_step_ids) + read_decisions",
                    "liveinfer": {"value": world * K / e2e_li_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_li_s / K,
                                  "h2d_bytes_per_step": int(3 * S * S), "d2h_bytes_per_step": 32,
                                  "api": "LiveInfer.input_video_stream + LiveInfer.__call__ per frame (demo/cli.py:31-38 loop), pinned-host clip, decision read back",
                                  "vs_engine_api": (world * K / e2e_li_s) / e2e_fps}},
            "roofline": roof, "roofline_attn": roof_attn, "roofline_step": roof_step, "kernel_classes": cls}
    if extras:
        line["extras"] = extras
    if world == 1 and not args.no_cpu_baseline:
        per_step, info = cpu_reference_times(2, 1, budget_s=45.0)
        line["cpu_baseline"] = {"value": 1.0 / per_step, "unit": UNIT, "cores": info["threads"], "kind": "port",
                                "sample": info["sample"], "host_cpus": os.cpu_count(), "extrapolated": info["extrapolated"],
                                "per_step_s": info["per_step_s"], "rel_std": info["rel_std"],
                                "vit_s_per_frame": info["vit_s_per_frame"], "decoder_s_per_step": info["decoder_s_per_step"]}
    if dist is not None:
        dist.destroy_process_group()
    return line


class _StdoutToStderr:
    """Everything except the ONE JSON line goes to stderr (NCCL prints its version banner on stdout)."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--encode-ahead", dest="encode_ahead", type=int, default=1,
                    help="frames per encode-ahead ViT pass on the side stream (1 = one frame at a time: the small-tile ViT "
                         "co-resides with the decoder step; >= 3 = 2-CTA tensor-bound GEMMs, serialised against the step)")
    ap.add_argument("--no-extras", dest="extras", action="store_false", help="skip the side measurements of the other BASELINE configs")
    ap.add_argument("--quick-extras", dest="quick_extras", action="store_true", help="shorter side measurements (dev runs)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write what the last timed frame step computed (frame embeddings, logits, decision) to DIR/<name>.npy; "
                         "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA engine's outputs; the reference arm has none")
    with _StdoutToStderr() as guard:
        line = run_reference_arm(args) if args.impl == "reference" else run_engine_arm(args)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
