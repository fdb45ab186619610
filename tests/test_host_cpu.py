"""CPU-side tests: C-ABI surface, host logic, tokenizer/template, weight packing, multi-process plumbing."""
import ctypes as C
import os
import pathlib
import re
import subprocess
import sys

import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol():
    from videollm_online_b200 import _lib
    lib = _lib.load()
    header = (ROOT / "include" / "vlo_b200.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(vlo_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/vlo_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)


def test_struct_layouts_match_header():
    from videollm_online_b200._lib import VloConfig, VloDecision
    assert C.sizeof(VloDecision) == 32
    assert C.sizeof(VloConfig) == 22 * 4


def test_no_gpu_means_loud_failure_not_fallback():
    from videollm_online_b200 import VloError, tiny_config
    from videollm_online_b200.engine import Engine
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(VloError):
        Engine(tiny_config(), "cuda:0")
    with pytest.raises(VloError):
        Engine(tiny_config(), "cpu")


def test_product_package_never_imports_the_oracle():
    pkg = ROOT / "videollm-online_b200"
    for f in list(pkg.glob("*.py")) + list((pkg / "csrc").glob("*")):
        txt = f.read_text(errors="ignore")
        assert "vlo_oracle" not in txt and "import oracle" not in txt, f


def test_chat_template_pieces():
    from videollm_online_b200 import tiny_config
    from videollm_online_b200.tokenization_live import ByteTokenizer, render_chat
    cfg = tiny_config()
    tok = ByteTokenizer(cfg)
    kw = dict(bos_token="<B>", eos_token="<E>")
    assert render_chat([{"role": "system", "content": "S"}], add_stream_prompt=True, **kw) == "<B>S\n\n["
    assert render_chat([{}], add_stream_prompt=True, **kw) == "\n["
    assert render_chat([{}], add_stream_generation_prompt=True, **kw) == "]\nAssistant:"
    assert render_chat([{"role": "user", "content": "Q"}], add_stream_query_prompt=True, add_generation_prompt=True, **kw) == "]\nUser: Q\nAssistant:"
    conv = [{"role": "system", "content": "S"}, {"role": "stream", "num_frames": 2}, {"role": "user", "content": "Q"},
            {"role": "assistant", "content": "A"}]
    ph = lambda n: ",".join(["<v>" * 10] * n)
    assert render_chat(conv, stream_placeholder=ph, **kw) == "<B>S\n\n[" + "<v>" * 10 + "," + "<v>" * 10 + "]\nUser: Q\nAssistant: A<E>"
    ids = tok.apply_chat_template([{}], add_stream_generation_prompt=True)
    assert ids[0] == cfg.stream_end_id                      # "]\n" is ONE id, as demo/inference.py:44 assumes
    assert tok.encode(",") == [cfg.frame_token_interval_id]
    assert tok.decode(tok.encode("hello, wörld")) == "hello, wörld"


def test_parse_args_two_pass_presets():
    from videollm_online_b200.config import parse_args
    a = parse_args([])
    assert (a.live_version, a.frame_num_tokens, a.frame_token_pooled, a.frame_token_interval, a.max_num_frames) == ("live1+", 10, [3, 3], ",", 1200)
    b = parse_args(["--live_version", "live1", "--frame_fps", "10"])
    assert (b.frame_num_tokens, b.frame_token_pooled, b.frame_token_interval, b.max_num_frames, b.frame_fps) == (1, None, "", 7200, 10)


def test_pack_layout_and_lora_merge():
    from videollm_online_b200 import tiny_config, weights as W
    from videollm_online_b200.dist import engine_weight_spec
    cfg = tiny_config()
    sd, vs = W.synthetic_llm_state(cfg), W.synthetic_vision_state(cfg)
    packed = W.pack_llm_for_engine(cfg, sd, "cpu", 256)
    packed.update(W.pack_vision_for_engine(cfg, vs, "cpu"))
    spec = engine_weight_spec(cfg, 256)
    assert set(spec) == set(packed)
    for k, (shape, dt) in spec.items():
        assert tuple(packed[k].shape) == tuple(shape) and packed[k].dtype == dt, k
    assert torch.equal(packed["L0.qkv"][: cfg.num_attention_heads * 128], sd["model.layers.0.self_attn.q_proj.weight"])
    # gate | up are tile-interleaved: 128-row tile j = gate rows 64j..64j+63, then the matching up rows
    gu = packed["L1.gate_up"].view(cfg.intermediate_size // 64, 2, 64, cfg.hidden_size)
    assert torch.equal(gu[:, 0].reshape(cfg.intermediate_size, -1), sd["model.layers.1.mlp.gate_proj.weight"])
    assert torch.equal(gu[:, 1].reshape(cfg.intermediate_size, -1), sd["model.layers.1.mlp.up_proj.weight"])
    # LoRA merge == unmerged forward (y = W x + 2 B A x) up to bf16 rounding of the merged weight
    g = torch.Generator().manual_seed(0)
    r = 8
    key = "model.layers.0.self_attn.q_proj"
    A = (torch.randn(r, cfg.hidden_size, generator=g) * 0.05).bfloat16()
    B = (torch.randn(cfg.num_attention_heads * 128, r, generator=g) * 0.05).bfloat16()
    merged = W.merge_lora(sd, {f"base_model.model.{key}.lora_A.default.weight": A, f"base_model.model.{key}.lora_B.default.weight": B,
                               "base_model.model.connector.modules_to_save.default.0.bias": torch.ones(cfg.hidden_size)},
                          lora_alpha=16, lora_r=r)
    x = torch.randn(5, cfg.hidden_size, generator=g)
    want = x @ sd[key + ".weight"].float().t() + 2.0 * (x @ A.float().t()) @ B.float().t()
    got = x @ merged[key + ".weight"].float().t()
    assert (got - want).abs().max() < 0.05 * want.abs().max()
    assert torch.equal(merged["connector.0.bias"], torch.ones(cfg.hidden_size, dtype=torch.bfloat16))


def test_rope_tables_match_hf_formula():
    sys.path.insert(0, str(ROOT / "oracle"))
    import vlo_oracle as O
    from videollm_online_b200 import tiny_config, weights as W
    cfg = tiny_config()
    cos, sin = W.rope_tables(cfg, 300, "cpu")
    c2, s2 = O.rope_cos_sin(cfg, torch.arange(300)[None], torch.bfloat16)
    assert torch.equal(cos, c2[0, :, :64]) and torch.equal(sin, s2[0, :, :64])
    assert torch.equal(c2[0, :, :64], c2[0, :, 64:])


def test_decision_threshold_semantics():
    from videollm_online_b200.engine import Decision
    row_i = torch.tensor([7, 9, 0, 0, 0, 0, 7, 0], dtype=torch.int32)
    f = row_i.view(torch.float32).clone()
    f[2] = 0.7265625            # bf16 value just above 0.725: torch compares against bf16(0.725) = 0.7265625
    d = Decision(row_i, f)
    assert d.next_id(7, 0.725) == 7 and d.next_id(7, 0.727) == 7 and d.next_id(7, 0.74) == 9


@pytest.mark.timeout(180)
def test_weight_broadcast_two_ranks_gloo(tmp_path):
    """N>1 plumbing on CPU: rank 0 owns the weights, rank 1 receives identical tensors (gloo, 127.0.0.1)."""
    script = tmp_path / "bc.py"
    script.write_text(f"""
import sys, torch, torch.distributed as dist
sys.path.insert(0, {str(ROOT)!r})
import vlo_bootstrap
from videollm_online_b200 import tiny_config, weights as W
from videollm_online_b200.dist import broadcast_weights
dist.init_process_group('gloo')
cfg = tiny_config()
full = W.pack_llm_for_engine(cfg, W.synthetic_llm_state(cfg), 'cpu', 128)
full.update(W.pack_vision_for_engine(cfg, W.synthetic_vision_state(cfg), 'cpu'))
got = broadcast_weights(cfg, full if dist.get_rank() == 0 else None, 'cpu', 128, dist)
assert set(got) == set(full) and all(torch.equal(got[k], full[k]) for k in full)
# coalesced: <= 8 flat buffers carry every tensor, each view 256-byte aligned inside its buffer
stores = {{t.untyped_storage().data_ptr() for t in got.values()}}
assert len(stores) <= 8 and all((t.data_ptr() - t.untyped_storage().data_ptr()) % 256 == 0 for t in got.values())
# static stream -> rank assignment: round-robin, every stream owned by exactly one rank
streams = list(range(5)); mine = [s for s in streams if s % dist.get_world_size() == dist.get_rank()]
cnt = torch.tensor([len(mine)]); dist.all_reduce(cnt); assert int(cnt) == 5
sys.stdout.write('rank %d ok\\n' % dist.get_rank()); sys.stdout.flush()   # one write per rank: the two ranks share the pipe
""")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    import socket
    with socket.socket() as so:          # a free rendezvous port (a fixed one can still be in TIME_WAIT from the last run)
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), str(script)], capture_output=True, text=True, env=env, timeout=170)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout


@pytest.mark.timeout(300)
def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs) prints exactly one JSON line with the contract keys."""
    import json
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_checkpoint_directory_loader_roundtrip(tmp_path):
    """SURVEY 8(f).1: base-model safetensors shards + a PEFT adapter directory (LoRA A/B on the Linear layers the
    reference targets, `modules_to_save=['connector']`, both saved-key spellings) + a SigLIP directory, read by the
    same code path `build_live(llm_pretrained=..., resume_from_checkpoint=...)` uses, equal the in-memory packing."""
    from safetensors.torch import save_file
    from videollm_online_b200 import tiny_config, weights as W
    from videollm_online_b200.modeling_live import _load_checkpoints
    cfg = tiny_config()
    full, vs = W.synthetic_llm_state(cfg, seed=4), W.synthetic_vision_state(cfg, seed=5)
    base = {k: v for k, v in full.items() if not k.startswith("connector.")}     # the base LLM has no connector
    keys = sorted(base)
    llm_dir, ad_dir, vis_dir = tmp_path / "llm", tmp_path / "adapter", tmp_path / "siglip"
    for d in (llm_dir, ad_dir, vis_dir):
        d.mkdir()
    save_file({k: base[k].contiguous() for k in keys[: len(keys) // 2]}, str(llm_dir / "model-00001-of-00002.safetensors"))
    save_file({k: base[k].contiguous() for k in keys[len(keys) // 2:]}, str(llm_dir / "model-00002-of-00002.safetensors"))
    g = torch.Generator().manual_seed(9)
    r, alpha = 8, 16
    adapter = {}
    for i in range(cfg.num_hidden_layers):
        for j, name in enumerate(("self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", "self_attn.o_proj",
                                  "mlp.gate_proj", "mlp.up_proj", "mlp.down_proj")):
            w = base[f"model.layers.{i}.{name}.weight"]
            infix = ".default" if (i + j) % 2 else ""        # PEFT state_dict() vs saved-adapter spelling
            adapter[f"base_model.model.model.layers.{i}.{name}.lora_A{infix}.weight"] = (torch.randn(r, w.shape[1], generator=g) * 0.05).bfloat16()
            adapter[f"base_model.model.model.layers.{i}.{name}.lora_B{infix}.weight"] = (torch.randn(w.shape[0], r, generator=g) * 0.05).bfloat16()
    adapter["base_model.model.lm_head.lora_A.weight"] = (torch.randn(r, cfg.hidden_size, generator=g) * 0.05).bfloat16()
    adapter["base_model.model.lm_head.lora_B.weight"] = (torch.randn(cfg.vocab_size, r, generator=g) * 0.05).bfloat16()
    for k in ("connector.0.weight", "connector.0.bias", "connector.2.weight", "connector.2.bias"):
        adapter["base_model.model." + k] = full[k].contiguous()
    save_file(adapter, str(ad_dir / "adapter_model.safetensors"))
    save_file({"vision_model." + k: v.contiguous() for k, v in vs.items()} | {"text_model.unused": torch.zeros(3)},
              str(vis_dir / "model.safetensors"))
    cfg.vision_pretrained = str(vis_dir)
    got = _load_checkpoints(cfg, str(llm_dir), str(ad_dir), True, "cpu", 256, r, alpha)
    want = W.pack_llm_for_engine(cfg, W.merge_lora(dict(base), adapter, lora_alpha=alpha, lora_r=r), "cpu", 256)
    want.update(W.pack_vision_for_engine(cfg, vs, "cpu"))
    assert set(got) == set(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    # adapter_config.json (written by PEFT next to the weights) overrides the CLI defaults for r / lora_alpha
    import json
    (ad_dir / "adapter_config.json").write_text(json.dumps({"r": r, "lora_alpha": alpha, "peft_type": "LORA"}))
    got2 = _load_checkpoints(cfg, str(llm_dir), str(ad_dir), False, "cpu", 256, 999, 1.0)
    assert torch.equal(got2["L0.qkv"], want["L0.qkv"]) and torch.equal(got2["lm_head"], want["lm_head"])
    # the adapter really changed the weights, and the connector came from the adapter
    assert not torch.equal(got["L0.qkv"], W.pack_llm_for_engine(cfg, full, "cpu", 256)["L0.qkv"])
    assert torch.equal(got["conn.0.w"], full["connector.0.weight"])
    assert not torch.equal(got["lm_head"], full["lm_head.weight"])         # lora_modules ends with |lm_head$ (models/arguments_live.py:16)
    # missing directory: loud failure, no silent random init (the reference only warns, models/modeling_live.py:218)
    from videollm_online_b200._lib import VloError
    with pytest.raises(VloError):
        _load_checkpoints(cfg, str(tmp_path / "nope"), "", False, "cpu", 256, r, alpha)


def test_video_ingest_matches_ffmpeg_once_geometry(tmp_path):
    """SURVEY 8(f).2: decode + `-r fps` + scale/pad of data/utils.py:51-66, restated with OpenCV (no ffmpeg here)."""
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    from videollm_online_b200.video_ingest import letterbox_geometry, read_video_resampled, resample_indices
    # geometry of the filter chain: longer side -> R, shorter side even, centred
    assert letterbox_geometry(640, 360, 384) == (384, 216, 0, 84)
    assert letterbox_geometry(360, 640, 384) == (216, 384, 84, 0)
    assert letterbox_geometry(500, 500, 384) == (384, 384, 0, 0)
    assert letterbox_geometry(1280, 718, 384)[1] % 2 == 0
    # 30 fps -> 2 fps: output k shows the source frame nearest to k / 2 s
    assert resample_indices(60, 30.0, 2) == [0, 15, 30, 45]
    assert resample_indices(0, 30.0, 2) == [] and resample_indices(10, 30.0, 2) == [0]
    path = str(tmp_path / "clip.avi")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 30.0, (640, 360))
    if not w.isOpened():
        pytest.skip("no MJPG encoder in this OpenCV build")
    for i in range(60):
        f = np.full((360, 640, 3), 40, np.uint8)
        f[100:200, 8 * i:8 * i + 100] = (0, 0, 255)      # a red (BGR) square moving right, 8 px per source frame
        w.write(f)
    w.release()
    v = read_video_resampled(path, fps=2, resolution=384)
    assert v.dtype == torch.uint8 and tuple(v.shape) == (4, 3, 384, 384)
    assert int(v[:, :, :84].max()) == 0 and int(v[:, :, 300:].max()) == 0     # black bars above and below
    assert int(v[:, :, 84:300].float().mean()) > 20                            # picture in the middle band
    for k, src in enumerate((0, 15, 30, 45)):                                  # the square sits where source frame `src` had it
        red = v[k, 0, 84:300].float() - v[k, 2, 84:300].float()                # RGB order: R - B
        cols = (red.mean(0) > 60).nonzero().flatten()
        centre = float(cols.float().mean())
        want = (8 * src + 50) * 384 / 640
        assert abs(centre - want) < 4, (k, centre, want)
    raw = read_video_resampled(path)                                            # no resampling requested: every frame, native size
    assert tuple(raw.shape) == (60, 3, 360, 640)
    with pytest.raises(RuntimeError):
        read_video_resampled(str(tmp_path / "missing.mp4"))


def test_video_ingest_of_the_reference_demo_clips():
    """The clips demo/cli.py:12 plays (demo/assets/cooking.mp4 1440x1080, bicycle.mp4 512x384, 30 fps), streamed through
    the ingest at the demo's 2 FPS / 384 px: their first second as stored in tests/golden (make_golden.py clips; cooking
    scaled to 480x360, the same 4:3 letterbox)."""
    pytest.importorskip("cv2")
    from videollm_online_b200.video_ingest import letterbox_geometry, read_video_resampled
    assert letterbox_geometry(1440, 1080, 384) == (384, 288, 0, 48)
    for name, (w, h, n_src) in {"cooking": (480, 360, 30), "bicycle": (512, 384, 30)}.items():
        v = read_video_resampled(str(ROOT / "tests" / "golden" / f"demo_{name}_excerpt.mp4"), fps=2, resolution=384)
        n_out = round(n_src / 30.0 * 2)
        assert v.dtype == torch.uint8 and tuple(v.shape) == (n_out, 3, 384, 384), (name, tuple(v.shape))
        sw, sh, x0, y0 = letterbox_geometry(w, h, 384)
        assert (sw, sh, x0, y0) == (384, 288, 0, 48)
        assert int(v[:, :, :y0].max()) == 0 and int(v[:, :, y0 + sh:].max()) == 0         # black bars of the pad filter
        band = v[:, :, y0:y0 + sh].float()
        assert band.mean() > 30 and band.std() > 20                                         # a real picture in between
        assert (v[0].float() - v[-1].float()).abs().mean() > 2                              # and it changes over the clip


def test_offline_encode_directory_layout_and_sharding(tmp_path, tiny):
    """SURVEY 8(f).3: the host loop of distributed_encode (data/utils.py:86-104) - clip -> batches -> tokens -> .pt,
    round-robin over ranks - driven here with the CPU oracle's SigLIP encode as the `vision_encode` callable."""
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    sys.path.insert(0, str(ROOT / "oracle"))
    import vlo_oracle as O
    from videollm_online_b200.offline_encode import encode_directory, encoded_root
    cfg, _, vs = tiny
    R = cfg.frame_resolution
    src = tmp_path / "clips_2fps_384"
    src.mkdir()
    rng = np.random.default_rng(0)
    n_frames = {"a.avi": 5, "b.avi": 3, "c.avi": 4}
    for name, n in n_frames.items():
        w = cv2.VideoWriter(str(src / name), cv2.VideoWriter_fourcc(*"MJPG"), 2.0, (R, R))
        if not w.isOpened():
            pytest.skip("no MJPG encoder in this OpenCV build")
        for _ in range(n):
            w.write(rng.integers(0, 256, (R, R, 3), dtype=np.uint8))
        w.release()
    calls = []

    def vision_encode(encoder, frames):
        calls.append(int(frames.shape[0]))
        return O.siglip_vision_encode(vs, cfg, frames)

    kw = dict(src_root=str(src) + "/", vision_pretrained="google/siglip-large-patch16-384", vision_encode=vision_encode,
              batch_size=2, embed_mark="2fps_384_1+3x3", save_bf16=True, world_size=2)
    w0 = encode_directory(rank=0, **kw)
    w1 = encode_directory(rank=1, **kw)
    dst = encoded_root(str(src), "2fps_384_1+3x3", "google/siglip-large-patch16-384")
    assert dst.endswith("clips_2fps_384_1+3x3_google--siglip-large-patch16-384")
    assert [os.path.basename(p) for p in w0] == ["a.pt", "c.pt"] and [os.path.basename(p) for p in w1] == ["b.pt"]
    assert calls == [2, 2, 1, 2, 2, 2, 1]                                  # batches of <= 2 frames per clip
    for name, n in n_frames.items():
        t = torch.load(os.path.join(dst, name.replace(".avi", ".pt")), weights_only=True)
        assert t.dtype == torch.bfloat16 and tuple(t.shape) == (n, cfg.frame_num_tokens, cfg.vision_hidden_size)
    # the saved tokens are the encoder's tokens of the decoded frames
    from videollm_online_b200.video_ingest import read_video_resampled
    fr = read_video_resampled(str(src / "b.avi"))
    want = O.siglip_vision_encode(vs, cfg, fr).to(torch.bfloat16)
    assert torch.equal(torch.load(os.path.join(dst, "b.pt"), weights_only=True), want)


def test_committed_bench_records_carry_the_contract_keys():
    """The bench lines measured on the B200 box this round (profiles/r01_bench_n*.json) have every key the driver's
    contract names; guards bench.py's JSON against silently dropping one."""
    import json
    base = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}
    for n in (1, 4, 8):
        d = json.loads((ROOT / "profiles" / f"r01_bench_n{n}.json").read_text().strip().splitlines()[-1])
        assert base <= set(d), base - set(d)
        assert d["n_gpus"] == n and d["scaling"] == "weak" and d["higher_is_better"] is True and d["vs_baseline"] is None
        assert "workload" in d["config"] and "model" not in d["config"]
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
        assert d["e2e"]["h2d_bytes_per_step"] >= 3 * 384 * 384 and d["e2e"]["d2h_bytes_per_step"] == 32   # frame in, decision out
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
        assert d["gpu_launches"] > 0 and d["warmup"] >= 3
        assert abs(d["value"] - n * d["steps"] / (d["ms_per_step"] * d["steps"] / 1e3)) < 1e-6 * d["value"]
        if n == 1:
            assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
    d1 = json.loads((ROOT / "profiles" / "r01_bench_n1.json").read_text().strip().splitlines()[-1])
    d8 = json.loads((ROOT / "profiles" / "r01_bench_n8.json").read_text().strip().splitlines()[-1])
    assert d8["value"] / d1["value"] >= 7.5            # north_star: >= 7.5x aggregate frames/s at 8 GPUs vs 1


def test_streamk_plan_through_the_c_abi_matches_its_definition():
    """Stream-K decomposition of the persistent weight-streaming GEMM (csrc/streamk.h), queried through the C ABI's
    planning call (d_out = NULL: no GPU work): units = (128-row tile, 64-wide k-block), CTA c owns
    [floor(c*U/G), floor((c+1)*U/G)); a tile's partial planes = contributing CTAs.  The fix-up kernels unroll 8 planes."""
    import bisect
    import ctypes as C
    from videollm_online_b200 import _lib
    lib = _lib.load()

    def planes_by_definition(rows_w, k, G, x_tiles=1):
        tiles, kb = -(-rows_w // 128) * x_tiles, k // 64
        U = tiles * kb
        G = min(G, U)
        lo = [(c * U) // G for c in range(G + 1)]
        owner = lambda u: bisect.bisect_right(lo, u) - 1
        return max(owner((t + 1) * kb - 1) - owner(t * kb) + 1 for t in range(tiles))

    shapes = {"qkv": (6144, 4096), "o": (4096, 4096), "gate_up": (28672, 4096), "down": (4096, 14336),
              "vit_out": (1024, 1024), "vit_fc2": (1024, 4096), "tiny": (256, 128), "one_tile": (128, 64)}
    for name, (n, k) in shapes.items():
        for G in (148, 132, 16, 3, 1):
            for T in (11, 88):
                got = C.c_int(-1)
                rc = lib.vlo_op_gemm_ws(1, 0, None, n, None, T, k, None, n, T * n, None, 0, G, 0, C.byref(got), None)
                assert rc == 0, lib.vlo_last_error()
                bn = 16 if T <= 16 else 32 if T <= 32 else 64 if T <= 64 else 128
                want = planes_by_definition(n, k, G, -(-T // bn))
                assert got.value == want, (name, G, T, got.value, want)
                if G == 148 and name in ("qkv", "o", "gate_up", "down"):
                    assert got.value <= 8          # kFixMaxPlanes of the decoder fix-up kernels
