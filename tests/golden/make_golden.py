"""Generate the golden fixtures by RUNNING THE REFERENCE's own modules (CPU) on seeded inputs.

    python tests/golden/make_golden.py            # tiny_reference.pt
    python tests/golden/make_golden.py forward    # reference_forward.json: digests of the reference's forward on this host
    python tests/golden/make_golden.py clips      # demo_{bicycle,cooking}_excerpt.mp4: excerpts of the demo's clips

Each reads a checkout of the reference (VLO_REFERENCE), the first two with transformers, the third with OpenCV;
the tests need only the fixtures.
The reference (showlab/videollm-online @ e2c78ec) has no numeric tests, so these
fixtures are the pin for oracle/vlo_oracle.py: same seeded weights (videollm_online_b200.weights),
same inputs, outputs of `LiveLlamaForCausalLM` / `_siglip_vision_encode` / `fast_greedy_generate` /
`LiveInfer` methods executed unmodified under transformers 5.5.0.  Import recipe from SURVEY.md §8(c):
import transformers.Trainer first, insert a stub `peft`, shim torchvision.io.read_video.
"""
import hashlib
import importlib.machinery
import json
import os
import pathlib
import sys
import types
from functools import partial

import torch

ROOT = pathlib.Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
import vlo_bootstrap  # noqa: E402,F401
from videollm_online_b200 import tiny_config  # noqa: E402
from videollm_online_b200 import weights as W  # noqa: E402
from videollm_online_b200.config import SYSTEM_PROMPT  # noqa: E402
from videollm_online_b200.tokenization_live import ByteTokenizer  # noqa: E402

REF = os.environ.get("VLO_REFERENCE", "/root/reference")
OUT = pathlib.Path(__file__).resolve().parent


def import_reference():
    from transformers import TrainingArguments, Trainer  # noqa: F401  (must precede the peft stub)
    peft = types.ModuleType("peft")
    peft.__spec__ = importlib.machinery.ModuleSpec("peft", None)
    peft.LoraConfig = peft.get_peft_model = peft.PeftModel = object
    sys.modules["peft"] = peft
    import torchvision.io
    if not hasattr(torchvision.io, "read_video"):
        torchvision.io.read_video = lambda *a, **k: (_ for _ in ()).throw(RuntimeError("read_video shim"))
    import torchvision
    torchvision.set_video_backend = lambda *a, **k: None
    sys.path.insert(0, REF)
    import models  # noqa: F401
    from models.live_llama import LiveLlamaConfig, LiveLlamaForCausalLM
    from models.vision_live import _siglip_vision_encode
    from models.modeling_live import fast_greedy_generate
    import demo.inference as ref_inf
    return LiveLlamaConfig, LiveLlamaForCausalLM, _siglip_vision_encode, fast_greedy_generate, ref_inf


def build_reference_model(cfg, llm_state, vision_state):
    LiveLlamaConfig, LiveLlamaForCausalLM, _siglip_vision_encode, fgg, ref_inf = import_reference()
    from transformers import SiglipVisionConfig, SiglipVisionModel
    hf_cfg = LiveLlamaConfig(
        hidden_size=cfg.hidden_size, num_hidden_layers=cfg.num_hidden_layers, num_attention_heads=cfg.num_attention_heads,
        num_key_value_heads=cfg.num_key_value_heads, head_dim=cfg.head_dim, intermediate_size=cfg.intermediate_size,
        vocab_size=cfg.vocab_size, rms_norm_eps=cfg.rms_norm_eps, rope_theta=cfg.rope_theta,
        max_position_embeddings=cfg.max_position_embeddings, bos_token_id=cfg.bos_token_id, eos_token_id=cfg.eos_token_id,
        tie_word_embeddings=False, attention_bias=False, mlp_bias=False,
        vision_hidden_size=cfg.vision_hidden_size, frame_resolution=cfg.frame_resolution, frame_token_cls=cfg.frame_token_cls,
        frame_token_pooled=cfg.frame_token_pooled, frame_num_tokens=cfg.frame_num_tokens, v_placeholder_id=cfg.v_placeholder_id,
        frame_token_interval=cfg.frame_token_interval, frame_token_interval_id=cfg.frame_token_interval_id,
        attn_implementation="sdpa", torch_dtype=torch.bfloat16)
    # from_pretrained(torch_dtype=bf16) instantiates under a bf16 default dtype: parameters are bf16 while
    # the rotary inv_freq buffer is computed explicitly in fp32 (a later .to(bf16) would wrongly round it)
    torch.set_default_dtype(torch.bfloat16)
    try:
        model = LiveLlamaForCausalLM(hf_cfg).eval()
    finally:
        torch.set_default_dtype(torch.float32)
    assert model.model.rotary_emb.inv_freq.dtype == torch.float32 and model.lm_head.weight.dtype == torch.bfloat16
    assert abs(model.config.rope_parameters["rope_theta"] - cfg.rope_theta) < 1e-6
    missing, unexpected = model.load_state_dict(llm_state, strict=False)
    assert not unexpected and all("rotary" in m or "inv_freq" in m for m in missing), (missing, unexpected)
    vcfg = SiglipVisionConfig(hidden_size=cfg.vision_hidden_size, intermediate_size=cfg.vision_intermediate_size,
                              num_hidden_layers=cfg.vision_num_hidden_layers, num_attention_heads=cfg.vision_num_attention_heads,
                              image_size=cfg.frame_resolution, patch_size=cfg.vision_patch_size,
                              layer_norm_eps=cfg.vision_layer_norm_eps, attn_implementation="sdpa")
    vision = SiglipVisionModel(vcfg).vision_model.eval()
    missing, unexpected = vision.load_state_dict(vision_state, strict=False)
    assert not unexpected and all("position_ids" in m for m in missing), (missing, unexpected)
    # exactly what LiveMixin.set_vision_inside does (models/modeling_live.py:12-15), minus the hub download
    model.vision_encoder = vision
    model.vision_encode = partial(_siglip_vision_encode, frame_token_cls=cfg.frame_token_cls,
                                  frame_token_pooled=cfg.frame_token_pooled)
    model.requires_grad_(False)
    return model, fgg, ref_inf


class ScriptedModel:
    """Wraps the reference model: after each forward, boosts one scripted id in the LAST logits row.
    schedule[call_index] = token id (absent -> natural logits)."""

    def __init__(self, model, schedule):
        self.model, self.schedule, self.calls = model, schedule, 0
        self.config = model.config

    def get_input_embeddings(self):
        return self.model.get_input_embeddings()

    def visual_embed(self, frames):
        return self.model.visual_embed(frames)

    def __call__(self, **kw):
        out = self.model(**kw)
        tok = self.schedule.get(self.calls)
        self.calls += 1
        if tok is not None:
            out.logits[:, -1, tok] += 1000.0
        return out


def golden_schedule(cfg):
    """call index -> forced id.  Frames: silent, silent, speak | response: 2 natural tokens then EOS |
    frame after EOS: silent, speak | response: EOS at once | silent ..."""
    I, E, END = cfg.frame_token_interval_id, cfg.eos_token_id, cfg.stream_end_id
    return {0: I, 1: I, 2: END, 5: E, 6: I, 7: END, 8: E, 9: I, 10: I, 11: I}


def query_schedule(cfg):
    """Second scripted run, WITH user queries (demo/cli.py:23-26): the narration request at t = 0.0 (rule 2 of
    _call_for_streaming: answered right after the frame of that time) and a mid-stream query stamped 1.75 s that
    arrives before the 2.0 s frame is consumed (rule 1: answered before the next frame).
    call index -> forced id: frame0 (decision unused: the query pre-empts it) | response: 2 natural tokens, EOS |
    frames .5, 1.0 silent, 1.5 speak | response: 1 natural, EOS | query response: 1 natural, EOS |
    frames 2.0, 2.5 silent | 3.0 speak | response EOS | 3.5 silent."""
    I, E, END = cfg.frame_token_interval_id, cfg.eos_token_id, cfg.stream_end_id
    return {0: I, 3: E, 4: I, 5: I, 6: END, 8: E, 10: E, 11: I, 12: I, 13: END, 14: E, 15: I}


QUERY_0 = 'Please narrate the video in real time.'      # demo/cli.py:23
QUERY_MID = 'What is happening now?'
QUERY_MID_AT, QUERY_MID_BEFORE_ITER = 1.75, 4           # stamped 1.75 s, submitted before iteration 4 (t = 2.0 s)


class _HostIds(torch.Tensor):
    """ids tensor whose .to('cuda') is a no-op, so the reference's query branch (demo/inference.py:42) runs
    unmodified on a CPU host."""

    def to(self, *a, **k):
        return self


class _CpuTok:
    def __init__(self, tok):
        self._tok = tok

    def apply_chat_template(self, *a, **k):
        return self._tok.apply_chat_template(*a, **k).as_subclass(_HostIds)

    def decode(self, *a, **k):
        return self._tok.decode(*a, **k)


def run_reference_liveinfer(ref_inf, model, cfg, tok, schedule, video, queries_at_iter, n_iters=8):
    """The reference's LiveInfer methods, unmodified, on CPU with scripted decisions.  queries_at_iter:
    {iteration: [(query, video_time)]} submitted through input_query_stream before that iteration."""
    import collections
    li = ref_inf.LiveInfer.__new__(ref_inf.LiveInfer)
    li.model, li.tokenizer = ScriptedModel(model, schedule), _CpuTok(tok)
    li.hidden_size, li.frame_fps, li.frame_num_tokens = cfg.hidden_size, 2, cfg.frame_num_tokens
    li.frame_token_interval_id, li.frame_token_interval_threshold = cfg.frame_token_interval_id, 0.725
    li.eos_token_id = cfg.eos_token_id
    li.inplace_output_ids = torch.zeros(1, 100, dtype=torch.long)
    li._start_ids = tok.apply_chat_template([{'role': 'system', 'content': SYSTEM_PROMPT}], add_stream_prompt=True, return_tensors='pt')
    li._added_stream_prompt_ids = tok.apply_chat_template([{}], add_stream_prompt=True, return_tensors='pt')
    li._added_stream_generation_ids = tok.apply_chat_template([{}], add_stream_generation_prompt=True, return_tensors='pt')
    li.query_queue, li.frame_embeds_queue = collections.deque(), collections.deque()
    li.video_time, li.last_frame_idx = 0, -1
    li.last_ids, li.past_key_values = torch.tensor([[]], dtype=torch.long), None
    li.video_tensor = video
    trace, notes = [], []
    for i in range(n_iters):
        for q, vt in queries_at_iter.get(i, []):
            notes.append(li.input_query_stream(q, video_time=vt))
        li.input_video_stream(i / li.frame_fps)
        query, response = li()
        kv = li.past_key_values.get_seq_length()
        trace.append((i, query, response, int(li.last_ids.reshape(-1)[-1]), kv))
    return trace, li.model.calls, notes


def stream_eval_sample(cfg, tok):
    """A two-turn conversation for stream_evaluate (models/modeling_live.py:44-168): system prompt, 3 frames, an
    assistant reply, 2 frames, an assistant reply.  Labels follow data/stream.py's convention: the LAST <v> of a frame
    predicts "," (keep watching) or "]\n" (speak); assistant text is teacher-forced; everything else is ignored."""
    msgs = [{'role': 'system', 'content': 'sys'}, {'role': 'stream', 'num_frames': 3}, {'role': 'assistant', 'content': 'ab'},
            {'role': 'stream', 'num_frames': 2}, {'role': 'assistant', 'content': 'c'}]
    ids = tok.apply_chat_template(msgs, return_tensors='pt')
    input_id = ids[0]
    label = torch.full_like(input_id, -100)
    n, fnt, v_id = input_id.numel(), cfg.frame_num_tokens, cfg.v_placeholder_id
    i = 0
    while i < n:
        if input_id[i] == v_id and (i + 1 == n or input_id[i + 1] != v_id):       # last <v> of a frame
            label[i] = input_id[i + 1]
        i += 1
    # assistant spans: tokens after "Assistant:" up to and including EOS are learned (shifted by one)
    txt_colon = tok.encode(':')[0]
    eos = cfg.eos_token_id
    for e in (input_id == eos).nonzero()[:, 0].tolist():
        st = e
        while input_id[st] != txt_colon:
            st -= 1
        for j in range(st, e):
            label[j] = input_id[j + 1]
    return ids, label[None]


def craft_silent_lm_head(llm_state, cfg, hidden, positions):
    """Random weights never predict the interval token, so stream_evaluate's "reply after the turn" branch (:110-141)
    would stay dark.  Give the interval id an lm_head row aligned with the final hidden states at `positions`
    (|h_p|^2 dominates the cross terms), which makes exactly those frames read as "keep watching"."""
    row = hidden[positions].float().sum(0)
    row = row / row.norm() * 40.0
    sd = dict(llm_state)
    w = sd["lm_head.weight"].clone()
    w[cfg.frame_token_interval_id] = row.to(w.dtype)
    sd["lm_head.weight"] = w
    return sd, w[cfg.frame_token_interval_id].clone()


@torch.no_grad()
def main():
    torch.manual_seed(0)
    cfg = tiny_config()
    llm_state = W.synthetic_llm_state(cfg, seed=0)
    # a larger lm_head scale gives healthy top-1/top-2 margins for the greedy-id checks
    llm_state["lm_head.weight"] = (llm_state["lm_head.weight"].float() * 8).to(torch.bfloat16)
    vision_state = W.synthetic_vision_state(cfg, seed=1)
    model, fast_greedy_generate, ref_inf = build_reference_model(cfg, llm_state, vision_state)
    g = torch.Generator().manual_seed(123)
    S = cfg.frame_resolution
    frames = torch.randint(0, 256, (4, 3, S, S), dtype=torch.uint8, generator=g)
    fx = {"frames": frames}

    # ---- vision: tokens before the connector and visual_embed after it
    fx["vit_tokens"] = model.vision_encode(model.vision_encoder, frames).float()
    fx["visual_embed"] = model.visual_embed(frames)

    # ---- decoder: chunked KV-append forward (17, 11, 11, 1, 1 tokens), all-position logits per chunk
    from transformers import DynamicCache
    embeds_all = torch.randn(41, cfg.hidden_size, generator=g).to(torch.bfloat16)
    fx["step_embeds"] = embeds_all
    chunks, cache, logits, off = [17, 11, 11, 1, 1], None, [], 0
    for c in chunks:
        out = model(inputs_embeds=embeds_all[None, off:off + c], use_cache=True, past_key_values=cache)
        cache = out.past_key_values
        logits.append(out.logits[0].clone())
        off += c
    fx["step_chunks"] = torch.tensor(chunks)
    fx["step_logits"] = torch.cat(logits, 0)
    fx["kv_k0"], fx["kv_v0"] = cache.layers[0].keys[0].clone(), cache.layers[0].values[0].clone()
    L = cfg.num_hidden_layers - 1
    fx["kv_kL"], fx["kv_vL"] = cache.layers[L].keys[0].clone(), cache.layers[L].values[0].clone()
    one = model(inputs_embeds=embeds_all[None], use_cache=True, past_key_values=None)
    fx["step_logits_onepass"] = one.logits[0].clone()

    # ---- greedy generation after a 14-token prompt
    prompt = torch.randn(1, 14, cfg.hidden_size, generator=g).to(torch.bfloat16)
    fx["gen_prompt"] = prompt[0]
    buf = torch.zeros(1, 12, dtype=torch.long)
    ids, _ = fast_greedy_generate(model=model, inputs_embeds=prompt, past_key_values=None, eos_token_id=cfg.eos_token_id,
                                  inplace_output_ids=buf)
    fx["gen_ids"] = ids[0].clone()

    # ---- state machine: the reference's LiveInfer methods, unmodified, on CPU with scripted decisions
    tok = ByteTokenizer(cfg)
    video = torch.randint(0, 256, (8, 3, S, S), dtype=torch.uint8, generator=g)
    fx["sm_video"] = video
    fx["sm_trace"], fx["sm_calls"], _ = run_reference_liveinfer(ref_inf, model, cfg, tok, golden_schedule(cfg), video, {})
    # ---- same, with user queries (demo/cli.py:23 + a mid-stream query): rules 1 and 2 of _call_for_streaming and the
    #      query branch of _call_for_response
    fx["smq_trace"], fx["smq_calls"], fx["smq_notes"] = run_reference_liveinfer(
        ref_inf, model, cfg, tok, query_schedule(cfg), video,
        {0: [(QUERY_0, 0.0)], QUERY_MID_BEFORE_ITER: [(QUERY_MID, QUERY_MID_AT)]})

    # ---- joint_embed (models/modeling_live.py:29-42): ids with <v> placeholders + frames
    v_id = cfg.v_placeholder_id
    jids = torch.tensor([[5, 7] + [v_id] * cfg.frame_num_tokens + [cfg.frame_token_interval_id] + [v_id] * cfg.frame_num_tokens + [9]])
    fx["joint_ids"] = jids
    fx["joint_embed"] = model.joint_embed(jids, frames[:2]).clone()
    fx["joint_logits"] = model(input_ids=jids, frames=frames[:2], use_cache=False).logits[0].clone()

    # ---- stream_evaluate (models/modeling_live.py:44-168): the reference's own method on a two-turn sample.
    #      trim_past_key_values (:170-171) assumes the legacy tuple cache and breaks on transformers 5.5's DynamicCache
    #      (SURVEY 8c); it is replaced by its meaning: a copy of the cache cropped to the first `stop` positions.
    import copy
    sys.path.insert(0, str(ROOT / "oracle"))
    import vlo_oracle as O
    se_ids, se_labels = stream_eval_sample(cfg, tok)
    se_frames = torch.randint(0, 256, (5, 3, S, S), dtype=torch.uint8, generator=g)
    hid = O.llama_forward(llm_state, cfg, O.joint_embed(llm_state, vision_state, cfg, se_ids[0], se_frames),
                          O.KVCache(cfg.num_hidden_layers), return_hidden=True)
    v_last = [i for i in range(se_ids.shape[1]) if se_labels[0, i] != -100 and se_ids[0, i] == cfg.v_placeholder_id]
    se_state, se_row = craft_silent_lm_head(llm_state, cfg, hid, v_last[:3])      # the three frames of turn 1 stay silent
    model.lm_head.weight.data[cfg.frame_token_interval_id] = se_row
    type(model).trim_past_key_values = lambda self, pkv, start, stop: (lambda c: (c.crop(stop), c)[1])(copy.deepcopy(pkv))
    fx["se_ids"], fx["se_labels"], fx["se_frames"], fx["se_lm_head_row"] = se_ids, se_labels, se_frames, se_row
    for thr in (0.0, 0.9):
        fx[f"se_metrics_thr{thr}"] = model.stream_evaluate(se_ids, se_labels, se_frames, frame_token_interval_threshold=thr).clone()
    model.lm_head.weight.data[cfg.frame_token_interval_id] = llm_state["lm_head.weight"][cfg.frame_token_interval_id]

    torch.save(fx, OUT / "tiny_reference.pt")
    for k, v in fx.items():
        print(k, tuple(v.shape) if isinstance(v, torch.Tensor) else v)


def digest(t: torch.Tensor) -> str:
    """SHA-256 of a tensor's dtype, shape and raw bytes: equal digests <=> bit-identical tensors."""
    h = hashlib.sha256(f"{t.dtype} {tuple(t.shape)}".encode())
    h.update(t.detach().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def bf16_gemm_fingerprint(cfg) -> str:
    """Digest of plain bf16 CPU GEMMs at the tiny decoder's projection shapes.  torch picks its bf16 GEMM kernel by
    ISA (AMX / avx512_bf16 / AVX-512 accumulate in different orders), so two hosts with the same fingerprint compute
    the same bf16 forward bit for bit, and hosts with different ones may differ by an ulp."""
    g = torch.Generator().manual_seed(0)
    h = hashlib.sha256()
    q = cfg.num_attention_heads * cfg.head_dim
    for m in (1, 11, 17):
        for k, n in ((cfg.hidden_size, q), (cfg.hidden_size, cfg.intermediate_size), (cfg.intermediate_size, cfg.hidden_size),
                     (cfg.hidden_size, cfg.vocab_size)):
            x = torch.randn(m, k, generator=g).to(torch.bfloat16)
            w = torch.randn(n, k, generator=g).to(torch.bfloat16)
            h.update(torch.nn.functional.linear(x, w).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


@torch.no_grad()
def forward_digests():
    """reference_forward.json: digests of the reference's forward on the inputs of tiny_reference.pt (per-chunk logits
    of the KV-append forward, last-layer K / V, logits of forward(input_ids, frames)) and the GEMM fingerprint of the
    host that ran it.  Stored as digests because the claim they carry is bit-identity on such a host."""
    cfg = tiny_config()
    llm_state = W.synthetic_llm_state(cfg, seed=0)
    llm_state["lm_head.weight"] = (llm_state["lm_head.weight"].float() * 8).to(torch.bfloat16)
    model, _, _ = build_reference_model(cfg, llm_state, W.synthetic_vision_state(cfg, seed=1))
    fx = torch.load(OUT / "tiny_reference.pt", weights_only=False)
    rec, cache, off = {"bf16_gemm_fingerprint": bf16_gemm_fingerprint(cfg), "chunk_logits": []}, None, 0
    for c in fx["step_chunks"].tolist():
        out = model(inputs_embeds=fx["step_embeds"][None, off:off + c], use_cache=True, past_key_values=cache)
        cache = out.past_key_values
        rec["chunk_logits"].append(digest(out.logits[0]))
        off += c
    L = cfg.num_hidden_layers - 1
    rec["kv_kL"], rec["kv_vL"] = digest(cache.layers[L].keys[0]), digest(cache.layers[L].values[0])
    rec["joint_logits"] = digest(model(input_ids=fx["joint_ids"], frames=fx["frames"][:2], use_cache=False).logits[0])
    (OUT / "reference_forward.json").write_text(json.dumps(rec, indent=1) + "\n")
    print(json.dumps(rec, indent=1))


def demo_clip_excerpts():
    """The first second of the two clips the reference's demo plays (demo/assets/cooking.mp4 1440x1080, bicycle.mp4
    512x384, 30 fps), as the 2 FPS ingest sees it: source frames 0 and 15, each held for 15 frames, 30 fps, MPEG-4
    part 2 (the encoder OpenCV ships).  cooking is scaled to 480x360 (same 4:3 letterbox) to keep the file small."""
    import cv2
    for name, size in (("bicycle", None), ("cooking", (480, 360))):
        cap = cv2.VideoCapture(os.path.join(REF, "demo", "assets", name + ".mp4"))
        src = [cap.read()[1] for _ in range(30)]
        cap.release()
        if size is not None:
            src = [cv2.resize(f, size, interpolation=cv2.INTER_AREA) for f in src]
        h, w = src[0].shape[:2]
        path = OUT / f"demo_{name}_excerpt.mp4"
        wr = cv2.VideoWriter(str(path), cv2.CAP_FFMPEG, cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (w, h),
                             [cv2.VIDEOWRITER_PROP_KEY_INTERVAL, 1000])
        for i in range(30):
            wr.write(src[i - i % 15])
        wr.release()
        print(path, w, h, path.stat().st_size)


if __name__ == "__main__":
    # no argument: tiny_reference.pt; `forward`: reference_forward.json; `clips`: the demo clip excerpts
    {"forward": forward_digests, "clips": demo_clip_excerpts}.get(sys.argv[1] if len(sys.argv) > 1 else None, main)()
