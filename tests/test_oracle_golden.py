"""Pin oracle/vlo_oracle.py against outputs of the reference's own modules (tests/golden/make_golden.py)."""
import sys
import pathlib

import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "oracle"))
import vlo_oracle as O  # noqa: E402
import pytest  # noqa: E402


def _assert_bf16_pinned(got, ref, what):
    """Bit-exact on the machine that generated the fixture.  torch's CPU bf16 GEMMs pick ISA-specific kernels (AMX /
    avx512_bf16 / plain AVX-512 accumulate in different orders), so on a DIFFERENT host the same reference code moves
    single logits by one bf16 ulp: there the committed fixture is held to <= 2 ulp (of max(|x|, 4): the logit scale) per element, and the bit-exact claim
    is re-proved against digests of the reference's outputs recorded on a host of the same kind (test_*_bit_exact_vs_live_reference)."""
    if torch.equal(got, ref):
        return
    a, b = got.float(), ref.float()
    ulp = torch.exp2(torch.floor(torch.log2(b.abs().clamp_min(4.0))) - 7)
    worst = ((a - b).abs() / ulp).max().item()
    frac = (got != ref).float().mean().item()
    assert worst <= 2.0 and frac < 0.35, f"{what}: {worst:.1f} ulp, {frac:.3f} of the elements differ"


def test_vision_tokens_match_reference(golden, tiny):
    cfg, llm, vis = tiny
    tok = O.siglip_vision_encode(vis, cfg, golden["frames"])
    assert tok.shape == golden["vit_tokens"].shape
    torch.testing.assert_close(tok, golden["vit_tokens"], rtol=1e-4, atol=1e-5)


def test_visual_embed_matches_reference(golden, tiny):
    cfg, llm, vis = tiny
    out = O.visual_embed(llm, vis, cfg, golden["frames"])
    ref = golden["visual_embed"]
    assert out.dtype == torch.bfloat16 and out.shape == ref.shape
    # bf16 connector on fp32 tokens that agree to 1e-5: allow a couple of bf16 ulps
    torch.testing.assert_close(out.float(), ref.float(), rtol=2e-2, atol=2e-2)
    assert (out == ref).float().mean() > 0.98


def test_chunked_kv_append_forward_is_bit_exact(golden, tiny):
    cfg, llm, vis = tiny
    cache = O.KVCache(cfg.num_hidden_layers)
    logits, off = [], 0
    for c in golden["step_chunks"].tolist():
        logits.append(O.llama_forward(llm, cfg, golden["step_embeds"][off:off + c], cache))
        off += c
    logits = torch.cat(logits, 0)
    _assert_bf16_pinned(logits, golden["step_logits"], "chunked logits")
    assert torch.equal(cache.k[0][0], golden["kv_k0"]) and torch.equal(cache.v[0][0], golden["kv_v0"])
    L = cfg.num_hidden_layers - 1
    _assert_bf16_pinned(cache.k[L][0], golden["kv_kL"], "last-layer K")
    _assert_bf16_pinned(cache.v[L][0], golden["kv_vL"], "last-layer V")


@torch.no_grad()
def test_chunked_kv_append_bit_exact_vs_live_reference(golden, tiny):
    """Same inputs through LiveLlamaForCausalLM.forward (the reference, run by `make_golden.py forward`, which recorded
    digests of its outputs and the bf16 GEMM fingerprint of its host) and the oracle: bit-identical logits and cache
    contents on a host with the same fingerprint.  A host with another one is held to the cross-host bound of
    _assert_bf16_pinned against the committed reference values."""
    import json
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden as MG
    cfg, llm, vis = tiny
    rec = json.loads((ROOT / "tests" / "golden" / "reference_forward.json").read_text())
    cache, off, chunks = O.KVCache(cfg.num_hidden_layers), 0, []
    for c in golden["step_chunks"].tolist():
        chunks.append(O.llama_forward(llm, cfg, golden["step_embeds"][off:off + c], cache))
        off += c
    L = cfg.num_hidden_layers - 1
    emb = O.joint_embed(llm, vis, cfg, golden["joint_ids"][0], golden["frames"][:2])
    joint = O.llama_forward(llm, cfg, emb, O.KVCache(cfg.num_hidden_layers))
    if MG.bf16_gemm_fingerprint(cfg) == rec["bf16_gemm_fingerprint"]:
        assert [MG.digest(x) for x in chunks] == rec["chunk_logits"]
        assert MG.digest(cache.k[L][0]) == rec["kv_kL"] and MG.digest(cache.v[L][0]) == rec["kv_vL"]
        assert MG.digest(joint) == rec["joint_logits"]
    else:
        _assert_bf16_pinned(torch.cat(chunks, 0), golden["step_logits"], "chunked logits")
        _assert_bf16_pinned(cache.k[L][0], golden["kv_kL"], "last-layer K")
        _assert_bf16_pinned(cache.v[L][0], golden["kv_vL"], "last-layer V")
        _assert_bf16_pinned(joint, golden["joint_logits"], "joint logits")


def test_chunked_equals_one_pass(golden):
    # SURVEY.md Appendix C.1: streaming in chunks == one causal pass (bf16: equal up to rounding)
    a, b = golden["step_logits"].float(), golden["step_logits_onepass"].float()
    assert (a - b).abs().max() < 0.5 and (a.argmax(-1) == b.argmax(-1)).float().mean() > 0.9


def test_greedy_ids_bit_exact(golden, tiny):
    cfg, llm, vis = tiny
    ids = O.fast_greedy_generate(llm, cfg, golden["gen_prompt"], O.KVCache(cfg.num_hidden_layers), cfg.eos_token_id, max_new=12)
    assert ids == golden["gen_ids"].tolist()


def test_state_machine_matches_reference_liveinfer(golden, tiny):
    cfg, llm, vis = tiny
    from videollm_online_b200.config import SYSTEM_PROMPT
    from videollm_online_b200.tokenization_live import ByteTokenizer
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    from make_golden import golden_schedule
    sched, calls = golden_schedule(cfg), [0]

    def hook(logits, kind):
        tok = sched.get(calls[0])
        calls[0] += 1
        if tok is not None:
            logits = logits.clone()
            logits[tok] += 1000.0
        return logits

    li = O.OracleLiveInfer(llm, vis, cfg, ByteTokenizer(cfg), frame_fps=2, system_prompt=SYSTEM_PROMPT, logit_hook=hook)
    li.load_video(golden["sm_video"])
    trace = []
    for i in range(8):
        li.input_video_stream(i / 2)
        query, response = li()
        trace.append((i, query, response, int(li.last_ids.reshape(-1)[-1]), li.cache.get_seq_length()))
    assert trace == golden["sm_trace"]
    assert calls[0] == golden["sm_calls"]


def test_decide_rule():
    # demo/inference.py:76-79: below-threshold interval probability is zeroed before the argmax
    x = torch.full((16,), -10.0, dtype=torch.bfloat16)
    x[3], x[5] = 2.0, 1.5          # p(3) ~ 0.62 < 0.725 -> second best wins when 3 is the interval id
    assert O.decide(x.clone(), 3, 0.725) == 5
    assert O.decide(x.clone(), 3, 0.5) == 3
    assert O.decide(x.clone(), 7, 0.725) == 3


def _oracle_liveinfer(tiny, schedule):
    cfg, llm, vis = tiny
    from videollm_online_b200.config import SYSTEM_PROMPT
    from videollm_online_b200.tokenization_live import ByteTokenizer
    calls = [0]

    def hook(logits, kind):
        tok = schedule.get(calls[0])
        calls[0] += 1
        if tok is not None:
            logits = logits.clone()
            logits[tok] += 1000.0
        return logits

    return O.OracleLiveInfer(llm, vis, cfg, ByteTokenizer(cfg), frame_fps=2, system_prompt=SYSTEM_PROMPT, logit_hook=hook), calls


def test_state_machine_with_queries_matches_reference_liveinfer(golden, tiny):
    """The query path (demo/cli.py:23 narration request at t=0 + a mid-stream query): rules 1 and 2 of
    _call_for_streaming (demo/inference.py:57-59, 72-74) and the user-query branch of _call_for_response (:42),
    against the trace of the reference's own methods."""
    cfg, llm, vis = tiny
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden as MG
    li, calls = _oracle_liveinfer(tiny, MG.query_schedule(cfg))
    li.load_video(golden["sm_video"])
    trace = []
    for i in range(8):
        if i == 0:
            li.input_query_stream(MG.QUERY_0, video_time=0.0)
        if i == MG.QUERY_MID_BEFORE_ITER:
            li.input_query_stream(MG.QUERY_MID, video_time=MG.QUERY_MID_AT)
        li.input_video_stream(i / 2)
        query, response = li()
        trace.append((i, query, response, int(li.last_ids.reshape(-1)[-1]), li.cache.get_seq_length()))
    assert trace == golden["smq_trace"]
    assert calls[0] == golden["smq_calls"]


def test_joint_embed_matches_reference(golden, tiny):
    """models/modeling_live.py:29-42 and forward(input_ids, frames) (models/live_llama/modeling_live_llama.py:24-67)."""
    cfg, llm, vis = tiny
    ids = golden["joint_ids"]
    emb = O.joint_embed(llm, vis, cfg, ids[0], golden["frames"][:2])
    ref = golden["joint_embed"][0]
    assert emb.shape == ref.shape and emb.dtype == ref.dtype
    is_v = ids[0] == cfg.v_placeholder_id
    assert torch.equal(emb[~is_v], ref[~is_v])                       # token rows: exact gather
    torch.testing.assert_close(emb[is_v].float(), ref[is_v].float(), rtol=2e-2, atol=2e-2)   # as test_visual_embed_matches_reference
    logits = O.llama_forward(llm, cfg, ref, O.KVCache(cfg.num_hidden_layers))
    _assert_bf16_pinned(logits, golden["joint_logits"], "joint logits")


def _se_state(golden, tiny):
    cfg, llm, vis = tiny
    sd = dict(llm)
    w = sd["lm_head.weight"].clone()
    w[cfg.frame_token_interval_id] = golden["se_lm_head_row"]     # see make_golden.craft_silent_lm_head
    sd["lm_head.weight"] = w
    return cfg, sd, vis


def test_stream_evaluate_matches_reference(golden, tiny):
    """models/modeling_live.py:44-168 on a two-turn sample: turn 1 takes the look-ahead branch (:110-141, trimmed
    cache + appended frames), turn 2 the in-turn branch (:105-107).  Same four metrics as the reference's own method."""
    cfg, sd, vis = _se_state(golden, tiny)
    for thr in (0.0, 0.9):
        got = O.stream_evaluate(sd, vis, cfg, golden["se_ids"], golden["se_labels"], golden["se_frames"],
                                frame_token_interval_threshold=thr)
        ref = golden[f"se_metrics_thr{thr}"]
        torch.testing.assert_close(got[1:], ref[1:].float(), rtol=0, atol=0)
        torch.testing.assert_close(got[0].log(), ref[0].float().log(), rtol=1e-5, atol=1e-5)
