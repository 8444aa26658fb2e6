"""CPU tests (no GPU): host logic added in round 2 -- LoRA merge on load, the oracles against the golden vectors of the
unmodified reference (tests/golden/lm_round2.npz, oracle/gen_golden_lm.py), the ABI exactly as INTEGRATION.md binds it,
shard/scheduler host logic."""
import ctypes
import dataclasses
import os
import re

import numpy as np
import pytest
import torch

from oracle import infer_oracle as IO
from oracle import lm_oracle as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "lm_round2.npz"))


def test_lora_factors_are_merged_on_load_like_merge_lora_weights(gold):
    """A checkpoint with lora_A / lora_B (llama_streaming.py:95-97, 203-215) loads into the product GPT as the merged
    weights the reference's merge_lora_weights (:1120-1124) produces -- GQA layout, key LoRA disabled (zero_pad)."""
    from rstnet_b200.lm import GPT, Config
    cfg = dataclasses.replace(L.SMALL, n_query_groups=2)
    w = L.synthetic_weights(cfg, seed=27, dtype=torch.float32, std=0.05)
    lw = L.synthetic_lora(cfg, seed=28, r=4, enable=(True, False, True))
    m = GPT(Config(block_size=cfg.block_size, n_layer=cfg.n_layer, n_embd=cfg.n_embd, n_head=cfg.n_head, head_size=cfg.head_size,
                   n_query_groups=2, intermediate_size=cfg.intermediate_size, padded_vocab_size=cfg.padded_vocab_size,
                   audio_card=cfg.audio_card, n_q=cfg.n_q, dep_q=cfg.dep_q, codecformer_dim=cfg.codecformer_dim,
                   codecformer_heads=cfg.codecformer_heads, codecformer_layers=cfg.codecformer_layers,
                   codecformer_dim_feedforward=cfg.codecformer_dim_feedforward, context=cfg.context,
                   lora_r=4, lora_alpha=8, lora_query=True, lora_key=False, lora_value=True, lora_projection=True, lora_mlp=True,
                   lora_head=True))
    m.load_state_dict({**w, **lw}, strict=True)
    sd = m.state_dict()
    assert not any("lora_" in k for k in sd)
    for i, name in enumerate(gold["lora_names"]):
        # the reference's merged weight = base + its stored rank-r update (reconstructed to 1e-7)
        ref = w[str(name)] + torch.from_numpy(gold[f"lora_update_{i}_u"]) @ torch.from_numpy(gold[f"lora_update_{i}_v"])
        assert not torch.equal(sd[str(name)], w[str(name)])
        assert (sd[str(name)] - ref).abs().max().item() <= 2e-6, name
    assert (sd["lm_head.linear.weight"][:64] - torch.from_numpy(gold["lora_head_rows"])).abs().max().item() <= 2e-6
    # the key rows of the QKV weight stay untouched (lora_key False -> zero padding, llama_streaming.py:255-328)
    hs, group = cfg.head_size, cfg.n_head // 2 + 2
    rows = torch.arange(sd["transformer.h.0.attn.attn.linear.weight"].shape[0])
    krows = ((rows // hs) % group) == group - 2
    assert torch.equal(sd["transformer.h.0.attn.attn.linear.weight"][krows], w["transformer.h.0.attn.attn.linear.weight"][krows])


def test_inference_imp_oracle_reproduces_reference_tokens(gold):
    """oracle/infer_oracle.py against the tokens of the UNMODIFIED InferenceImp (fp32, both deterministic modes)."""
    cfg = L.SMALL
    w = L.synthetic_weights(cfg, seed=7, dtype=torch.float32, std=0.05)
    seq = torch.from_numpy(gold["infer_seq"])
    for mode, use_sampling in (("greedy", False), ("top1", True)):
        with torch.no_grad():
            r = IO.inference_imp_tts(w, cfg, seq.clone(), use_sampling)
        ref = torch.from_numpy(gold[f"infer_f32_{mode}_codes"])
        frames = torch.from_numpy(gold[f"infer_f32_{mode}_frames"])
        # fp32 near-ties (margin < 1e-3) may flip across BLAS builds; everything before the first one must match
        m = torch.from_numpy(gold[f"infer_f32_{mode}_margins"]).flatten()
        first = int((m < 1e-3).nonzero()[0]) if bool((m < 1e-3).any()) else m.numel()
        assert torch.equal(r["frames"].flatten()[:first], frames.flatten()[:first])
        if first == m.numel():
            assert torch.equal(r["codes"], ref)
    x = torch.arange(8 * 6).view(8, 6)
    rd = IO.reverse_delay(x)
    assert rd.shape == (8, 5) and torch.equal(rd[0], x[0, :-1]) and torch.equal(rd[1:], x[1:, 1:])
    assert torch.equal(IO.reverse_delay(x.t()), rd)
    from rstnet_b200.infer import reverse_delay
    assert torch.equal(reverse_delay(x), rd) and torch.equal(reverse_delay(x.t()), rd)


def test_gqa_partial_rope_oracle_reproduces_reference(gold):
    """GQA + rotary_percentage 0.5 + rope_adjustments: the streaming oracle against the reference's fp32 tokens, and the
    non-streaming forward_global_full / forward_local against its outputs."""
    cfg = dataclasses.replace(L.SMALL, n_query_groups=2, rotary_percentage=0.5,
                              rope_adjustments={"factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                                                "original_max_seq_len": 32})
    w = L.synthetic_weights(cfg, seed=17, dtype=torch.float32, std=0.05)
    seqs = torch.from_numpy(gold["gqa_seqs"])
    gs = L.GPTStream(w, cfg, 3)
    agree = total = 0
    with torch.no_grad():
        for f in range(6):
            o = L.greedy_frame(gs, seqs[f])
            ref = torch.from_numpy(gold["gqa_f32_tokens"][f])
            agree += int((o[3] == ref).sum()); total += ref.numel()
            if not torch.equal(o[3], ref):
                break                                           # greedy loop: a near-tie flip changes what follows
        T = gold["gqa_f32_full_out"].shape[1]
        full = torch.cat([seqs[f] for f in range(T)], dim=2)
        out, tl = L.forward_global_full(w, cfg, full)
        assert (out - torch.from_numpy(gold["gqa_f32_full_out"])).abs().max().item() <= 1e-4
        toks = torch.from_numpy(gold["gqa_f32_local_tokens"])
        loc = L.forward_local(w, cfg, L.scaled_embedding(toks[:, 0, :], w["codecformer_text_emb.weight"]), toks[:, 1:, :],
                              torch.from_numpy(gold["gqa_f32_full_out"]))
        cols = torch.from_numpy(gold["gqa_local_logits_cols"])      # fixed sample of the vocabulary
        assert (loc[..., cols] - torch.from_numpy(gold["gqa_f32_local_logits_sampled"])).abs().max().item() <= 1e-4
    assert agree >= 0.95 * total


def _parse_header_struct(name):
    hdr = open(os.path.join(ROOT, "include", "rstnet_b200.h")).read()
    end = hdr.index("} " + name + ";")
    body = hdr[hdr.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        typ = "ptr" if "*" in decl else ("i64" if "int64_t" in decl else "i32")
        names = [n.strip().lstrip("*") for n in re.sub(r"^(const\s+)?\w+\s*\**", "", decl, count=1).split(",")]
        fields += [(n, typ) for n in names]
    return fields


def test_integration_md_binding_matches_the_header():
    """The ctypes stub INTEGRATION.md shows must describe the struct the library reads: same fields, order and size as
    include/rstnet_b200.h (round 1's stub stopped before `taps` / `tap_stride`)."""
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    code = re.search(r"class GemmRowsArgs\(ctypes\.Structure\):.*?\n(?=\ndef )", doc, re.S).group(0)
    ns = {"ctypes": ctypes}
    exec(code, ns)
    doc_struct = ns["GemmRowsArgs"]
    from rstnet_b200._lib import GemmRowsArgs
    hdr = _parse_header_struct("rstnet_gemm_rows_args")
    kind = {ctypes.c_void_p: "ptr", ctypes.c_int64: "i64", ctypes.c_int32: "i32"}
    for struct in (doc_struct, GemmRowsArgs):
        got = [(n, kind[t]) for n, t in struct._fields_]
        assert got == hdr, (struct, got, hdr)
    assert ctypes.sizeof(doc_struct) == ctypes.sizeof(GemmRowsArgs)
    from rstnet_b200._lib import TcGemmDesc
    got = [(n, kind[t]) for n, t in TcGemmDesc._fields_]
    assert got == _parse_header_struct("rstnet_tc_gemm_desc")


def test_frame_scheduler_host_logic():
    """Admission / release bookkeeping of the batched frame scheduler (no GPU: a stub engine)."""
    from rstnet_b200.serve import FrameScheduler

    class Stub:
        def __init__(self):
            self.resets, self.steps = [], 0

        def reset_rows(self, rows):
            self.resets.append(list(rows))

        def step(self, pcm_rows, active):
            self.steps += 1
            return {r: (f"tok{r}", f"pcm{r}") for r in active}

    eng = Stub()
    s = FrameScheduler(eng, capacity=3)
    a, b = s.admit("A"), s.admit("B")
    assert (a, b) == (0, 1) and eng.resets == [[0], [1]]
    s.push("A", "a0"); s.push("B", "b0")
    out = s.tick()
    assert set(out) == {"A", "B"} and out["A"] == ("tok0", "pcm0")
    s.push("A", "a1")                                   # B has no audio this tick: it is not stepped (stays aligned)
    out = s.tick()
    assert set(out) == {"A"}
    s.release("A")
    c, d = s.admit("C"), s.admit("D")
    assert c == 0 and d == 2 and eng.resets[-2:] == [[0], [2]]
    with pytest.raises(RuntimeError):
        s.admit("E")                                    # full
    assert s.free_rows() == 0 and s.sessions() == {"B": 1, "C": 0, "D": 2}


def test_moshi_oracle_reproduces_reference_lmgen(golden_dir):
    """oracle/moshi_oracle.py (LMModel.forward_text / depformer_step / LMGen.step, models/model.py:364-597) against the
    unmodified reference's fp32 tokens (tests/golden/moshi_small.npz)."""
    from oracle import moshi_oracle as M
    gold = np.load(os.path.join(golden_dir, "moshi_small.npz"))
    cfg = M.SMALL
    w = M.synthetic_weights(cfg, seed=5)
    inputs = torch.from_numpy(gold["inputs"])
    ref = torch.from_numpy(gold["f32_out"])
    ora = M.LMGenOracle(w, cfg, inputs.shape[1])
    outs = []
    with torch.no_grad():
        for t in range(8):
            o = ora.step(inputs[t])
            assert (o is None) == (t < max(cfg.delays))
            if o is not None:
                outs.append(o)
    mine = torch.stack(outs)
    agree = float((mine == ref[:len(outs)]).float().mean())
    assert agree >= 0.9, agree        # bit-equal on the generating machine; a BLAS with another summation order may flip near-ties
    # product class: same state_dict keys as the reference module
    from rstnet_b200.moshi import LMModel
    m = LMModel(**cfg.reference_kwargs())
    assert set(m.state_dict().keys()) == set(w.keys())
    m.load_state_dict(w, strict=True)
    assert m.num_codebooks == 17 and m.initial_token_id == cfg.card and m.text_initial_token_id == cfg.text_card
    with pytest.raises(NotImplementedError):
        LMModel(**{**cfg.reference_kwargs(), "norm": "layer_norm"})
