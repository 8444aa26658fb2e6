"""Generate tests/golden/lm_small.npz and lm_round2.npz by running the UNMODIFIED reference GPT (streaming decode).

Run:  python -m oracle.gen_golden_lm <MLLM_v2 directory of the original RSTnet checkout>

The reference `models.llama_streaming.GPT` (small config, seeded synthetic weights from
oracle/lm_oracle.synthetic_weights) is stepped for a few frames under `with gpt.streaming(B)` with
greedy sampling, in fp32 and in bf16; the oracle restatement must reproduce it bit for bit, and the
reference outputs are stored.

Every fixture stays under 1 MB, so the large tensors are stored in a smaller but equivalent form:
  *_sha256      SHA-256 of the float32 bytes, for tensors the tests compare bit for bit;
  *_bits        bf16 results as their raw 16-bit patterns (lossless);
  *_sampled     a fixed seeded sample of vocabulary columns (*_cols), for tensors compared within a tolerance;
  lora_update_* the reference's merged weight minus the seeded base weight, as rank-r factors u @ v (exact to 1e-7).
"""
from __future__ import annotations

import hashlib
import os
import sys

os.environ.setdefault("NO_TORCH_COMPILE", "1")
os.environ.setdefault("NO_CUDA_GRAPH", "1")
sys.dont_write_bytecode = True
REF = ""          # set by main() from the command line

import numpy as np
import torch

from . import lm_oracle as L
from .gen_golden import GOLDEN_THREADS, weights_digest

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
LOGIT_SAMPLE = 128     # vocabulary columns kept of a tolerance-compared logit tensor


def f32_sha256(t: torch.Tensor) -> str:
    """Digest of the float32 bytes (C order): equal digests <=> bit-equal tensors."""
    return hashlib.sha256(t.float().contiguous().numpy().tobytes()).hexdigest()


def bf16_bits(t: torch.Tensor) -> np.ndarray:
    """bf16 values as int16 bit patterns; torch.from_numpy(a).view(torch.bfloat16) restores them exactly."""
    return t.to(torch.bfloat16).contiguous().view(torch.int16).numpy()


def sample_cols(n: int) -> torch.Tensor:
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:LOGIT_SAMPLE].sort().values


def reference_frames(w, cfg, seqs, dtype):
    sys.path.insert(0, REF)
    from models.llama_streaming import GPT, Config
    m = GPT(Config(**cfg.reference_kwargs())).eval()
    sd = m.state_dict()
    assert set(sd.keys()) == set(w.keys()), set(sd.keys()) ^ set(w.keys())
    m.load_state_dict({k: v.float() for k, v in w.items()}, strict=True)
    m = m.to(dtype)
    B = seqs[0].shape[0]
    outs = []
    with torch.no_grad(), m.streaming(B):
        for seq in seqs:
            out, tl = m.forward_global(seq)
            tt = torch.argmax(tl.float(), dim=-1)
            toks, prev, al = [tt[:, 0]], tt[:, :, None], []
            with m.codecformer.streaming(B):
                for k in range(cfg.dep_q):
                    lg = m.forward_codecformer(k, prev, out)
                    al.append(lg[:, 0, 0])
                    prev = torch.argmax(lg.float(), dim=-1)
                    toks.append(prev[:, 0, 0])
            outs.append((out, tl, torch.stack(al, 1), torch.stack(toks, 1)))
    return outs


def load_reference_inference_imp():
    """The reference's InferenceImp / reverse_delay, UNMODIFIED: infer_no_streaming.py cannot be imported as a module here
    (it pulls omegaconf / torchaudio / HF downloads at import time), so only those two definitions are compiled, straight
    from the reference file, into a namespace holding the reference's own sampling functions."""
    import ast
    sys.path.insert(0, REF)
    from utils.sampling import sample_token, sample_token_audio, sample_token_audio_2048
    path = os.path.join(REF, "infer_no_streaming.py")
    tree = ast.parse(open(path).read())
    keep = [n for n in tree.body if isinstance(n, (ast.ClassDef, ast.FunctionDef)) and n.name in ("InferenceImp", "reverse_delay")]
    assert len(keep) == 2
    ns = {"torch": torch, "sample_token": sample_token, "sample_token_audio": sample_token_audio,
          "sample_token_audio_2048": sample_token_audio_2048}
    exec(compile(ast.Module(body=keep, type_ignores=[]), path, "exec"), ns)
    return ns["InferenceImp"], ns["reverse_delay"]


def reference_gpt(w, cfg, dtype, **extra):
    sys.path.insert(0, REF)
    from models.llama_streaming import GPT, Config
    m = GPT(Config(**cfg.reference_kwargs(), **extra)).eval()
    return m


def tts_sequence(P: int, G: int, seed: int) -> torch.Tensor:
    """A TTS-format [9, P+G] sequence: P prompt frames (text ids + audio), then G frames marked text-empty (to generate)."""
    g = torch.Generator().manual_seed(seed)
    seq = torch.randint(0, 2048, (9, P + G), generator=g)
    seq[0, :P] = torch.randint(0, 1000, (P,), generator=g)
    seq[0, P:] = 128002
    return seq


def gen_infer(save):
    """InferenceImp goldens (infer_no_streaming.py:169-308) in the two deterministic modes, fp32 and bf16."""
    from . import infer_oracle as IO
    RefImp, ref_reverse_delay = load_reference_inference_imp()
    cfg = L.SMALL
    P, G = 5, 8     # g_len > minlen from g_idx 4 on: both candidate-set rules fire
    seq = tts_sequence(P, G, seed=11)
    save["infer_seq"] = seq.numpy()
    x = torch.arange(8 * 5).view(8, 5)
    assert torch.equal(IO.reverse_delay(x), ref_reverse_delay(x))
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        w = L.synthetic_weights(cfg, seed=7, dtype=torch.float32, std=0.05)
        m = reference_gpt(w, cfg, dtype)
        m.load_state_dict({k: v.float() for k, v in w.items()}, strict=True)
        m = m.to(dtype)
        wd = {k: v.to(dtype) for k, v in w.items()}
        for mode, use_sampling, tk in (("greedy", False, 0), ("top1", True, 1)):
            imp = RefImp(None, m, "sampling", 0.7, tk, 0.8, tk, "TTS")
            imp.use_sampling = use_sampling        # instance attribute; the class hard-codes True (:162)
            with torch.no_grad():
                ref = imp(seq.clone(), torch.ones(9, P + G))
                mine = IO.inference_imp_tts(wd, cfg, seq.clone(), use_sampling)
            assert torch.equal(ref.cpu(), mine["codes"]), f"oracle InferenceImp != reference ({tag}, {mode})"
            save[f"infer_{tag}_{mode}_codes"] = ref.cpu().numpy()
            save[f"infer_{tag}_{mode}_frames"] = mine["frames"].numpy()
            save[f"infer_{tag}_{mode}_margins"] = mine["margins"].numpy()
            print(f"InferenceImp {tag} {mode}: oracle == reference, codes {tuple(ref.shape)}, min margin {float(mine['margins'].min()):.4f}")


def gen_variant(save):
    """GQA + partial rotary + Llama-3.1 rope adjustments (llama_streaming.py:952-982, lit_model.py:110-144, 441-488):
    streaming decode, the non-streaming forward_global over T frames (the prefill's yardstick) and forward_local."""
    import dataclasses
    cfg = dataclasses.replace(L.SMALL, n_query_groups=2, rotary_percentage=0.5,
                              rope_adjustments={"factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                                                "original_max_seq_len": 32})
    B, frames, T = 3, 20, 12
    g = torch.Generator().manual_seed(199)
    seqs = []
    for f in range(frames):
        s = torch.randint(0, 2048, (B, cfg.n_q + 1, 1), generator=g)
        s[:, 0] = torch.randint(0, 150000, (B, 1), generator=g)
        seqs.append(s)
    save["gqa_seqs"] = torch.stack(seqs).numpy()
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        w = L.synthetic_weights(cfg, seed=17, dtype=torch.float32, std=0.05)
        wd = {k: v.to(dtype) for k, v in w.items()}
        ref = reference_frames(w, cfg, seqs, dtype)
        gs = L.GPTStream(wd, cfg, B)
        with torch.no_grad():
            for f, seq in enumerate(seqs):
                o = L.greedy_frame(gs, seq)
                for a, b, name in zip(o, ref[f], ("out", "text_logits", "audio_logits", "tokens")):
                    assert torch.equal(a, b), f"oracle != reference (gqa): {tag} frame {f} {name}"
        print(f"gqa/partial-rope {tag}: oracle == reference on {frames} streaming frames")
        keep = (0, 1, 15, 16, 19)
        if tag == "bf16":     # the fp32 run's streaming outputs are checked through its tokens only
            save["gqa_bf16_out"] = torch.stack([ref[f][0].float() for f in keep]).numpy()
            save["gqa_bf16_audio_logits_bits"] = bf16_bits(torch.stack([ref[f][2] for f in keep]))
        save[f"gqa_{tag}_tokens"] = torch.stack([ref[f][3] for f in range(frames)]).numpy()
        save["gqa_keep"] = np.array(keep)
        # non-streaming forms on the first T frames (T < context: equal to T streaming steps up to rounding)
        m = reference_gpt(w, cfg, dtype)
        m.load_state_dict({k: v.float() for k, v in w.items()}, strict=True)
        m = m.to(dtype)
        full = torch.cat(seqs[:T], dim=2)
        with torch.no_grad():
            r_out, r_tl = m.forward_global(full)
            o_out, o_tl = L.forward_global_full(wd, cfg, full)
            assert torch.equal(r_out, o_out) and torch.equal(r_tl, o_tl), f"oracle forward_global_full != reference ({tag})"
            toks = torch.stack([ref[f][3] for f in range(T)], 2)          # [B, 9, T] the reference's own greedy tokens
            start = m.codecformer_text_emb(toks[:, 0, :])
            r_loc = m.forward_local(local_start_token=start, sequence=toks[:, 1:, :], transformer_out=r_out)
            o_loc = L.forward_local(wd, cfg, L.scaled_embedding(toks[:, 0, :], wd["codecformer_text_emb.weight"]), toks[:, 1:, :], o_out)
            # forward_local slices [B*T, 8, D] activations per step (x[:, t]): on CPU those strided GEMMs take MKL paths
            # that depend on the operands' page alignment (bitwise-equal inputs at other addresses differ by 1 ulp), so
            # this one comparison is to rounding, not bit for bit (B*T == 1 -- the InferenceImp loop -- is bit-exact)
            d = (r_loc.float() - o_loc.float()).abs().max().item()
            assert d <= (2e-6 if dtype == torch.float32 else 4e-2) * max(1.0, r_loc.float().abs().max().item()), (tag, d)
        print(f"gqa/partial-rope {tag}: oracle forward_global_full == reference; forward_local max |diff| {d:.2e} (T={T})")
        save[f"gqa_{tag}_full_out"] = r_out.float().numpy()
        if tag == "bf16":
            save["gqa_bf16_full_text_top"] = r_tl.float().topk(8, dim=-1).values.numpy()
            save["gqa_bf16_local_argmax"] = r_loc.float().argmax(-1).numpy()
        cols = sample_cols(r_loc.shape[-1])
        save["gqa_local_logits_cols"] = cols.numpy()
        save[f"gqa_{tag}_local_logits_sampled"] = r_loc.float()[..., cols].numpy()
        save[f"gqa_{tag}_local_tokens"] = toks.numpy()
    save["gqa_weights_sha256"] = np.array(weights_digest(L.synthetic_weights(cfg, seed=17, dtype=torch.float32, std=0.05)))


def gen_lora(save):
    """LoRA merge (llama_streaming.py:113-143, 368-406, 1120-1124): a reference GPT with lora_r > 0 on every wrapped
    linear, seeded lora_A / lora_B, merged by the reference's merge_lora_weights; the merged weights are the golden."""
    sys.path.insert(0, REF)
    from models.llama_streaming import merge_lora_weights
    import dataclasses
    cfg = dataclasses.replace(L.SMALL, n_query_groups=2)
    lora = dict(lora_r=4, lora_alpha=8, lora_dropout=0.0, lora_query=True, lora_key=False, lora_value=True,
                lora_projection=True, lora_mlp=True, lora_head=True)
    w = L.synthetic_weights(cfg, seed=27, dtype=torch.float32, std=0.05)
    m = reference_gpt(w, cfg, torch.float32, **lora)
    sd = m.state_dict()
    lw = L.synthetic_lora(cfg, seed=28, r=4, enable=(True, False, True))
    assert {k for k in sd if "lora_" in k} == set(lw.keys()), {k for k in sd if "lora_" in k} ^ set(lw.keys())
    m.load_state_dict({**w, **lw}, strict=True)
    merge_lora_weights(m)
    msd = m.state_dict()
    names = ["transformer.h.0.attn.attn.linear.weight", "transformer.h.1.attn.proj.linear.weight",
             "transformer.h.0.mlp.fc_1.linear.weight", "transformer.h.1.mlp.fc_2.linear.weight",
             "transformer.h.0.mlp.proj.linear.weight"]
    for i, n in enumerate(names):
        assert not torch.equal(msd[n], w[n])
        u, s, v = torch.linalg.svd((msd[n].double() - w[n].double()), full_matrices=False)
        r = int((s > 1e-6 * s[0]).sum())
        u, v = (u[:, :r] * s[:r]).float(), v[:r].float()
        assert (w[n] + u @ v - msd[n]).abs().max().item() <= 1e-7, n       # the tests compare to 2e-6
        save[f"lora_update_{i}_u"], save[f"lora_update_{i}_v"] = u.numpy(), v.numpy()
    save["lora_names"] = np.array(names)
    save["lora_head_rows"] = msd["lm_head.linear.weight"][:64].numpy()
    print("lora: merged weights stored")


def main():
    global REF
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "models")):
        sys.exit("usage: python -m oracle.gen_golden_lm <MLLM_v2 directory of the original RSTnet checkout>")
    REF = os.path.abspath(sys.argv[1])
    torch.set_num_threads(GOLDEN_THREADS)
    os.makedirs(GOLDEN, exist_ok=True)
    extra = {}
    gen_infer(extra)
    gen_variant(extra)
    gen_lora(extra)
    np.savez_compressed(os.path.join(GOLDEN, "lm_round2.npz"), **extra)
    print("wrote", os.path.join(GOLDEN, "lm_round2.npz"))
    cfg = L.SMALL
    B, frames = 3, 20  # 20 > context (16): the ring wraps
    g = torch.Generator().manual_seed(99)
    seqs = []
    for f in range(frames):
        s = torch.randint(0, 2048, (B, cfg.n_q + 1, 1), generator=g)
        s[:, 0] = torch.randint(0, 150000, (B, 1), generator=g)
        if f == 0:
            s[:, 1:] = cfg.audio_card          # initial audio token (llama_streaming.py:609)
            s[:, 0] = 151655                    # hard-coded text_initial_token_id (:598-604)
        if f == 3:
            s[0, 2] = -1                        # zero_token_id row (ScaledEmbedding, :505-517)
        seqs.append(s)
    save = {}
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        w = L.synthetic_weights(cfg, seed=7, dtype=torch.float32, std=0.05)
        wd = {k: v.to(dtype) for k, v in w.items()}
        ref = reference_frames(w, cfg, seqs, dtype)
        gs = L.GPTStream(wd, cfg, B)
        with torch.no_grad():
            for f, seq in enumerate(seqs):
                o = L.greedy_frame(gs, seq)
                for a, b, name in zip(o, ref[f], ("out", "text_logits", "audio_logits", "tokens")):
                    assert torch.equal(a, b), f"oracle != reference: {tag} frame {f} {name}: {(a.float() - b.float()).abs().max()}"
        print(f"{tag}: oracle == reference on {frames} frames (bit for bit)")
        keep = (0, 1, 3, 15, 16, 19)
        save[f"{tag}_out"] = torch.stack([ref[f][0].float() for f in keep]).numpy()
        save[f"{tag}_text_top"] = torch.stack([ref[f][1].float().topk(8, dim=-1).values for f in keep]).numpy()
        save[f"{tag}_audio_logits_sha256"] = np.array([f32_sha256(ref[f][2]) for f in keep])
        if tag == "bf16":
            save["bf16_audio_logits_bits"] = bf16_bits(torch.stack([ref[f][2] for f in keep]))
        save[f"{tag}_tokens"] = torch.stack([ref[f][3] for f in range(frames)]).numpy()
        save[f"{tag}_keep"] = np.array(keep)
        if tag == "f32":
            save["weights_sha256"] = np.array(weights_digest(w))
    save["seqs"] = torch.stack(seqs).numpy()
    np.savez_compressed(os.path.join(GOLDEN, "lm_small.npz"), **save)
    print("wrote", os.path.join(GOLDEN, "lm_small.npz"))


if __name__ == "__main__":
    main()
