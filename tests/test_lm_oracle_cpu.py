"""CPU suite: the LM oracle against the golden vectors of the unmodified reference (oracle/gen_golden_lm.py),
and host-side checks of the product GPT mirror (no GPU)."""
import os

import numpy as np
import pytest
import torch

from oracle import lm_oracle as L
from oracle.gen_golden import weights_digest
from oracle.gen_golden_lm import f32_sha256


@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("bf16", torch.bfloat16)])
def test_lm_oracle_matches_reference_golden(golden_dir, tag, dtype):
    g = np.load(os.path.join(golden_dir, "lm_small.npz"))
    cfg = L.SMALL
    w = L.synthetic_weights(cfg, seed=7, dtype=torch.float32, std=0.05)
    assert weights_digest(w) == str(g["weights_sha256"])
    wd = {k: v.to(dtype) for k, v in w.items()}
    seqs = torch.from_numpy(g["seqs"])
    gs = L.GPTStream(wd, cfg, seqs.shape[1])
    keep = list(g[f"{tag}_keep"])
    with torch.no_grad():
        for f in range(seqs.shape[0]):
            out, tl, al, toks = L.greedy_frame(gs, seqs[f])
            assert np.array_equal(toks.numpy(), g[f"{tag}_tokens"][f])                 # bit-exact greedy tokens
            if f in keep:
                i = keep.index(f)
                assert np.array_equal(out.float().numpy(), g[f"{tag}_out"][i])
                assert f32_sha256(al) == str(g[f"{tag}_audio_logits_sha256"][i])          # bit-exact audio logits


def test_ring_labels_oldest_slot_as_end_offset():
    """RingKVCache.complete quirk (lit_model.py:648-655): once wrapped, the oldest entry is masked."""
    r = L.Ring(1, 1, 4, 4, torch.float32)
    for t in range(6):
        _, _, pos = r.complete(torch.zeros(1, 1, 1, 4), torch.zeros(1, 1, 1, 4))
    assert pos.tolist() == [4, 5, 6, 3] or sorted(pos.tolist()) == [3, 4, 5, 6]
    assert int(pos[r.end_offset % 4]) == r.end_offset  # labelled with a FUTURE position -> never attended


def test_product_gpt_state_dict_keys_and_token_ids():
    from rstnet_b200.lm import GPT, Config
    cfg = L.SMALL
    m = GPT(Config(block_size=cfg.block_size, n_layer=cfg.n_layer, n_embd=cfg.n_embd, n_head=cfg.n_head, head_size=cfg.head_size,
                   intermediate_size=cfg.intermediate_size, padded_vocab_size=cfg.padded_vocab_size, audio_card=cfg.audio_card,
                   n_q=cfg.n_q, dep_q=cfg.dep_q, codecformer_dim=cfg.codecformer_dim, codecformer_heads=cfg.codecformer_heads,
                   codecformer_layers=cfg.codecformer_layers, codecformer_dim_feedforward=cfg.codecformer_dim_feedforward,
                   context=cfg.context))
    spec = {n: s for n, s, _ in L.param_spec(cfg)}
    sd = m.state_dict()
    assert set(sd) == set(spec)
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), k
    w = L.synthetic_weights(cfg, seed=7, std=0.05)
    old = dict(w)
    old["lm_head.weight"] = old.pop("lm_head.linear.weight")                       # base-checkpoint names
    old["transformer.h.0.attn.attn.weight"] = old.pop("transformer.h.0.attn.attn.linear.weight")
    m.load_state_dict(old, strict=True)
    assert torch.equal(m.state_dict()["transformer.h.0.attn.attn.linear.weight"], w["transformer.h.0.attn.attn.linear.weight"])
    t = m._get_initial_token()
    assert t.shape == (1, 9, 1) and int(t[0, 0, 0]) == 151655 and int(t[0, 1, 0]) == cfg.audio_card
    from rstnet_b200._lib import RstnetError
    with pytest.raises(RstnetError):
        m.streaming_forever(2)   # CPU / fp32: refused, no fallback


def test_reverse_delay_matches_the_reference_rule():
    """infer_no_streaming.py:311-323: codebook 0 keeps frames [0, L-1), codebooks 1..7 are shifted left by one frame;
    an [L, 8] input is transposed first.  Checked against a direct restatement of that rule."""
    from rstnet_b200.infer import reverse_delay
    g = torch.Generator().manual_seed(3)
    x = torch.randint(0, 2048, (8, 11), generator=g)
    want = torch.ones_like(x)
    want[0, :-1] = x[0, :-1]
    want[1:, :-1] = x[1:, 1:]
    want = want[:, :-1]
    assert torch.equal(reverse_delay(x), want)
    assert torch.equal(reverse_delay(x.t().contiguous()), want)
    assert reverse_delay(x).shape == (8, 10)
