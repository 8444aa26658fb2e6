"""GPU parity tests of the LM decode step (-m gpu): CUDA kernels vs the CPU oracle (oracle/lm_oracle.py)
and vs the golden vectors of the unmodified reference (tests/golden/lm_small.npz).

bf16 tolerance (SURVEY.md §8d cfg 3): activations / logits rel. error <= 2e-2 of the tensor's scale and
cosine similarity >= 0.999; greedy tokens equal except on near-ties (>= 90 % of frames under teacher forcing).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import lm_oracle as L
from rstnet_b200 import _lib, ops
from rstnet_b200.lm import GPT, Config, SkinnyGemm

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF = torch.bfloat16


def _cos(a, b):
    a, b = a.float().flatten().cpu(), b.float().flatten().cpu()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp(min=1e-12))


def _rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-6))


@pytest.mark.parametrize("M,K,N,res", [(64, 4096, 512, False), (64, 256, 768, False), (3, 256, 152064 // 64, True), (64, 11008, 256, True),
                                       (17, 1024, 2050, False), (64, 2816, 1024, True), (128, 512, 640, False)])
def test_skinny_gemm_vs_torch(M, K, N, res):
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g).to(BF)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(BF)
    r = torch.randn(M, N, generator=g).to(BF) if res else None
    ref = x.float() @ w.float().t()
    if res:
        ref = ref + r.float()
    xd, wd = x.to(DEV), w.to(DEV)
    out = r.to(DEV).clone() if res else torch.empty(M, N, dtype=BF, device=DEV)
    ws = torch.empty(8 * M * N, dtype=torch.float32, device=DEV)
    plan = SkinnyGemm(xd, wd, out, out if res else None, ws)
    plan.run()
    torch.cuda.synchronize()
    err = (out.float().cpu() - ref).abs().max().item()
    assert err <= 2e-2 * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("M,K,I", [(64, 1024, 2816), (5, 256, 96), (128, 512, 704)])
def test_skinny_gemm_interleaved_silu_gating(M, K, I):
    """fin_mode 3: SiLU gating inside the GEMM epilogue on row-interleaved weights == the finalize-kernel form (fin_mode 2)
    on the stacked [gate; value] weight, bit for bit (same roundings), and == torch within bf16 tolerance."""
    from rstnet_b200.lm import interleave_gate_rows
    g = torch.Generator().manual_seed(M + K + I)
    x = torch.randn(M, K, generator=g).to(BF).to(DEV)
    w1 = (torch.randn(I, K, generator=g) / K ** 0.5).to(BF).to(DEV)
    w2 = (torch.randn(I, K, generator=g) / K ** 0.5).to(BF).to(DEV)
    ws = torch.empty(8 * M * 2 * I, dtype=torch.float32, device=DEV)
    out_a = torch.zeros(M, I, dtype=BF, device=DEV)
    out_b = torch.zeros(M, I, dtype=BF, device=DEV)
    SkinnyGemm(x, torch.cat([w1, w2], 0).contiguous(), None, None, ws, silu_out=out_a).run()
    SkinnyGemm(x, interleave_gate_rows(w1, w2), None, None, None, silu_out=out_b, interleaved=True).run()
    torch.cuda.synchronize()
    a = (x.float() @ w1.float().t()).to(BF).float()
    b = (x.float() @ w2.float().t()).to(BF).float()
    ref = F.silu(a).to(BF).float() * b
    assert _rel(out_b, ref) <= 2e-2
    if I % 4 == 0:
        # one K slice on both sides would be bit-identical; the finalize form may split K, so compare to bf16 rounding
        assert _rel(out_b, out_a) <= 2e-2


@pytest.mark.parametrize("hs,cap,context,steps", [(128, 32, 32, 70), (64, 16, 16, 20), (128, 2048, 2048, 3)])
def test_rope_append_and_ring_decode_attention(hs, cap, context, steps):
    """RoPE + ring append + single-query attention vs the oracle's Ring / SDPA, including ring wrap."""
    B, nh = 3, 4
    cfg = L.LMConfig(n_head=nh, head_size=hs, context=context, block_size=max(128, steps + 1))
    cos, sin = L.rope_cache(cfg, BF)
    ring = L.Ring(B, nh, hs, cap, BF)
    kv = torch.zeros(2, B, nh, cap, hs, dtype=BF, device=DEV)
    offset = torch.zeros(1, dtype=torch.int64, device=DEV)
    g = torch.Generator().manual_seed(hs + cap)
    lib = _lib.lib()
    cos_d, sin_d = cos.to(DEV).contiguous(), sin.to(DEV).contiguous()
    for step in range(steps):
        qkv = torch.randn(B, nh, 3, hs, generator=g).to(BF)
        q, k, v = [qkv[:, :, i][:, :, None] for i in range(3)]  # [B,nh,1,hs]
        c, s = cos[step:step + 1], sin[step:step + 1]
        qr, kr = L.apply_rope(q, c, s), L.apply_rope(k, c, s)
        kk, vv, pos_k = ring.complete(kr, v)
        pos_k = pos_k.view(1, -1)
        delta = step - pos_k
        mask = (pos_k >= 0) & (delta >= 0) & (delta < context)
        ref = F.scaled_dot_product_attention(qr.float(), kk.float(), vv.float(), attn_mask=mask, scale=1.0 / hs ** 0.5)[:, :, 0]
        qd = torch.empty(B, nh * hs, dtype=BF, device=DEV)
        out = torch.empty(B, nh * hs, dtype=BF, device=DEV)
        st = ops._stream()
        qkv_d = qkv.to(DEV).contiguous()
        _lib.check(lib.rstnet_lm_rope_kv_append_bf16(qkv_d.data_ptr(), cos_d.data_ptr(), sin_d.data_ptr(), cos_d.shape[0], hs,
                                                     offset.data_ptr(), 0, qd.data_ptr(), kv.data_ptr(), B, B, nh, nh, hs, cap, st))
        _lib.check(lib.rstnet_lm_ring_decode_attention_bf16(qd.data_ptr(), kv.data_ptr(), offset.data_ptr(), 0, out.data_ptr(), B, B,
                                                            nh, nh, hs, cap, context, None, st))
        ops.counter_add(offset, 1)
        torch.cuda.synchronize()
        assert torch.equal(qd.cpu().view(B, nh, hs), qr[:, :, 0]), "rotated q must match bit for bit"
        err = (out.float().cpu().view(B, nh, hs) - ref).abs().max().item()
        assert err <= 1.5e-2, (step, err)
    assert torch.equal(kv.cpu(), ring.cache)


def test_norms_silu_embed_vs_oracle():
    g = torch.Generator().manual_seed(1)
    lib, st = _lib.lib(), ops._stream()
    x = (torch.randn(5, 1, 256, generator=g) * 2).to(BF)
    w = (1 + 0.1 * torch.randn(256, generator=g)).to(BF)
    for ky, ref in ((0, L.rms_norm(x, w, 1e-5)), (1, L.rms_norm_f32(x, w.view(1, 1, -1), 1e-8))):
        y = torch.empty(5, 256, dtype=BF, device=DEV)
        xd, wd = x.to(DEV).contiguous(), w.to(DEV).contiguous()
        _lib.check(lib.rstnet_lm_rms_norm_bf16(xd.data_ptr(), wd.data_ptr(), y.data_ptr(), 5, 256, 1e-5 if ky == 0 else 1e-8, ky, st))
        torch.cuda.synchronize()
        d = (y.float().cpu() - ref[:, 0].float()).abs().max().item()
        assert d <= 2e-2, (ky, d)  # at most one bf16 ulp at |y| ~ 4
    ab = torch.randn(7, 2 * 96, generator=g).to(BF)
    ref = F.silu(ab[:, :96]) * ab[:, 96:]
    out = torch.empty(7, 96, dtype=BF, device=DEV)
    abd = ab.to(DEV).contiguous()
    _lib.check(lib.rstnet_lm_silu_mul_bf16(abd.data_ptr(), out.data_ptr(), 7, 96, st))
    torch.cuda.synchronize()
    assert (out.float().cpu() - ref.float()).abs().max().item() <= 4e-2


def test_sampling_greedy_and_distribution():
    lib, st = _lib.lib(), ops._stream()
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(6, 5000, generator=g).to(BF)
    logits[2, 100] = logits[2, 4000] = 9.0  # tie -> first maximum
    toks = torch.zeros(6, 3, dtype=torch.int64, device=DEV)
    logits_d = logits.to(DEV).contiguous()
    _lib.check(lib.rstnet_lm_sample_bf16(logits_d.data_ptr(), 6, 5000, 5000, 0, 1.0, 1, None, toks.data_ptr() + 8, 3, st))
    assert torch.equal(toks[:, 1].cpu(), torch.argmax(logits.float(), -1)) and int(toks[2, 1]) == 100
    # n_valid masks the tail (sample_token_audio_2048: ids >= 2048 never sampled)
    _lib.check(lib.rstnet_lm_sample_bf16(logits_d.data_ptr(), 6, 5000, 90, 0, 1.0, 1, None, toks.data_ptr(), 3, st))
    assert int(toks[:, 0].max()) < 90
    # distribution of the exponential-noise multinomial over the top-k (utils/sampling.py:157-175 self-test)
    ps = torch.tensor([5.0, 2.0, 12.0, 6.0, 8.0, 1.0, 0.5, 4.0])
    lg = torch.log(ps).to(BF).repeat(4000, 1).contiguous().to(DEV)
    out = torch.zeros(4000, dtype=torch.int64, device=DEV)
    _lib.check(lib.rstnet_lm_sample_bf16(lg.data_ptr(), 4000, 8, 8, 8, 1.0, 77, None, out.data_ptr(), 1, st))
    cnt = torch.bincount(out.cpu(), minlength=8).float()
    target = torch.exp(torch.log(ps).to(BF).float())
    assert (cnt / cnt.sum() - target / target.sum()).abs().max().item() < 2.5e-2
    # top-k restricts the support
    _lib.check(lib.rstnet_lm_sample_bf16(lg.data_ptr(), 4000, 8, 8, 3, 1.0, 78, None, out.data_ptr(), 1, st))
    assert set(out.cpu().tolist()) <= {2, 4, 3}


def test_sampling_large_vocab_candidate_list_matches_full_scan():
    """The 152k-entry text head goes through the histogram-select candidate list; it must pick exactly what the plain
    top_k-pass scan picks (same seed, same (value desc, index asc) order), ties at the threshold included."""
    lib, st = _lib.lib(), ops._stream()
    g = torch.Generator().manual_seed(11)
    rows, V, small = 32, 151936, 4000
    logits = (torch.randn(rows, V, generator=g) * 2.0).to(BF)
    logits[:, small:] = torch.minimum(logits[:, small:], torch.tensor(1.0).to(BF))   # the whole top-k lives in ids < small
    logits[:, :small] += 3.0
    logits[3, 10:40] = 7.5      # 30 equal values straddling the top-25 boundary -> lowest ids win
    logits[4, :] = 0.25         # massive tie: falls back to the full scan
    ld = logits.to(DEV).contiguous()
    a = torch.zeros(rows, dtype=torch.int64, device=DEV)
    b = torch.zeros(rows, dtype=torch.int64, device=DEV)
    for top_k, seed in ((25, 5), (64, 6), (2, 7)):
        _lib.check(lib.rstnet_lm_sample_bf16(ld.data_ptr(), rows, V, small, top_k, 0.8, seed, None, a.data_ptr(), 1, st))
        _lib.check(lib.rstnet_lm_sample_bf16(ld.data_ptr(), rows, V, V, top_k, 0.8, seed, None, b.data_ptr(), 1, st))
        torch.cuda.synchronize()
        keep = torch.ones(rows, dtype=torch.bool); keep[4] = False   # row 4's top-k is not inside ids < small
        assert torch.equal(a.cpu()[keep], b.cpu()[keep]), top_k
        topk = torch.topk(logits.float(), top_k, dim=-1).values[:, -1:]
        picked = logits.float().gather(1, b.cpu()[:, None])
        assert (picked >= topk).all()
        assert int(b[4]) < top_k     # all-equal row: the top-k are ids 0..top_k-1
    _lib.check(lib.rstnet_lm_sample_bf16(ld.data_ptr(), rows, V, V, 0, 1.0, 1, None, b.data_ptr(), 1, st))
    assert torch.equal(b.cpu(), torch.argmax(logits.float(), -1))


@pytest.fixture(scope="module")
def small_lm():
    cfg = L.SMALL
    w32 = L.synthetic_weights(cfg, seed=7, dtype=torch.float32, std=0.05)
    m = GPT(Config(block_size=cfg.block_size, n_layer=cfg.n_layer, n_embd=cfg.n_embd, n_head=cfg.n_head, head_size=cfg.head_size,
                   intermediate_size=cfg.intermediate_size, norm_eps=cfg.norm_eps, padded_vocab_size=cfg.padded_vocab_size,
                   audio_card=cfg.audio_card, n_q=cfg.n_q, dep_q=cfg.dep_q, codecformer_dim=cfg.codecformer_dim,
                   codecformer_heads=cfg.codecformer_heads, codecformer_layers=cfg.codecformer_layers,
                   codecformer_dim_feedforward=cfg.codecformer_dim_feedforward, context=cfg.context))
    assert set(m.state_dict().keys()) == set(w32.keys())
    m.load_state_dict(w32, strict=True)
    return m.to(DEV, BF).eval(), {k: v.to(BF) for k, v in w32.items()}, cfg


@pytest.mark.parametrize("graphs", [False, True])
def test_streaming_decode_vs_reference_golden(golden_dir, small_lm, graphs):
    """20 teacher-forced frames (ring wraps at 16) vs the reference's bf16 outputs."""
    m, w, cfg = small_lm
    gold = np.load(os.path.join(golden_dir, "lm_small.npz"))
    seqs = torch.from_numpy(gold["seqs"])
    keep = list(gold["bf16_keep"])
    m.use_cuda_graphs = graphs
    tok_ok, n_tok = 0, 0
    # fp32 evaluation of the same bf16-valued weights: the yardstick for "bf16 noise"
    truth = L.GPTStream({k: v.float() for k, v in w.items()}, cfg, 3)
    worst = 0.0
    with m.streaming(3):
        for f in range(seqs.shape[0]):
            seq = seqs[f].to(DEV)
            with torch.no_grad():
                t_out, _ = truth.forward_global(seqs[f])
                truth.start_depth()
                t_al = []
                for k in range(cfg.dep_q):
                    prev_t = torch.from_numpy(gold["bf16_tokens"][f])[:, k].view(3, 1, 1)
                    t_al.append(truth.forward_codecformer(k, prev_t, t_out)[:, 0, 0])
                t_al = torch.stack(t_al, 1)
            out, tl = m.forward_global(seq)
            assert out.shape == (3, 1, cfg.n_embd) and tl.shape == (3, 1, cfg.padded_vocab_size)
            ref_tokens = torch.from_numpy(gold["bf16_tokens"][f])
            al = []
            with m.codecformer.streaming(3):
                prev = ref_tokens[:, 0].view(3, 1, 1).to(DEV)   # teacher forcing with the reference's tokens
                for k in range(cfg.dep_q):
                    lg = m.forward_codecformer(k, prev, out)
                    assert lg.shape == (3, 1, 1, cfg.audio_card)
                    al.append(lg[:, 0, 0])
                    prev = ref_tokens[:, k + 1].view(3, 1, 1).to(DEV)
            al = torch.stack(al, 1)
            my_tokens = torch.cat([tl.float().argmax(-1), al.float().argmax(-1)], 1).cpu()
            tok_ok += int((my_tokens == ref_tokens).sum())
            n_tok += ref_tokens.numel()
            if f in keep:
                i = keep.index(f)
                ro, ra = torch.from_numpy(gold["bf16_out"][i]), torch.from_numpy(gold["bf16_audio_logits_bits"][i]).view(BF).float()
                assert _cos(out, ro) >= 0.999 and _cos(al, ra) >= 0.999, (f, _cos(out, ro), _cos(al, ra))
                # our deviation from the fp32 evaluation must be of the same size as the reference's own bf16 deviation
                e_mine, e_ref = _rel(out, t_out), _rel(ro, t_out)
                a_mine, a_ref = _rel(al, t_al), _rel(ra, t_al)
                worst = max(worst, e_mine / max(e_ref, 1e-3), a_mine / max(a_ref, 1e-3))
                assert e_mine <= 2.0 * e_ref + 1e-2 and a_mine <= 2.0 * a_ref + 1e-2, (f, e_mine, e_ref, a_mine, a_ref)
                top = tl.float().topk(8, dim=-1).values.cpu()
                assert _rel(top, torch.from_numpy(gold["bf16_text_top"][i])) <= 8e-2
    print(f"worst (our bf16 error) / (reference bf16 error) vs fp32 evaluation: {worst:.2f}")
    print(f"greedy token agreement with the reference: {tok_ok}/{n_tok}")
    assert tok_ok / n_tok >= 0.9


def test_forward_step_matches_stepwise_api(small_lm):
    """forward_step (one graph per frame, device-side sampling) == forward_global + 8 x forward_codecformer, greedy."""
    m, w, cfg = small_lm
    g = torch.Generator().manual_seed(3)
    seqs = [torch.randint(0, 2048, (3, 9, 1), generator=g).to(DEV) for _ in range(4)]
    m.use_cuda_graphs = True
    a = []
    with m.streaming(3):
        for s in seqs:
            a.append(m.forward_step(s, use_sampling=False))
    b = []
    with m.streaming(3):
        for s in seqs:
            out, tl = m.forward_global(s)
            toks = [tl.float().argmax(-1)[:, 0]]
            with m.codecformer.streaming(3):
                prev = toks[0].view(3, 1, 1)
                for k in range(cfg.dep_q):
                    lg = m.forward_codecformer(k, prev, out)
                    prev = lg.float().argmax(-1)
                    toks.append(prev[:, 0, 0])
            b.append(torch.stack(toks, 1))
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    with m.streaming(3):
        t = m.forward_step(seqs[0], use_sampling=True)
        assert t.shape == (3, 9) and int(t[:, 1:].max()) < 2049 and int(t.min()) >= 0


def _replay_ok(frames, seq, w, cfg, use_sampling, tol):
    """Every decision of a closed-loop run, checked under the oracle teacher-forced with those very tokens: the chosen
    id must be allowed by the candidate-set rule and within `tol` of the oracle's best logit (exactly the argmax
    unless the top candidates are a bf16 near-tie)."""
    from oracle import infer_oracle as IO
    with torch.no_grad():
        r = IO.inference_imp_tts(w, cfg, seq.clone(), use_sampling, force=frames)
    d = r["deficit"]
    assert torch.isfinite(d).all(), "a masked id (>= 2048 / 2049) was chosen"
    assert float(d.max()) <= tol, f"a chosen token is {float(d.max()):.3f} below the oracle's best logit"
    return int((d == 0).sum()), d.numel()


@pytest.mark.parametrize("mode,use_sampling,tk", [("greedy", False, 0), ("top1", True, 1)])
def test_inference_imp_vs_reference_loop(golden_dir, small_lm, mode, use_sampling, tk):
    """InferenceImp (infer_no_streaming.py:169-308) as a streaming loop (prefill + forward_step) against the UNMODIFIED
    reference's O(T^2) loop: the reference's bf16 tokens (tests/golden/lm_round2.npz, generated by
    oracle/gen_golden_lm.py from the original project) must be reproduced up to the first bf16 near-tie, and every decision of
    our own closed loop must be (near-)optimal under the oracle restatement of that loop (pinned bit for bit to the
    reference), which also checks the 2048 / 2049 candidate rules, the delay bookkeeping and the prompt handling."""
    from rstnet_b200.infer import InferenceImp, reverse_delay
    m, w, cfg = small_lm
    gold = np.load(os.path.join(golden_dir, "lm_round2.npz"))
    seq = torch.from_numpy(gold["infer_seq"])
    ref_frames = torch.from_numpy(gold[f"infer_bf16_{mode}_frames"])
    ref_codes = torch.from_numpy(gold[f"infer_bf16_{mode}_codes"])
    margins = torch.from_numpy(gold[f"infer_bf16_{mode}_margins"])
    imp = InferenceImp(None, m, "sampling", 0.7, tk, 0.8, tk, "TTS")
    imp.use_sampling = use_sampling
    m.use_cuda_graphs = True
    codes, raw = imp.generate(seq.unsqueeze(0).to(DEV), return_frames=True)
    out = imp(seq.to(DEV), torch.ones_like(seq).to(DEV))
    assert out.shape == ref_codes.shape and out.dtype == torch.int64
    assert torch.equal(out.cpu(), codes[0].cpu())                      # deterministic, __call__ == generate
    mine = raw[0].cpu()
    assert torch.equal(reverse_delay(mine[:, 1:]), codes[0].cpu())
    # (1) against the reference's tokens: identical up to the first near-tie decision (then the loops diverge by design)
    tol = 0.07   # ~ 4 bf16 ulps at |logit| ~ 2-4, the size of the bf16 evaluation noise of this model
    flat_m, flat_r, flat_o = margins.flatten(), ref_frames.flatten(), mine.flatten()
    first_tie = int((flat_m <= tol).nonzero()[0]) if bool((flat_m <= tol).any()) else flat_m.numel()
    assert torch.equal(flat_o[:first_tie], flat_r[:first_tie]), "tokens differ from the reference before any near-tie"
    # (2) every decision of our closed loop under the oracle
    exact, n = _replay_ok(mine, seq, w, cfg, use_sampling, tol)
    print(f"{mode}: identical to the reference for the first {first_tie}/{flat_m.numel()} decisions; "
          f"{exact}/{n} decisions are the oracle's exact argmax, the rest within {tol}")
    assert exact >= 0.8 * n


def test_inference_imp_batched_and_sampling(small_lm):
    """B > 1 generation (BASELINE cfg 4's shape class): identical rows give identical tokens; sampling mode respects
    the candidate sets."""
    from rstnet_b200.infer import InferenceImp
    m, w, cfg = small_lm
    g = torch.Generator().manual_seed(11)
    P, G = 7, 6
    seq = torch.randint(0, 2048, (9, P + G), generator=g)
    seq[0, :P] = torch.randint(0, 1000, (P,), generator=g)
    seq[0, P:] = 128002
    imp = InferenceImp(None, m, "sampling", 0.7, 25, 0.8, 30, "TTS")
    imp.use_sampling = False
    one = imp(seq.to(DEV), torch.ones(9, P + G).to(DEV))
    many = imp.generate(seq.unsqueeze(0).expand(5, -1, -1).contiguous().to(DEV))
    assert many.shape == (5, 8, G - 1)
    for b in range(5):
        assert torch.equal(many[b], one)
    imp.use_sampling = True
    sam, raw = imp.generate(seq.unsqueeze(0).expand(4, -1, -1).contiguous().to(DEV), return_frames=True)
    assert sam.shape == (4, 8, G - 1) and int(raw[:, :, 1:].max()) < 2049 and int(raw.min()) >= 0
    assert int(raw[:, 1:, 1].max()) < 2048          # codebook 0 after the first generated frame: ids < 2048 only


def _variant_cfg():
    import dataclasses
    return dataclasses.replace(L.SMALL, n_query_groups=2, rotary_percentage=0.5,
                               rope_adjustments={"factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                                                 "original_max_seq_len": 32})


def _product_config(cfg, **kw):
    return Config(block_size=cfg.block_size, n_layer=cfg.n_layer, n_embd=cfg.n_embd, n_head=cfg.n_head, head_size=cfg.head_size,
                  n_query_groups=cfg.n_kv, rotary_percentage=cfg.rotary_percentage, rope_adjustments=cfg.rope_adjustments,
                  intermediate_size=cfg.intermediate_size, norm_eps=cfg.norm_eps, padded_vocab_size=cfg.padded_vocab_size,
                  audio_card=cfg.audio_card, n_q=cfg.n_q, dep_q=cfg.dep_q, codecformer_dim=cfg.codecformer_dim,
                  codecformer_heads=cfg.codecformer_heads, codecformer_layers=cfg.codecformer_layers,
                  codecformer_dim_feedforward=cfg.codecformer_dim_feedforward, context=cfg.context, **kw)


@pytest.fixture(scope="module")
def gqa_lm(golden_dir):
    from oracle.gen_golden import weights_digest
    cfg = _variant_cfg()
    w32 = L.synthetic_weights(cfg, seed=17, dtype=torch.float32, std=0.05)
    gold = np.load(os.path.join(golden_dir, "lm_round2.npz"))
    assert weights_digest(w32) == str(gold["gqa_weights_sha256"])
    m = GPT(_product_config(cfg))
    assert set(m.state_dict().keys()) == set(w32.keys())
    m.load_state_dict(w32, strict=True)
    return m.to(DEV, BF).eval(), {k: v.to(BF) for k, v in w32.items()}, cfg, gold


def test_gqa_partial_rope_streaming_vs_reference_golden(gqa_lm):
    """Grouped-query attention (K/V stored once per group), rotary_percentage 0.5 and Llama-3.1 rope adjustments
    (llama_streaming.py:952-982, lit_model.py:110-144): 20 teacher-forced streaming frames vs the reference's bf16 run."""
    m, w, cfg, gold = gqa_lm
    seqs = torch.from_numpy(gold["gqa_seqs"])
    keep = list(gold["gqa_keep"])
    ref_tokens = torch.from_numpy(gold["gqa_bf16_tokens"])
    tok_ok = n_tok = 0
    m.use_cuda_graphs = True
    with m.streaming(3):
        for f in range(seqs.shape[0]):
            out, tl = m.forward_global(seqs[f].to(DEV))
            al = []
            with m.codecformer.streaming(3):
                prev = ref_tokens[f][:, 0].view(3, 1, 1).to(DEV)
                for k in range(cfg.dep_q):
                    al.append(m.forward_codecformer(k, prev, out)[:, 0, 0])
                    prev = ref_tokens[f][:, k + 1].view(3, 1, 1).to(DEV)
            al = torch.stack(al, 1)
            mine = torch.cat([tl.float().argmax(-1), al.float().argmax(-1)], 1).cpu()
            tok_ok += int((mine == ref_tokens[f]).sum()); n_tok += mine.numel()
            if f in keep:
                i = keep.index(f)
                ro = torch.from_numpy(gold["gqa_bf16_out"][i])
                ra = torch.from_numpy(gold["gqa_bf16_audio_logits_bits"][i]).view(BF).float()
                assert _cos(out, ro) >= 0.999 and _cos(al, ra) >= 0.999, (f, _cos(out, ro), _cos(al, ra))
                assert _rel(out, ro) <= 5e-2 and _rel(al, ra) <= 5e-2
    print(f"gqa greedy token agreement with the reference: {tok_ok}/{n_tok}")
    assert tok_ok / n_tok >= 0.9


def test_prefill_equals_single_steps_and_reference_full_forward(gqa_lm):
    """forward_global over T > 1 positions in one call (SURVEY.md §8f-2, llama_streaming.py:651-692): same KV rings and
    outputs as T single-step calls, and the reference's NON-streaming forward_global golden (T < context)."""
    m, w, cfg, gold = gqa_lm
    seqs = torch.from_numpy(gold["gqa_seqs"])
    T = gold["gqa_bf16_full_out"].shape[1]
    full = torch.cat([seqs[f] for f in range(T)], dim=2).to(DEV)       # [3, 9, T]
    m.use_cuda_graphs = False
    with m.streaming(3):
        o_chunk, l_chunk = m.forward_global(full)
        kv_chunk = [k.clone() for k in m._state.kv]
        assert int(m._state.offset[0]) == T
        nxt_a = m.forward_global(seqs[T].to(DEV))[0]
    with m.streaming(3):
        outs, lgs = zip(*[m.forward_global(seqs[f].to(DEV)) for f in range(T)])
        kv_step = [k.clone() for k in m._state.kv]
        nxt_b = m.forward_global(seqs[T].to(DEV))[0]
    o_step, l_step = torch.cat(outs, 1), torch.cat(lgs, 1)
    for a, b in zip(kv_chunk, kv_step):
        assert torch.equal(a, b), "prefill must leave exactly the KV rings the single steps leave"
    assert torch.equal(o_chunk, o_step) and torch.equal(l_chunk, l_step) and torch.equal(nxt_a, nxt_b)
    ref = torch.from_numpy(gold["gqa_bf16_full_out"])
    assert _cos(o_chunk, ref) >= 0.999 and _rel(o_chunk, ref) <= 5e-2
    assert _rel(l_chunk.float().topk(8, dim=-1).values, torch.from_numpy(gold["gqa_bf16_full_text_top"])) <= 8e-2
    # the non-streaming form (no scope): same numbers, nothing kept
    o_ns, l_ns = m.forward_global(full)
    assert m._state is None and torch.equal(o_ns, o_chunk) and torch.equal(l_ns, l_chunk)
    # prompt-only feed (no outputs) leaves the same rings
    with m.streaming(3):
        m.prefill(full)
        for a, b in zip(m._state.kv, kv_step):
            assert torch.equal(a, b)


def test_prefill_across_ring_wrap_matches_single_steps(small_lm):
    """context 16, 20 positions: the chunked path must fall back to single positions once the ring would wrap."""
    m, w, cfg = small_lm
    g = torch.Generator().manual_seed(5)
    full = torch.randint(0, 2048, (3, 9, 20), generator=g).to(DEV)
    m.use_cuda_graphs = False
    with m.streaming(3):
        a, _ = m.forward_global(full)
    with m.streaming(3):
        b = torch.cat([m.forward_global(full[:, :, t:t + 1])[0] for t in range(20)], 1)
    assert torch.equal(a, b)


def test_forward_local_vs_reference_golden(gqa_lm):
    """GPT.forward_local (llama_streaming.py:694-725) vs the reference's bf16 output on its own greedy tokens."""
    m, w, cfg, gold = gqa_lm
    toks = torch.from_numpy(gold["gqa_bf16_local_tokens"]).to(DEV)           # [3, 9, T]
    t_out = torch.from_numpy(gold["gqa_bf16_full_out"]).to(DEV, BF)
    start = m.codecformer_text_emb(toks[:, 0, :])
    lg = m.forward_local(local_start_token=start, sequence=toks[:, 1:, :], transformer_out=t_out)
    ref_argmax = torch.from_numpy(gold["gqa_bf16_local_argmax"])                # over the whole vocabulary
    assert lg.shape[:-1] == ref_argmax.shape and lg.shape[-1] == cfg.audio_card
    ref = torch.from_numpy(gold["gqa_bf16_local_logits_sampled"])               # a fixed sample of the vocabulary
    got = lg[..., torch.from_numpy(gold["gqa_local_logits_cols"]).to(DEV)]
    assert _cos(got, ref) >= 0.999 and _rel(got, ref) <= 5e-2, (_cos(got, ref), _rel(got, ref))
    agree = float((lg.float().argmax(-1).cpu() == ref_argmax).float().mean())
    print(f"forward_local argmax agreement with the reference: {agree:.3f}")
    assert agree >= 0.9


def test_cfg3_shape_wrapped_ring_vs_reference_eager_on_gpu():
    """BASELINE cfg 3's shape class (SURVEY.md §8d): 7B widths (n_embd 4096, 32 heads x 128, intermediate 11008,
    depth 1024 / 16 heads / ff 4224, vocab 152064), B = 64, KV ring capacity 2048 pre-filled AND wrapped, 2 of the 32
    layers -- against the oracle restatement executed on the same GPU in bf16 (the ATen calls of the reference eager).
    Tolerance: rel 2e-2 of the tensor scale / cosine >= 0.999."""
    B, KV = 64, 2048
    cfg = L.LMConfig(n_layer=2, context=KV, block_size=4096)
    m = GPT(_product_config(cfg), device=DEV, dtype=BF).eval()
    w = {k: v.detach() for k, v in m.state_dict().items()}
    gs = L.GPTStream(w, cfg, B)
    g = torch.Generator(device=DEV).manual_seed(3)
    start = KV + 37                                    # wrapped: every step attends the full (cap - 1)-key window
    m.use_cuda_graphs = True
    with m.streaming(B):
        st = m._state
        for l in range(cfg.n_layer):
            st.kv[l].normal_(generator=g)
            gs.rings[l].cache.copy_(st.kv[l])
            gs.rings[l].end_offset = start
        gs.offset = start
        st.offset.fill_(start); st.pos_host[:] = start
        for step in range(3):
            seq = torch.randint(0, 2048, (B, 9, 1), device=DEV, generator=g)
            seq[:, 0] = torch.randint(0, 128256, (B, 1), device=DEV, generator=g)
            with torch.no_grad():
                r_out, r_tl = gs.forward_global(seq)
            out, tl = m.forward_global(seq)
            assert _cos(out, r_out) >= 0.999 and _rel(out, r_out) <= 2e-2, (step, _cos(out, r_out), _rel(out, r_out))
            assert _cos(tl, r_tl) >= 0.999 and _rel(tl, r_tl) <= 2e-2, (step, _cos(tl, r_tl), _rel(tl, r_tl))
            toks = r_tl.float().argmax(-1)                       # teacher forcing with the reference's tokens
            gs.start_depth()
            with m.codecformer.streaming(B):
                prev = toks[:, :, None]
                for k in range(cfg.dep_q):
                    with torch.no_grad():
                        r_lg = gs.forward_codecformer(k, prev, r_out)
                    lg = m.forward_codecformer(k, prev, r_out)
                    assert _cos(lg, r_lg) >= 0.999 and _rel(lg, r_lg) <= 2e-2, (step, k, _cos(lg, r_lg), _rel(lg, r_lg))
                    prev = r_lg.float().argmax(-1)
            for l in range(cfg.n_layer):                          # the appended K/V rows (bf16 RoPE arithmetic as eager)
                slot = (start + step) % KV
                a, b_ = st.kv[l][:, :, :, slot], gs.rings[l].cache[:, :, :, slot]
                assert _rel(a, b_) <= 2e-2


@pytest.mark.parametrize("B,split", [(4, False), (64, False), (64, True), (37, True)])
def test_attention_full_window_2047_keys_vs_sdpa(B, split):
    """ring_decode_attention at head 128, capacity 2048, wrapped: vs SDPA over exactly the keys RingKVCache.complete
    leaves attendable (MHA and a GQA grouping).  `split`: the persistent key-split form (taken when rows x heads exceed
    the resident CTAs) -- must agree with the one-CTA-per-job form to bf16 rounding and be run-to-run deterministic;
    streams at different fill levels (few keys, partially filled ring, wrapped) exercise empty key chunks."""
    lib, st_ = _lib.lib(), ops._stream()
    hs, cap = 128, 2048
    g = torch.Generator().manual_seed(9)
    for nh, nkv in ((8, 8), (16, 4)):
        kv = torch.randn(2, B, nkv, cap, hs, generator=g).to(BF).to(DEV)
        q = torch.randn(B, nh, hs, generator=g).to(BF).to(DEV)
        pos_b = torch.full((B,), cap + 100, dtype=torch.int64)  # the query's own key sits at slot pos % cap
        if B > 8:
            pos_b[1], pos_b[2], pos_b[3], pos_b[4] = 0, 5, 40, 1000
        offset = pos_b.to(DEV)
        out = torch.empty(B, nh * hs, dtype=BF, device=DEV)
        ws = torch.zeros(lib.rstnet_lm_attention_split_workspace(B, nh, hs), dtype=torch.uint8, device=DEV) if split else None
        outs = []
        for rep in range(2 if split else 1):
            out.zero_()
            _lib.check(lib.rstnet_lm_ring_decode_attention_bf16(q.data_ptr(), kv.data_ptr(), offset.data_ptr(), 1, out.data_ptr(), B, B,
                                                                nh, nkv, hs, cap, cap, ws.data_ptr() if split else None, st_))
            outs.append(out.clone())
        if split:
            assert torch.equal(outs[0], outs[1]), "key-split attention must be deterministic (and its counters self-resetting)"
            assert int(ws[:B * nh * 4].view(torch.int32).abs().sum()) == 0
        slots = torch.arange(cap, device=DEV)
        k_, v_ = kv[0].float(), kv[1].float()
        rep = nh // nkv
        k_, v_ = k_.repeat_interleave(rep, 1), v_.repeat_interleave(rep, 1)
        mask = torch.zeros(B, 1, 1, cap, dtype=torch.bool, device=DEV)
        for b in range(B):
            pos = int(pos_b[b])
            if pos >= cap - 1:
                mask[b, 0, 0] = slots != (pos + 1) % cap        # labelled end_offset -> masked (the ring quirk)
            else:
                mask[b, 0, 0] = slots <= pos
        ref = F.scaled_dot_product_attention(q.float()[:, :, None], k_, v_, attn_mask=mask, scale=1.0 / hs ** 0.5)[:, :, 0]
        err = (out.float().view(B, nh, hs) - ref).abs().max().item()
        assert err <= 1.5e-2, (nh, nkv, err)


def test_per_stream_reset_and_state_swap(small_lm):
    """reset_streaming(streams=[i]) restarts row i only (SURVEY.md §8f-1 admission): row i then reproduces a fresh
    stream bit for bit while the other rows continue undisturbed; get/set_streaming_state swap whole scopes."""
    m, w, cfg = small_lm
    g = torch.Generator().manual_seed(21)
    seqs = [torch.randint(0, 2048, (3, 9, 1), generator=g).to(DEV) for _ in range(10)]
    m.use_cuda_graphs = True
    with m.streaming(3):                                  # uninterrupted run
        base = [m.forward_step(s, use_sampling=False) for s in seqs]
    with m.streaming(3):
        for t in range(4):
            m.forward_step(seqs[t], use_sampling=False)
        m.reset_streaming(streams=[1])
        got = []
        for t in range(4, 10):
            # row 1 is a NEW stream fed the inputs a fresh stream would see from its first frame; rows 0, 2 continue
            s = seqs[t].clone()
            s[1] = seqs[t - 4][1]
            got.append(m.forward_step(s, use_sampling=False))
        saved = m.get_streaming_state()
    for i, t in enumerate(range(4, 10)):
        assert torch.equal(got[i][0], base[t][0]) and torch.equal(got[i][2], base[t][2]), "other rows must be undisturbed"
        assert torch.equal(got[i][1], base[t - 4][1]), "the reset row must reproduce a fresh stream"
    assert m._state is None
    m.set_streaming_state(saved)                            # resume the saved scope
    nxt = m.forward_step(seqs[0], use_sampling=False)
    assert nxt.shape == (3, 9)
    m.set_streaming_state({"": None})
    with pytest.raises(RuntimeError):
        m.set_streaming_state({})


def test_block_size_and_bad_ids_fail_loudly(small_lm):
    """Positions beyond block_size raise on the host before the launch (cos.index_select would raise upstream); ids
    outside an embedding table poison the row and set the device error flag (nn.Embedding would raise)."""
    m, w, cfg = small_lm
    m.use_cuda_graphs = False
    seq = torch.randint(0, 2048, (3, 9, 1)).to(DEV)
    with m.streaming(3):
        m._state.offset.fill_(cfg.block_size - 1); m._state.pos_host[:] = cfg.block_size - 1
        m.forward_global(seq)
        with pytest.raises(IndexError):
            m.forward_global(seq)
    with m.streaming(3):
        bad = seq.clone(); bad[1, 3, 0] = cfg.audio_card + 5
        out, _ = m.forward_global(bad)
        assert torch.isnan(out[1].float()).all() and not torch.isnan(out[0].float()).any()
        with pytest.raises(IndexError):
            m.check_device_errors()
        m.check_device_errors()                               # cleared


def test_sampling_big_k_and_full_multinomial():
    """top_k > 64 (moshi's default is 250) and top_k == 0 with sampling (plain multinomial, utils/sampling.py:97-101)."""
    lib, st_ = _lib.lib(), ops._stream()
    g = torch.Generator().manual_seed(2)
    rows, V = 64, 2050
    logits = (torch.randn(rows, V, generator=g) * 2).to(BF)
    logits[5, :] = 0.5                                          # all equal: the support is ids 0..k-1
    ld = logits.to(DEV).contiguous()
    out = torch.zeros(rows, dtype=torch.int64, device=DEV)
    for k in (100, 250, 1000):
        seen = torch.zeros(rows, V, dtype=torch.bool)
        for seed in range(40):
            _lib.check(lib.rstnet_lm_sample_bf16(ld.data_ptr(), rows, V, 2048, k, 1.0, seed, None, out.data_ptr(), 1, st_))
            seen[torch.arange(rows), out.cpu()] = True
        lf = logits.float().clone(); lf[:, 2048:] = -float("inf")
        kth = lf.topk(k, dim=-1).values[:, -1:]
        assert not (seen & (lf < kth)).any(), k                 # nothing outside the top-k (ties included)
        assert int(seen[5].nonzero().max()) < k
        assert seen.sum(1).float().mean() > 10                  # it does sample
    # distribution of the full multinomial against softmax(l / temp)
    ps = torch.tensor([5.0, 2.0, 12.0, 6.0, 8.0, 1.0, 0.5, 4.0])
    lg = torch.log(ps).to(BF).repeat(8000, 1).contiguous().to(DEV)
    o2 = torch.zeros(8000, dtype=torch.int64, device=DEV)
    for temp in (1.0, 0.5):
        _lib.check(lib.rstnet_lm_sample_bf16(lg.data_ptr(), 8000, 8, 8, -1, temp, 3, None, o2.data_ptr(), 1, st_))
        cnt = torch.bincount(o2.cpu(), minlength=8).float()
        target = torch.softmax(torch.log(ps).to(BF).float() / temp, -1)
        assert (cnt / cnt.sum() - target).abs().max().item() < 2e-2, temp
    # a big-k pick over a 152k vocabulary with n_valid < V (candidate list path)
    big = (torch.randn(8, 151936, generator=g)).to(BF).to(DEV).contiguous()
    o3 = torch.zeros(8, dtype=torch.int64, device=DEV)
    _lib.check(lib.rstnet_lm_sample_bf16(big.data_ptr(), 8, 151936, 151936, 250, 0.7, 1, None, o3.data_ptr(), 1, st_))
    kth = big.float().topk(250, dim=-1).values[:, -1]
    assert (big.float().gather(1, o3[:, None])[:, 0] >= kth).all()


def test_default_config_gating_hidden_not_multiple_of_64():
    """The reference's default Config has codecformer_dim_feedforward 1024 -> hidden 682 (modules/gating.py:40-43): the
    depth GEMMs run on zero-padded weights; checked against the oracle."""
    import dataclasses
    cfg = dataclasses.replace(L.SMALL, codecformer_dim=256, codecformer_heads=4, codecformer_dim_feedforward=1023)   # hidden 682
    assert cfg.ff_hidden == 682
    w32 = L.synthetic_weights(cfg, seed=3, dtype=torch.float32, std=0.05)
    m = GPT(_product_config(cfg)); m.load_state_dict(w32, strict=True); m = m.to(DEV, BF).eval()
    w = {k: v.to(BF) for k, v in w32.items()}
    gs = L.GPTStream(w, cfg, 2)
    seq = torch.randint(0, 2048, (2, 9, 1))
    with torch.no_grad():
        r_out, r_tl = gs.forward_global(seq)
        gs.start_depth()
        r_lg = gs.forward_codecformer(0, r_tl.float().argmax(-1)[:, :, None], r_out)
    with m.streaming(2):
        out, tl = m.forward_global(seq.to(DEV))
        with m.codecformer.streaming(2):
            lg = m.forward_codecformer(0, r_tl.float().argmax(-1)[:, :, None].to(DEV), out)
    assert _cos(lg, r_lg) >= 0.999 and _rel(lg, r_lg) <= 5e-2


def test_depth_frame_kernel_vs_multi_launch_path(small_lm):
    """csrc/lm_depth_frame.cu (the 8 depth steps + sampling of a frame in one persistent kernel) against the
    one-launch-per-op path it replaces and against the oracle: same logits to bf16 rounding, same greedy tokens away from
    near-ties; teacher-forced single steps and the whole sampled frame."""
    m, w, cfg = small_lm
    g = torch.Generator().manual_seed(31)
    seqs = [torch.randint(0, 2048, (5, 9, 1), generator=g).to(DEV) for _ in range(3)]

    def run(flag):
        m.use_depth_frame_kernel = flag
        m._packed = None
        outs = []
        with m.streaming(5):
            assert (m._state.df is not None) == flag
            for s in seqs:
                out, tl = m.forward_global(s)
                prev = tl.float().argmax(-1)[:, :, None]
                lgs = []
                with m.codecformer.streaming(5):
                    for k in range(cfg.dep_q):
                        lg = m.forward_codecformer(k, prev, out)
                        lgs.append(lg[:, 0, 0])
                        prev = seqs[0][:, k + 1:k + 2, :]                 # teacher forcing with fixed ids
                outs.append(torch.stack(lgs, 1))
            toks = [m.forward_step(s, use_sampling=False) for s in seqs]
            samp = m.forward_step(seqs[0], use_sampling=True, top_k=30, temp=0.8, audio_valid=2048)
        return outs, toks, samp

    try:
        new, new_t, new_s = run(True)
        old, old_t, old_s = run(False)
    finally:
        m.use_depth_frame_kernel = False
        m._packed = None
    for a, b in zip(new, old):
        assert _cos(a, b) >= 0.9995 and _rel(a, b) <= 3e-2, (_cos(a, b), _rel(a, b))
    agree = sum(int((a == b).sum()) for a, b in zip(new_t, old_t)) / sum(a.numel() for a in new_t)
    print(f"depth frame kernel vs multi-launch path: greedy token agreement {agree:.3f}")
    assert agree >= 0.85                       # closed loop inside a frame: one near-tie flip changes the later codebooks
    assert int(new_s[:, 1:].max()) < 2048 and int(new_s.min()) >= 0
    # against the oracle (bf16), teacher-forced
    gs = L.GPTStream(w, cfg, 5)
    with torch.no_grad():
        r_out, r_tl = gs.forward_global(seqs[0].cpu())
        gs.start_depth()
        prev = r_tl.float().argmax(-1)[:, :, None]
        ref = []
        for k in range(cfg.dep_q):
            ref.append(gs.forward_codecformer(k, prev, r_out)[:, 0, 0])
            prev = seqs[0][:, k + 1:k + 2, :].cpu()
    ref = torch.stack(ref, 1)
    assert _cos(new[0], ref) >= 0.999 and _rel(new[0], ref) <= 5e-2, (_cos(new[0], ref), _rel(new[0], ref))
    m.check_device_errors()


def test_in_kernel_finalize_tail_opt_in():
    """RSTNET_SKINNY_TAIL=1 (read once per process): split-K partials are reduced, normalised / gated inside the GEMM
    kernel by the CTAs of each tile instead of by a finalize launch.  Same arithmetic, so the GEMM, whole-frame and 7B-width
    tests must pass unchanged in a child process with the switch on."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, RSTNET_SKINNY_TAIL="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider",
                        "-k", "skinny_gemm_vs_torch or forward_step_matches_stepwise_api or cfg3_shape_wrapped_ring"],
                       env=env, capture_output=True, text=True, timeout=900, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-1000:]
    assert " passed" in r.stdout
