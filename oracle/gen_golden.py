"""Generate tests/golden/*.npz by running the UNMODIFIED reference in the build container.

Run:  python -m oracle.gen_golden          (needs /root/reference; not available on the GPU box)

For every fixture the reference (imported from /root/reference/MLLM_v2, fp32, CPU,
NO_TORCH_COMPILE=1) and the oracle restatement (oracle/mimi_oracle.py) are run on the same seeded
synthetic weights/inputs; the script asserts they agree (bit-for-bit where the same ATen ops are
used) and stores the REFERENCE outputs.  The weights themselves are not stored: they are
re-derived from the seed by oracle/mimi_spec.synthetic_weights (same torch build on both boxes);
a checksum of the weights is stored to catch RNG drift.
"""
from __future__ import annotations

import hashlib
import os
import sys

os.environ.setdefault("NO_TORCH_COMPILE", "1")
os.environ.setdefault("NO_CUDA_GRAPH", "1")
sys.dont_write_bytecode = True
REF = "/root/reference/MLLM_v2"

import numpy as np
import torch

from . import mimi_oracle as O
from . import mimi_spec as S

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# intra-op threads of every fixture run: torch's CPU float32 convolutions split their sums by thread count, so the
# tests that compare the oracle with the fixtures bit for bit (or to 1e-6) use the same count
GOLDEN_THREADS = 8


def weights_digest(w) -> str:
    h = hashlib.sha256()
    for k in sorted(w):
        h.update(k.encode())
        h.update(w[k].contiguous().numpy().tobytes())
    return h.hexdigest()


def build_reference_codec(w):
    sys.path.insert(0, REF)
    from tools.tokenizer.MimiCodec.model.models.MimiCodec import MimiCodec  # noqa
    m = MimiCodec(encoder_rates=[8, 6, 5, 4], codebook_size=2048, codebook_dim=256, rvq_layers=8).eval()
    sd = m.state_dict()
    assert set(sd.keys()) == set(w.keys()), (set(sd.keys()) ^ set(w.keys()))
    for k in sd:
        assert tuple(sd[k].shape) == tuple(w[k].shape), k
    m.load_state_dict(w, strict=True)
    return m


def build_reference_mimimodel(w):
    """moshi MimiModel assembled as loaders.get_mimi minus load_model (moshi/models/loaders.py:108-139)."""
    sys.path.insert(0, REF)
    from moshi.models import loaders
    from moshi.models.compression import MimiModel
    from moshi.modules import SEANetEncoder, SEANetDecoder, transformer
    from moshi.quantization import SplitResidualVectorQuantizer
    enc = SEANetEncoder(**loaders._seanet_kwargs)
    dec = SEANetDecoder(**loaders._seanet_kwargs)
    et = transformer.ProjectedTransformer(device="cpu", **loaders._transformer_kwargs)
    dt = transformer.ProjectedTransformer(device="cpu", **loaders._transformer_kwargs)
    q = SplitResidualVectorQuantizer(**loaders._quantizer_kwargs)
    model = MimiModel(enc, dec, q, channels=1, sample_rate=loaders.SAMPLE_RATE, frame_rate=loaders.FRAME_RATE,
                      encoder_frame_rate=loaders.SAMPLE_RATE / enc.hop_length, causal=True,
                      resample_method="conv", encoder_transformer=et, decoder_transformer=dt).eval()
    sd = model.state_dict()
    # loaders._quantizer_kwargs builds 32 codebooks and keeps the first 8 (set_num_codebooks(8));
    # levels >= 8 never run, so only they may be missing from the 8-level synthetic state_dict.
    missing = set(sd.keys()) - set(w.keys())
    assert all(".vq.layers." in k and int(k.split(".vq.layers.")[1].split(".")[0]) >= 7 for k in missing), missing
    model.load_state_dict({k: w[k] for k in sd if k in w}, strict=False)
    model.set_num_codebooks(8)
    return model


def main():
    torch.set_num_threads(GOLDEN_THREADS)
    os.makedirs(GOLDEN, exist_ok=True)
    cfg = S.OFFICIAL
    w = S.synthetic_weights(cfg, seed=41, codebook_scale=S.CODEBOOK_SCALE)
    digest = weights_digest(w)
    ref = build_reference_codec(w)

    # ---------------- cfg 1: 1 s clip, B=1, encode -> decode (BASELINE.json configs[0])
    x = S.synthetic_audio(1, 24000, seed=0)
    with torch.no_grad():
        z_enc = ref.encoder(x)
        z_tr = ref.encoder_transformer(z_enc)[0]
        z_lat = ref.downsample(z_tr)
        codes = ref.encode(x)
        q = ref.quantizer.decode(codes)
        up = ref.upsample(q)
        d_tr = ref.decoder_transformer(up)[0]
        wav = ref.decode(codes)
        # oracle must reproduce the reference
        o_codes = O.encode(x, w, cfg)
        o_wav = O.decode(codes, w, cfg)
        o_lat = O.encode_latent(x, w, cfg)
    assert codes.shape == (1, 8, 13) and wav.shape == (1, 1, 24960), (codes.shape, wav.shape)
    assert torch.equal(o_codes, codes), "oracle codes != reference codes"
    print("cfg1: oracle==reference codes; latent max|d| =", (o_lat - z_lat).abs().max().item(),
          " wav max|d| =", (o_wav - wav).abs().max().item())
    assert (o_lat - z_lat).abs().max().item() <= 1e-5
    assert (o_wav - wav).abs().max().item() <= 1e-5
    margins = O.rvq_margins(z_lat, w, cfg)
    print("cfg1: min rel. RVQ margin per level:", [f"{v:.2e}" for v in margins.min(dim=1).values.tolist()])
    np.savez_compressed(
        os.path.join(GOLDEN, "mimi_cfg1.npz"),
        weights_sha256=np.array(digest), audio_seed=np.array(0), weight_seed=np.array(41),
        audio_head=x[0, 0, :64].numpy(),
        z_enc=z_enc.numpy(), z_tr=z_tr.numpy(), z_lat=z_lat.numpy(), codes=codes.numpy(),
        q=q.numpy(), up=up.numpy(), d_tr=d_tr.numpy(), wav=wav.numpy(), margins=margins.numpy(),
    )

    # ---------------- batch of 3 ragged-length clips (edge cases: L not a multiple of the frame)
    for L in (1920, 4000, 1):
        xb = S.synthetic_audio(2, L, seed=100 + L)
        with torch.no_grad():
            cb = ref.encode(xb)
            wb = ref.decode(cb)
            assert torch.equal(O.encode(xb, w, cfg), cb)
            assert (O.decode(cb, w, cfg) - wb).abs().max().item() <= 1e-5
        np.savez_compressed(os.path.join(GOLDEN, f"mimi_len{L}.npz"), weights_sha256=np.array(digest),
                            audio_seed=np.array(100 + L), codes=cb.numpy(), wav=wb.numpy(),
                            z_lat=ref.downsample(ref.encoder_transformer(ref.encoder(xb))[0]).detach().numpy())
        print(f"len {L}: codes {tuple(cb.shape)} wav {tuple(wb.shape)} ok")

    # ---------------- streaming: moshi MimiModel, 6 frames of 1920 samples, B=2
    mm = build_reference_mimimodel(w)
    xs = S.synthetic_audio(2, 1920 * 6, seed=7)
    sc = O.StreamingCodec(w, 2, cfg)
    s_codes, s_wav = [], []
    with torch.no_grad(), mm.streaming(2):
        for i in range(6):
            chunk = xs[..., i * 1920:(i + 1) * 1920]
            c = mm.encode(chunk)
            y = mm.decode(c)
            oc = sc.encode(chunk)
            oy = sc.decode(c)
            assert torch.equal(oc, c), f"streaming oracle codes differ at frame {i}"
            assert (oy - y).abs().max().item() <= 1e-5, (i, (oy - y).abs().max().item())
            s_codes.append(c)
            s_wav.append(y)
    s_codes = torch.cat(s_codes, dim=-1)
    s_wav = torch.cat(s_wav, dim=-1)
    with torch.no_grad():
        b_codes = mm.encode(xs)
        b_wav = mm.decode(b_codes)
    print("streaming vs batch (reference property): codes equal:", torch.equal(b_codes, s_codes),
          " wav max|d|:", (b_wav - s_wav).abs().max().item())
    np.savez_compressed(os.path.join(GOLDEN, "mimi_stream6.npz"), weights_sha256=np.array(digest),
                        audio_seed=np.array(7), codes=s_codes.numpy(), wav=s_wav.numpy(),
                        batch_codes=b_codes.numpy())
    print("golden fixtures written to", GOLDEN)


if __name__ == "__main__":
    main()
