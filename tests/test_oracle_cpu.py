"""CPU suite (-m "not gpu"): the oracle against the golden vectors produced by the unmodified
reference (oracle/gen_golden.py), host-side logic, and the C-ABI export list."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import mimi_oracle as O
from oracle import mimi_spec as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(autouse=True)
def golden_threads():
    """Run the oracle with the thread count the fixtures were made with: its float32 convolutions round by it."""
    from oracle.gen_golden import GOLDEN_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def test_oracle_cfg1_matches_reference_golden(golden_dir, official_weights):
    g = np.load(os.path.join(golden_dir, "mimi_cfg1.npz"))
    x = S.synthetic_audio(1, 24000, seed=int(g["audio_seed"]))
    assert np.array_equal(x[0, 0, :64].numpy(), g["audio_head"])
    with torch.no_grad():
        lat = O.encode_latent(x, official_weights)
        codes = O.rvq_encode(lat, official_weights)
        wav = O.decode(torch.from_numpy(g["codes"]), official_weights)
    assert codes.shape == (1, 8, 13)
    assert np.array_equal(codes.numpy(), g["codes"])                      # bit-exact indices
    assert np.abs(lat.numpy() - g["z_lat"]).max() <= 1e-6
    assert wav.shape == (1, 1, 24960)
    assert np.abs(wav.numpy() - g["wav"]).max() <= 1e-6


@pytest.mark.parametrize("L", [1, 1920, 4000])
def test_oracle_ragged_lengths(golden_dir, official_weights, L):
    g = np.load(os.path.join(golden_dir, f"mimi_len{L}.npz"))
    x = S.synthetic_audio(2, L, seed=int(g["audio_seed"]))
    with torch.no_grad():
        codes = O.encode(x, official_weights)
        wav = O.decode(codes, official_weights)
    assert np.array_equal(codes.numpy(), g["codes"])
    assert np.abs(wav.numpy() - g["wav"]).max() <= 1e-6
    assert codes.shape[-1] == -(-L // 1920) and wav.shape[-1] == codes.shape[-1] * 1920


def test_oracle_streaming_matches_reference_golden(golden_dir, official_weights):
    g = np.load(os.path.join(golden_dir, "mimi_stream6.npz"))
    x = S.synthetic_audio(2, 1920 * 6, seed=int(g["audio_seed"]))
    sc = O.StreamingCodec(official_weights, 2)
    cs, ws = [], []
    with torch.no_grad():
        for i in range(6):
            c = sc.encode(x[..., i * 1920:(i + 1) * 1920])
            cs.append(c)
            ws.append(sc.decode(c))
    codes, wav = torch.cat(cs, -1), torch.cat(ws, -1)
    assert np.array_equal(codes.numpy(), g["codes"])
    assert np.abs(wav.numpy() - g["wav"]).max() <= 1e-6
    # the reference's own property (moshi/modules/seanet_test.py): streaming == non-streaming
    assert np.array_equal(g["codes"], g["batch_codes"])


def test_oracle_empty_latent():
    w = S.synthetic_weights(S.TINY, seed=1)
    z = torch.zeros(2, S.TINY.dimension, 0)
    assert O.rvq_encode(z, w, S.TINY).shape == (2, S.TINY.n_q, 0)


def test_rvq_first_minimum_tie_break():
    """argmin keeps the first minimum (core_vq.py:183): duplicate centroids -> lower index."""
    emb = torch.randn(16, 8)
    emb[9] = emb[3]
    x = emb[3:4] + 1e-3
    assert int(O.quantize_nearest(x, emb)[0]) == 3


def test_tiny_config_streaming_equals_batch():
    cfg = S.TINY
    w = S.synthetic_weights(cfg, seed=3)
    x = S.synthetic_audio(2, cfg.frame_size * 5, seed=5)
    with torch.no_grad():
        ref = O.encode(x, w, cfg)
        sc = O.StreamingCodec(w, 2, cfg)
        got = torch.cat([sc.encode(x[..., i * cfg.frame_size:(i + 1) * cfg.frame_size]) for i in range(5)], -1)
    assert torch.equal(ref, got)


# ------------------------------------------------------------------ product host logic (no GPU)
def test_product_state_dict_keys_match_oracle_spec():
    from rstnet_b200.codec import MimiCodec
    m = MimiCodec(encoder_rates=[8, 6, 5, 4], codebook_size=2048, codebook_dim=256, rvq_layers=8)
    sd = m.state_dict()
    spec = {n: s for n, s, _ in S.param_spec(S.OFFICIAL)}
    spec.update({n: s for n, s in S.buffer_spec(S.OFFICIAL)})
    assert set(sd) == set(spec)
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), k
    assert m.frame_size == 1920 and m.hop_length == 960 and m.resample_stride == 2


def test_product_loads_reference_style_checkpoint_and_old_names(official_weights):
    from rstnet_b200.codec import MimiCodec
    m = MimiCodec(encoder_rates=[8, 6, 5, 4], codebook_size=2048, codebook_dim=256, rvq_layers=8)
    sd = dict(official_weights)
    p = "quantizer.rvq_first.vq.layers.0._codebook"
    sd[f"{p}.embed_sum"] = sd.pop(f"{p}.embedding_sum")   # old Kyutai names (core_vq.py:126-140)
    sd[f"{p}.cluster_size"] = sd.pop(f"{p}.cluster_usage")
    m.load_state_dict(sd, strict=True)
    assert torch.equal(m.state_dict()[f"{p}.embedding_sum"], official_weights[f"{p}.embedding_sum"])


def test_product_refuses_cpu():
    from rstnet_b200.codec import MimiCodec
    from rstnet_b200._lib import RstnetError
    m = MimiCodec(encoder_rates=[8, 6, 5, 4], codebook_size=2048, codebook_dim=256, rvq_layers=8)
    with pytest.raises(RstnetError):
        m.encode(torch.zeros(1, 1, 1920))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rstnet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f


# ------------------------------------------------------------------ C ABI
def _header_symbols():
    hdr = open(os.path.join(ROOT, "include", "rstnet_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(rstnet_[a-z0-9_]+)\s*\(", hdr)))


def test_cabi_library_exports_every_declared_symbol():
    from rstnet_b200 import _lib, build
    build.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    syms = _header_symbols()
    assert syms, "no symbols parsed from include/rstnet_b200.h"
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/rstnet_b200.h but not exported"
    assert sorted(_lib.SYMBOLS) == syms
    assert _lib.lib().rstnet_version() >= 100


def test_btk_adapter_only_transposes(monkeypatch):
    """MimiCodecBTK (AudioCodec-tree token layout [B, T, K]) must be a pure layout adapter around MimiCodec."""
    from rstnet_b200 import codec as C
    seen = {}

    def fake_encode(self, audio):
        return torch.arange(2 * 8 * 5).view(2, 8, 5)

    def fake_decode(self, codes):
        seen["codes"] = codes
        return torch.zeros(codes.shape[0], 1, 1920 * codes.shape[2])

    monkeypatch.setattr(C.MimiCodec, "encode", fake_encode)
    monkeypatch.setattr(C.MimiCodec, "decode", fake_decode)
    m = C.MimiCodecBTK(encoder_rates=[8, 6, 5, 4], codebook_size=2048, codebook_dim=256, rvq_layers=8)
    btk = m.encode(torch.zeros(2, 1, 9600))
    assert btk.shape == (2, 5, 8) and torch.equal(btk.transpose(1, 2), torch.arange(2 * 8 * 5).view(2, 8, 5))
    wav = m.decode(btk)
    assert seen["codes"].shape == (2, 8, 5) and torch.equal(seen["codes"], torch.arange(2 * 8 * 5).view(2, 8, 5))
    assert wav.shape == (2, 1, 9600)
