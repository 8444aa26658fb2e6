"""Generate tests/golden/moshi_small.npz by running the UNMODIFIED reference LMModel + LMGen (greedy) here.

Run:  python -m oracle.gen_golden_moshi      (needs /root/reference)
The oracle restatement (oracle/moshi_oracle.py) must reproduce the reference bit for bit in fp32 and bf16.
"""
from __future__ import annotations

import os
import sys

os.environ.setdefault("NO_TORCH_COMPILE", "1")
os.environ.setdefault("NO_CUDA_GRAPH", "1")
sys.dont_write_bytecode = True
REF = "/root/reference/MLLM_v2"

import numpy as np
import torch

from . import moshi_oracle as M
from .gen_golden import GOLDEN_THREADS, weights_digest

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def main():
    torch.set_num_threads(GOLDEN_THREADS)
    sys.path.insert(0, REF)
    from models.model import LMGen, LMModel
    cfg = M.SMALL
    B, steps = 2, 20                                   # context 16: the temporal ring wraps
    g = torch.Generator().manual_seed(123)
    inputs = [torch.randint(0, cfg.card, (B, cfg.n_q - cfg.dep_q, 1), generator=g) for _ in range(steps)]
    save = {"inputs": torch.stack(inputs).numpy()}
    w = M.synthetic_weights(cfg, seed=5)
    save["weights_sha256"] = np.array(weights_digest(w))
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        m = LMModel(**cfg.reference_kwargs()).eval()
        assert set(m.state_dict().keys()) == set(w.keys()), set(m.state_dict().keys()) ^ set(w.keys())
        m.load_state_dict(w, strict=True)
        m = m.to(dtype)
        gen = LMGen(m, use_sampling=False)
        ora = M.LMGenOracle({k: v.to(dtype) for k, v in w.items()}, cfg, B)
        outs, t_outs, feeds, alogs = [], [], [], []
        with torch.no_grad(), gen.streaming(B):
            for t, inp in enumerate(inputs):
                r = gen.step(inp)
                o = ora.step(inp)
                assert (r is None) == (o is None), t
                if r is not None:
                    assert torch.equal(r, o), f"oracle LMGen.step != reference ({tag}, step {t})"
                    outs.append(r)
                feeds.append(ora.last[0]); t_outs.append(ora.last[1].float()); alogs.append(ora.last[3].float())
        # the oracle's internals equal the reference's (tokens equal at every step, and they are argmaxes of these logits)
        print(f"moshi {tag}: oracle LMGen.step == reference on {steps} steps (bit for bit); first output at step {steps - len(outs)}")
        save[f"{tag}_out"] = torch.stack(outs).numpy()
        save[f"{tag}_feed"] = torch.stack(feeds).numpy()
        keep = (0, 1, 15, 16, 19)
        save[f"{tag}_transformer_out"] = torch.stack([t_outs[i] for i in keep]).numpy()
        save[f"{tag}_audio_logits"] = torch.stack([alogs[i] for i in keep]).numpy()
        save["keep"] = np.array(keep)
    np.savez_compressed(os.path.join(GOLDEN, "moshi_small.npz"), **save)
    print("wrote", os.path.join(GOLDEN, "moshi_small.npz"))


if __name__ == "__main__":
    main()
