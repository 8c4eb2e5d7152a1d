"""Golden vectors for the TRAINING path: parameter gradients of the UNMODIFIED reference generator under autograd.

    AERO_REFERENCE=<checkout of the reference> python tests/golden/make_golden_train.py

For every case: seed, build the reference ``src.models.aero.Aero``, apply ``tests.util.trained_like_``, switch to
``train()`` (batch-statistics BatchNorm in the FTB blocks), run ``out = model(mix)`` on seeded white noise, back-propagate
the scalar ``loss = sum(out * R) / out.numel()`` (model promoted to fp64: see below) with R a seeded noise tensor (so the gradient of the waveform is R / numel: a
dense, well-conditioned cotangent), and store, per parameter, the gradient's rms and 256 seeded samples, plus the training-mode
output (sub-sampled) and the BatchNorm running buffers after the step.  The consumer rebuilds inputs and weights from the same
recipes.  Tests read only the committed .npz files."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from util import ROOT, SEED, import_reference, sample_indices, trained_like_, weights_digest, white_noise  # noqa: E402

sys.path.insert(0, ROOT)
from aero_b200.config import aero_kwargs  # noqa: E402

CASES = [  # name, experiment, batch, low-rate length
    ("t1_4-16_hop256", "aero_4-16_512_256", 2, 6000),      # T = 95 (< 200: single LSTM window)
    ("t2_4-16_hop64", "aero_4-16_512_64", 2, 3600),        # T = 226 (> 200: three overlapping LSTM windows, zero-padded tail)
    ("t3_11-44_stereo", "aero_11-44_512_64", 1, 2400),     # stereo in / out (C_in = C_out = 2)
]


def cotangent(shape, seed):
    return white_noise(shape, seed=seed + 77)


def main():
    ref = import_reference()
    assert ref is not None, "set AERO_REFERENCE to a checkout of the reference"
    torch.set_num_threads(os.cpu_count())
    for name, exp, B, L in CASES:
        kw = aero_kwargs(exp)
        torch.manual_seed(SEED)
        model = ref["aero"].Aero(**kw)
        model.load_state_dict(trained_like_(model.state_dict()))
        digest = weights_digest(model.state_dict())
        # the reference runs in fp64 here (same fp32 weights and inputs, promoted): several gradients are small differences of
        # large terms (BatchNorm / GroupNorm backward over a few hundred samples), and an fp32 reference would carry ~1e-2
        # relative rounding noise of its own on exactly those parameters
        model = model.double().train()
        mix = white_noise((B, kw["in_channels"], L)).double()
        out = model(mix)
        R = cotangent(tuple(out.shape), SEED).double()
        loss = (out * R).sum() / out.numel()
        loss.backward()
        blob = {"digest": np.float64(digest), "B": B, "L": L, "exp": exp, "torch": torch.__version__, "loss": np.float64(float(loss)),
                "out_shape": np.array(out.shape)}
        flat = out.detach().reshape(-1)
        oi = sample_indices(flat.numel(), 16384, seed=11)
        blob["out_idx"], blob["out_val"] = oi.numpy().astype(np.int32), flat[oi].float().numpy()
        for k, p in model.named_parameters():
            gflat = p.grad.reshape(-1)
            idx = sample_indices(gflat.numel(), 256, seed=13)
            blob["g_idx/" + k] = idx.numpy().astype(np.int32)
            blob["g_val/" + k] = gflat[idx].float().numpy()
            blob["g_rms/" + k] = np.float64(gflat.double().pow(2).mean().sqrt())
        for k, b in model.named_buffers():
            if k.endswith(("running_mean", "running_var")):
                blob["buf/" + k] = b.detach().float().numpy()
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
        print(name, "out", tuple(out.shape), "loss", float(loss), "params", sum(1 for _ in model.named_parameters()))


if __name__ == "__main__":
    main()
