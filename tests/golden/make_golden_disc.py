"""Golden vectors for the MelGAN multi-scale discriminator (SURVEY.md section 8f rank 3) from the UNMODIFIED reference
(`src/models/discriminators.py:57-78`) in fp64:

    AERO_REFERENCE=<checkout of the reference> python tests/golden/make_golden_disc.py

Weights are a recipe (tests/util.disc_recipe_state: 16.9 M parameters would be 68 MB) plus a digest; stored are sub-sampled feature maps of every layer of every scale for a seeded waveform, and the
gradients (256 samples + rms per parameter, and the full input gradient) of  loss = sum over all feature maps of mean(feature * R)
with seeded cotangents R."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from util import SEED, disc_recipe_state, sample_indices, weights_digest, white_noise  # noqa: E402


def build_reference():
    import importlib
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "src" or k.startswith("src.")}
    path_saved = list(sys.path)
    sys.path[:] = [os.environ["AERO_REFERENCE"]] + [p for p in sys.path if os.path.abspath(p or ".") != os.path.dirname(os.path.dirname(HERE))]
    try:
        mod = importlib.import_module("src.models.discriminators")
    finally:
        sys.path[:] = path_saved
        for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    torch.manual_seed(SEED)
    return mod.Discriminator(3, 16, 4, 4)


def cot(shape, i, j):
    return white_noise(shape, seed=SEED + 1000 + 10 * i + j)


def main():
    torch.set_num_threads(os.cpu_count())
    ref = build_reference()
    ref.load_state_dict(disc_recipe_state(ref.state_dict()))
    digest = weights_digest(ref.state_dict())
    ref = ref.double()
    B, L = 2, 8192
    x = white_noise((B, 1, L), seed=SEED + 3).double().requires_grad_(True)
    feats = ref(x)
    loss = 0.0
    blob = {"digest": np.float64(digest), "B": B, "L": L, "torch": torch.__version__}
    for i, scale in enumerate(feats):
        for j, f in enumerate(scale):
            loss = loss + (f * cot(tuple(f.shape), i, j).double()).mean()
            flat = f.detach().reshape(-1)
            idx = sample_indices(flat.numel(), 2048, seed=17)
            blob[f"f_shape/{i}/{j}"] = np.array(f.shape)
            blob[f"f_idx/{i}/{j}"] = idx.numpy().astype(np.int32)
            blob[f"f_val/{i}/{j}"] = flat[idx].float().numpy()
    loss.backward()
    blob["loss"] = np.float64(float(loss))
    blob["dx"] = x.grad.float().numpy()
    for k, p in ref.named_parameters():
        gflat = p.grad.reshape(-1)
        idx = sample_indices(gflat.numel(), 256, seed=13)
        blob["g_idx/" + k] = idx.numpy().astype(np.int32)
        blob["g_val/" + k] = gflat[idx].float().numpy()
        blob["g_rms/" + k] = np.float64(gflat.pow(2).mean().sqrt())
    np.savez_compressed(os.path.join(HERE, "disc_melgan.npz"), **blob)
    print("disc golden: loss", float(loss), "features", [[tuple(f.shape) for f in s] for s in feats][0])


if __name__ == "__main__":
    main()
