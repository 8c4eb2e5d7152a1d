"""Shared helpers for the parity tests (CPU-only code; no kernels)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 2036          # reference conf/main_config.yaml:32


def trained_like_(state, seed=SEED):
    """Deterministically perturb a freshly initialised state_dict so that parameters which sit
    at (near-)identity after init -- LayerScale 1e-3, BatchNorm running stats 0/1, norm affine
    1/0, LocalState decay x0.01 / bias -2 (reference modules.py:88-90,138) -- take "trained"
    magnitudes.  At init they would hide bugs in exactly the kernels that use them.
    Pure function of (key order, shapes, seed): applied identically to the reference model
    (when generating golden vectors) and to aero_b200.Aero (when checking against them)."""
    g = torch.Generator().manual_seed(seed + 1)
    out = {}
    for k, v in state.items():
        v = v.clone()
        r = torch.randn(v.shape, generator=g) if v.dtype.is_floating_point else None
        if k.endswith("conv2.3.scale"):
            v = 0.25 + 0.15 * torch.tanh(r)
        elif k.endswith("running_mean"):
            v = 0.2 * r
        elif k.endswith("running_var"):
            v = 0.6 + 0.8 * torch.sigmoid(r)
        elif ".norm1." in k or ".norm2." in k or re_norm(k):
            v = (1.0 + 0.2 * r) if k.endswith("weight") else 0.1 * r
        elif "query_decay.weight" in k:
            v = v * 60.0
        elif "query_decay.bias" in k:
            v = -1.0 + r
        out[k] = v.to(state[k].dtype)
    return out


def re_norm(k):
    # GroupNorm inside DConv ('conv1.1', 'conv2.1') and BatchNorm affine inside FTB ('conv1.1', 'conv1d.1', 'conv2.1')
    return k.rsplit(".", 1)[0].endswith(("conv1.1", "conv2.1", "conv1d.1")) and k.endswith(("weight", "bias"))


def weights_digest(state):
    """Order-dependent fp64 checksum of a state_dict (to prove both sides hold the same weights)."""
    acc, i = 0.0, 0
    for k, v in state.items():
        if v.dtype.is_floating_point:
            i += 1
            acc += float(v.double().sum()) * (1 + (i % 7)) + float(v.double().abs().sum())
    return acc


def white_noise(shape, seed=SEED):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def sample_indices(numel, n=4096, seed=7):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def import_reference(ref_root=os.environ.get("AERO_REFERENCE", "")):
    """Import the unmodified reference package from a checkout of it at `ref_root` (default: the AERO_REFERENCE
    environment variable).  Only the golden-vector generators under tests/golden/ use it; returns None without one."""
    import importlib
    if not ref_root or not os.path.isdir(ref_root):
        return None
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "src" or k.startswith("src.")}
    path_saved = list(sys.path)
    sys.path[:] = [ref_root] + [p for p in sys.path if os.path.abspath(p or ".") != ROOT]
    try:
        mods = {n: importlib.import_module("src.models." + n) for n in ("aero", "spec", "modules", "stft_loss")}
    finally:
        sys.path[:] = path_saved
        for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    assert all(ref_root in m.__file__ for m in mods.values())
    return mods


def disc_recipe_state(state, seed=SEED):
    """Deterministic weights for the MelGAN discriminator (reference and aero_b200 share the state_dict keys): weight_v ~
    N(0, 0.02^2) as the reference's `weights_init`, weight_g = ||v|| moved off its init by up to +-30 %, biases N(0, 0.05^2).
    Pure function of (key order, shapes, seed), like `trained_like_`."""
    g = torch.Generator().manual_seed(seed + 5)
    out = {}
    for k, v in state.items():
        if k.endswith("weight_v"):
            out[k] = 0.02 * torch.randn(v.shape, generator=g)
    for k, v in state.items():
        r = torch.randn(v.shape, generator=g)
        if k.endswith("weight_g"):
            vv = out[k[:-1] + "v"]
            out[k] = vv.flatten(1).norm(dim=1).view(v.shape) * (1.0 + 0.3 * torch.tanh(r))
        elif k.endswith("bias"):
            out[k] = 0.05 * r
    return {k: out[k].to(state[k].dtype) for k in state}
