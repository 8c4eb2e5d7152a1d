"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

Run with a checkout of the reference:

    AERO_REFERENCE=<checkout of the reference> python tests/golden/make_golden.py [case ...]

For every case it (1) seeds torch, builds the reference ``src.models.aero.Aero`` from the
experiment kwargs, (2) applies ``tests.util.trained_like_`` to its state_dict, (3) runs
``Aero.forward(mix, return_spec=True, return_lr_spec=True)`` on seeded white noise under
``no_grad`` in fp32 on CPU, capturing block outputs with forward hooks, and (4) stores the
waveform, sub-sampled spectra / block activations and a digest of the weights in
``<case>.npz``.  Inputs and weights are *recipes* (seed + rule), not blobs: the consumer
rebuilds them with the same torch build.  A second file, ``stft_cases.npz``, holds
``spectro`` / ``ispectro`` outputs (reference src/models/spec.py) for the window/hop pairs the
path uses, ``mrstft_cases.npz`` the multi-resolution STFT loss and ``ref_blocks.npz`` single reference blocks
(``make_blocks``).  Naming cases regenerates only those.

Tests read only the committed .npz files.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from util import ROOT, SEED, import_reference, sample_indices, trained_like_, weights_digest, white_noise  # noqa: E402

sys.path.insert(0, ROOT)
from aero_b200.config import aero_kwargs  # noqa: E402

# name, experiment, batch, length (low-rate samples)
CASES = [
    ("c1_4-16_hop64_b2", "aero_4-16_512_64", 2, 8000),          # BASELINE configs[0]/[1] shape (2 s)
    ("c2_4-16_hop256_ragged", "aero_4-16_512_256", 1, 7777),    # ragged length -> right zero-pad; T<200: no LSTM windows
    ("c3_12-48_hop128", "aero_12-48_512_128", 1, 12000),        # BASELINE configs[2] geometry (1 s)
    ("c4_11-44_stereo", "aero_11-44_512_64", 1, 5500),          # stereo, in/out_channels=2 (0.5 s)
    ("c5_8-24_nonpow2", "aero_8-24_512_64", 1, 4000),           # hop 21 / win 170 -> hop 63 / win 510
    ("c6_4-16_hop64_short", "aero_4-16_512_64", 3, 1600),       # T=101 (<200): single LSTM window, B=3
    # full-shape cases (round 2): the waveform is stored sub-sampled (65536 seeded positions + its rms), not whole
    ("c7_12-48_hop128_b2_2s", "aero_12-48_512_128", 2, 24000),  # BASELINE configs[2] clip shape: T=751, 8 LSTM windows
    ("c8_11-44_stereo_4s", "aero_11-44_512_64", 1, 44100),      # T=2757: 28 LSTM windows, 44 attention key tiles
    ("c9_11-44_stereo_10s", "aero_11-44_512_64", 1, 110250),    # BASELINE configs[4] clip shape: T=6892 (69 windows, 108 key tiles)
]
SUBSAMPLED = {"c7_12-48_hop128_b2_2s", "c8_11-44_stereo_4s", "c9_11-44_stereo_10s"}

STFT_CASES = [  # n_fft, hop, win, batch-shape, length
    (512, 16, 128, (2, 1), 8000),
    (512, 64, 512, (1, 1), 32000),
    (512, 21, 170, (1, 2), 4011),
    (512, 63, 510, (1, 1), 12033),
    (2048, 512, 2048, (1,), 32000),
    (512, 128, 512, (3,), 1000),
]


def main():
    ref = import_reference()
    assert ref is not None, "set AERO_REFERENCE to a checkout of the reference"
    torch.set_num_threads(os.cpu_count())
    only = set(sys.argv[1:])
    for name, exp, B, L in CASES:
        if only and name not in only:
            continue
        kw = aero_kwargs(exp)
        torch.manual_seed(SEED)
        model = ref["aero"].Aero(**kw).eval()
        model.load_state_dict(trained_like_(model.state_dict()))
        digest = weights_digest(model.state_dict())
        mix = white_noise((B, kw["in_channels"], L))
        acts = {}

        def hook(tag):
            def fn(mod, inp, out):
                acts[tag] = out.detach()
            return fn
        handles = []
        for i, enc in enumerate(model.encoder):
            handles.append(enc.register_forward_hook(hook(f"encoder.{i}")))
            handles.append(enc.dconv.register_forward_hook(hook(f"encoder.{i}.dconv")))
            handles.append(enc.freq_attn_block.register_forward_hook(hook(f"encoder.{i}.ftb")))
        for j, dec in enumerate(model.decoder):
            handles.append(dec.register_forward_hook(hook(f"decoder.{j}")))
        with torch.no_grad():
            out, zc, zlr = model(mix, return_spec=True, return_lr_spec=True)
        for h in handles:
            h.remove()
        blob = {"digest": np.float64(digest), "B": B, "L": L, "exp": exp, "torch": torch.__version__}
        if name in SUBSAMPLED:
            flat = out.reshape(-1)
            oi = sample_indices(flat.numel(), 65536, seed=11)
            blob.update({"out_shape": np.array(out.shape), "out_idx": oi.numpy().astype(np.int32), "out_val": flat[oi].numpy(),
                         "out_rms": np.float64(flat.double().pow(2).mean().sqrt())})
        else:
            blob["out"] = out.numpy()
        zc_r, zlr_r = torch.view_as_real(zc).reshape(-1), torch.view_as_real(zlr).reshape(-1)
        blob["spec_idx"] = sample_indices(zc_r.numel(), 8192).numpy().astype(np.int32)
        blob["spec_val"] = zc_r[blob["spec_idx"].astype(np.int64)].numpy()
        blob["lrspec_idx"] = sample_indices(zlr_r.numel(), 8192).numpy().astype(np.int32)
        blob["lrspec_val"] = zlr_r[blob["lrspec_idx"].astype(np.int64)].numpy()
        for tag, a in acts.items():
            flat = a.reshape(-1)
            idx = sample_indices(flat.numel(), 2048)
            blob["act_idx/" + tag] = idx.numpy().astype(np.int32)
            blob["act_val/" + tag] = flat[idx].numpy()
            blob["act_rms/" + tag] = np.float64(flat.double().pow(2).mean().sqrt())
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
        print(name, "out", tuple(out.shape), "rms", float(out.pow(2).mean().sqrt()), "digest", digest)

    if only:
        return
    blob = {}
    for i, (n_fft, hop, win, lead, L) in enumerate(STFT_CASES):
        x = white_noise((*lead, L), seed=SEED + i)
        z = ref["spec"].spectro(x, n_fft, hop, win_length=win)
        y = ref["spec"].ispectro(z, hop, win_length=win)
        blob[f"{i}/params"] = np.array([n_fft, hop, win, L] + list(lead))
        zr = torch.view_as_real(z).reshape(-1)
        idx = sample_indices(zr.numel(), 32768)
        blob[f"{i}/z_idx"] = idx.numpy().astype(np.int32)
        blob[f"{i}/z_val"] = zr[idx].numpy()
        blob[f"{i}/y"] = y.numpy()
        print("stft case", i, tuple(z.shape), tuple(y.shape))
    np.savez_compressed(os.path.join(HERE, "stft_cases.npz"), **blob)
    make_mrstft(ref)
    make_blocks(ref)


def make_blocks(ref):
    """One BLSTM and one LocalState block of the reference (encoder 3, DConv layer 0) on a seeded activation, and the whole
    forward on a short seeded clip, for aero_4-16_512_128: 4096 seeded samples + the rms of each output, and the state_dict's
    key order and weight digest (tests/test_oracle.py::test_oracle_matches_reference_blocks_golden)."""
    kw = aero_kwargs("aero_4-16_512_128")
    torch.manual_seed(SEED)
    model = ref["aero"].Aero(**kw).eval()
    model.load_state_dict(trained_like_(model.state_dict()))
    sd = model.state_dict()
    h = white_noise((6, 96, 251), seed=5)
    layer = model.encoder[3].dconv.layers[0]
    with torch.no_grad():
        outs = {"lstm": layer["lstm"](h), "time_attn": layer["time_attn"](h), "forward": model(white_noise((1, 1, 5000)))}
    blob = {"digest": np.float64(weights_digest(sd)), "keys": np.array(list(sd))}
    for tag, a in outs.items():
        flat = a.reshape(-1)
        idx = sample_indices(flat.numel(), 4096)
        blob[tag + "/shape"] = np.array(a.shape)
        blob[tag + "/idx"] = idx.numpy().astype(np.int32)
        blob[tag + "/val"] = flat[idx].numpy()
        blob[tag + "/rms"] = np.float64(flat.double().pow(2).mean().sqrt())
        print("block", tag, tuple(a.shape))
    np.savez_compressed(os.path.join(HERE, "ref_blocks.npz"), **blob)


MRSTFT_CASES = [  # batch, length, seed offset, scale of the estimate's perturbation
    (2, 32000, 0, 0.3),
    (3, 9000, 1, 1.0),
]


def make_mrstft(ref):
    """Multi-resolution STFT loss (reference src/models/stft_loss.py:96-138) on seeded signals.  The reference's `stft()`
    (`:22`) calls torch.stft without return_complex and raises on torch >= 2: the module is used unmodified except that
    its `torch.stft` is wrapped to return the real view it expects (the one-line shim of SURVEY.md appendix C)."""
    mod = ref["stft_loss"]

    class _TorchShim:
        def __getattr__(self, name):
            return getattr(torch, name)

        @staticmethod
        def stft(x, fft_size, hop_size, win_length, window):
            return torch.view_as_real(torch.stft(x, fft_size, hop_size, win_length, window, return_complex=True))
    mod.torch = _TorchShim()
    loss = mod.MultiResolutionSTFTLoss()
    blob = {}
    for i, (B, L, so, eps) in enumerate(MRSTFT_CASES):
        y = white_noise((B, L), seed=SEED + 100 + so)
        x = y + eps * white_noise((B, L), seed=SEED + 200 + so)
        if i == 1:
            x[:, :2000] = 0.0                                   # exercise the 1e-7 clamp
        sc, mag = loss(x, y)
        blob[f"{i}/params"] = np.array([B, L, so], dtype=np.int64)
        blob[f"{i}/eps"] = np.array(eps)
        blob[f"{i}/sc"], blob[f"{i}/mag"] = np.array(float(sc)), np.array(float(mag))
        print("mrstft case", i, float(sc), float(mag))
    np.savez_compressed(os.path.join(HERE, "mrstft_cases.npz"), **blob)


if __name__ == "__main__":
    main()
