"""Pin the oracle: both forms of oracle/aero_oracle.py against the golden vectors produced by the
unmodified reference (tests/golden/make_golden.py), whole forwards and single blocks.  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from util import SEED, rel_l2, trained_like_, weights_digest, white_noise

from aero_b200 import Aero, aero_kwargs
from oracle import aero_oracle as O

CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "c*.npz")))
FAST = {"c2_4-16_hop256_ragged", "c5_8-24_nonpow2", "c6_4-16_hop64_short"}
# the 10-s stereo case costs ~1 minute and several GB of attention scores per oracle forward: the oracle is pinned on it
# only when asked for (AERO_SLOW_TESTS=1); its 4-s sibling c8 exercises the same windowing / key-tile regime every run
SLOW = {"c9_11-44_stereo_10s"}


def build_case(golden_dir, case):
    g = np.load(os.path.join(golden_dir, case + ".npz"))
    kw = aero_kwargs(str(g["exp"]))
    torch.manual_seed(SEED)
    model = Aero(**kw).eval()
    model.load_state_dict(trained_like_(model.state_dict()))
    assert weights_digest(model.state_dict()) == pytest.approx(float(g["digest"]), rel=1e-12), \
        "weights rebuilt from the seed recipe differ from the ones the golden vectors were made with"
    mix = white_noise((int(g["B"]), kw["in_channels"], int(g["L"])))
    return g, model, mix


def check_against_golden(g, out, zc, zlr, taps, tol):
    if "out" in g.files:
        assert out.shape == g["out"].shape
        assert rel_l2(out, g["out"]) < tol
    else:                       # full-shape cases: the waveform is committed as a 65536-position sample + its rms
        assert tuple(out.shape) == tuple(int(v) for v in g["out_shape"])
        flat = out.reshape(-1)
        assert rel_l2(flat[torch.from_numpy(g["out_idx"].astype(np.int64))], g["out_val"]) < tol
        assert abs(float(flat.double().pow(2).mean().sqrt()) / float(g["out_rms"]) - 1) < 1e-4
    zc_r = torch.view_as_real(zc).reshape(-1)[torch.from_numpy(g["spec_idx"].astype(np.int64))]
    assert rel_l2(zc_r, g["spec_val"]) < tol
    zl_r = torch.view_as_real(zlr).reshape(-1)[torch.from_numpy(g["lrspec_idx"].astype(np.int64))]
    assert rel_l2(zl_r, g["lrspec_val"]) < tol
    for key in g.files:
        if key.startswith("act_idx/"):
            tag = key.split("/", 1)[1]
            got = taps[tag].reshape(-1)[torch.from_numpy(g[key].astype(np.int64))]
            assert rel_l2(got, g["act_val/" + tag]) < tol, tag


@pytest.mark.parametrize("case", CASES)
def test_oracle_library_form_matches_reference_golden(golden_dir, case):
    if case in SLOW and not os.environ.get("AERO_SLOW_TESTS"):
        pytest.skip("slow (set AERO_SLOW_TESTS=1)")
    g, model, mix = build_case(golden_dir, case)
    taps = {}
    with torch.no_grad():
        out, zc, zlr = O.aero_forward(model.state_dict(), model.geom, mix, True, True, explicit=False, taps=taps)
    check_against_golden(g, out, zc, zlr, taps, tol=2e-5)


@pytest.mark.parametrize("case", [c for c in CASES if c in FAST])
def test_oracle_explicit_form_matches_reference_golden(golden_dir, case):
    g, model, mix = build_case(golden_dir, case)
    taps = {}
    with torch.no_grad():
        out, zc, zlr = O.aero_forward(model.state_dict(), model.geom, mix, True, True, explicit=True, taps=taps)
    check_against_golden(g, out, zc, zlr, taps, tol=1e-4)


def test_oracle_fp64_explicit_vs_library():
    """The two forms agree to fp64 round-off: the restatement is the same function."""
    kw = aero_kwargs("aero_4-16_512_256")
    torch.manual_seed(SEED)
    model = Aero(**kw).eval()
    sd = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in trained_like_(model.state_dict()).items()}
    mix = white_noise((1, 1, 4000)).double()
    with torch.no_grad():
        a = O.aero_forward(sd, model.geom, mix, explicit=False)
        b = O.aero_forward(sd, model.geom, mix, explicit=True)
    assert rel_l2(a, b) < 1e-10


def test_stft_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "stft_cases.npz"))
    i = 0
    while f"{i}/params" in g.files:
        n_fft, hop, win, L, *lead = [int(v) for v in g[f"{i}/params"]]
        x = white_noise((*lead, L), seed=SEED + i)
        for explicit in (False, True):
            z = O.stft(x, n_fft, hop, win, explicit)
            zr = torch.view_as_real(z).reshape(-1)[torch.from_numpy(g[f"{i}/z_idx"].astype(np.int64))]
            assert rel_l2(zr, g[f"{i}/z_val"]) < 1e-5
            y = O.istft(z, hop, win, explicit)
            assert y.shape == g[f"{i}/y"].shape
            assert rel_l2(y, g[f"{i}/y"]) < 1e-5
        i += 1
    assert i >= 6


def test_oracle_matches_reference_blocks_golden(golden_dir):
    """One BLSTM and one LocalState block, in both forms, and the whole forward against the reference's own modules
    (tests/golden/make_golden.py::make_blocks): seeded samples of each output and its rms."""
    g = np.load(os.path.join(golden_dir, "ref_blocks.npz"))
    kw = aero_kwargs("aero_4-16_512_128")
    torch.manual_seed(SEED)
    mine = Aero(**kw).eval()
    mine.load_state_dict(trained_like_(mine.state_dict()))
    sd = mine.state_dict()
    assert list(sd) == list(g["keys"])
    assert weights_digest(sd) == pytest.approx(float(g["digest"]), rel=1e-12)

    def check(tag, a):
        assert tuple(a.shape) == tuple(int(v) for v in g[tag + "/shape"])
        flat = a.reshape(-1)
        assert rel_l2(flat[torch.from_numpy(g[tag + "/idx"].astype(np.int64))], g[tag + "/val"]) < 1e-5, tag
        assert abs(float(flat.double().pow(2).mean().sqrt()) / float(g[tag + "/rms"]) - 1) < 1e-5, tag
    h = white_noise((6, 96, 251), seed=5)
    with torch.no_grad():
        for explicit in (False, True):
            check("lstm", O.blstm(h, sd, "encoder.3.dconv.layers.0.lstm", explicit=explicit))
            check("time_attn", O.local_state(h, sd, "encoder.3.dconv.layers.0.time_attn", explicit=explicit))
        check("forward", O.aero_forward(sd, mine.geom, white_noise((1, 1, 5000))))


def _mrstft_inputs(g, i):
    B, L, so = (int(v) for v in g[f"{i}/params"])
    eps = float(g[f"{i}/eps"])
    y = white_noise((B, L), seed=SEED + 100 + so)
    x = y + eps * white_noise((B, L), seed=SEED + 200 + so)
    if i == 1:
        x[:, :2000] = 0.0
    return x, y


def test_mrstft_loss_oracle_matches_reference_golden(golden_dir):
    """SURVEY.md section 8f rank 2: the loss restatement against values produced by the reference's own module
    (tests/golden/make_golden.py::make_mrstft)."""
    g = np.load(os.path.join(golden_dir, "mrstft_cases.npz"))
    i = 0
    while f"{i}/params" in g.files:
        x, y = _mrstft_inputs(g, i)
        sc, mag = O.mrstft_loss(x, y)
        assert abs(float(sc) - float(g[f"{i}/sc"])) <= 1e-6 * abs(float(g[f"{i}/sc"])) + 1e-9
        assert abs(float(mag) - float(g[f"{i}/mag"])) <= 1e-6 * abs(float(g[f"{i}/mag"])) + 1e-9
        i += 1
    assert i >= 2
