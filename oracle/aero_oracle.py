"""CPU oracle for the AERO generator forward  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` leg may import this module.  Nothing under ``aero_b200/`` does.

What it is: a functional restatement (state_dict in, tensors out; NCHW like the reference) of
the reference's algorithm, in plain torch-CPU ops, fp32 or fp64.  Every function cites the
reference lines it restates.  The arithmetic of the reference lives in PyTorch (pinned
``torch==1.12.1`` in reference ``requirements.txt:10``; 2.11.0 here), so each library op the
reference calls is available in two forms:

  * ``explicit=False`` -- the same library call the reference makes (``torch.stft``,
    ``torch.lstm``, ``einsum`` + ``softmax``): performance-equivalent to the reference, used
    as the timed CPU baseline ("port");
  * ``explicit=True``  -- the published algorithm written out (framing + rFFT, LSTM cell
    recurrence, attention with the decay penalty in closed form, GroupNorm by moments):
    an independent statement the CUDA kernels are compared against.

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4, 8c), so parity is pinned
against the reference *itself*: ``tests/golden/make_golden.py`` imports the reference
unmodified, runs ``Aero.forward`` and single blocks on seeded inputs and commits the outputs;
``tests/test_oracle.py`` checks both forms of this oracle against those vectors.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------- STFT / iSTFT


def hann_padded(win_length, n_fft, like):
    """Periodic Hann computed in fp32 then cast (reference spec.py:15 ``th.hann_window(win).to(x)``),
    centred zero-pad to n_fft as torch.stft does."""
    w = torch.hann_window(win_length).to(like)
    left = (n_fft - win_length) // 2
    return F.pad(w, (left, n_fft - win_length - left))


def stft(x, n_fft, hop, win_length, explicit=False):
    """reference spec.py:9-22 ``spectro``: normalized, centred (reflect), one-sided.
    x [..., L] real -> [..., n_fft/2+1, 1+L//hop] complex."""
    *lead, length = x.shape
    x2 = x.reshape(-1, length)
    if not explicit:
        z = torch.stft(x2, n_fft, hop, window=torch.hann_window(win_length).to(x2), win_length=win_length,
                       normalized=True, center=True, return_complex=True, pad_mode="reflect")
    else:
        w = hann_padded(win_length, n_fft, x2)
        xp = F.pad(x2[:, None], (n_fft // 2, n_fft // 2), mode="reflect")[:, 0]
        frames = xp.unfold(-1, n_fft, hop)                      # [N, T, n_fft]
        z = torch.fft.rfft(frames * w, dim=-1) * (n_fft ** -0.5)
        z = z.transpose(1, 2)
    return z.reshape(*lead, z.shape[-2], z.shape[-1])


def istft(z, hop, win_length, explicit=False):
    """reference spec.py:25-38 ``ispectro``: n_fft = 2*(bins-1); output length hop*(T-1)."""
    *lead, bins, frames = z.shape
    n_fft = 2 * bins - 2
    z2 = z.reshape(-1, bins, frames)
    if not explicit:
        x = torch.istft(z2, n_fft, hop, window=torch.hann_window(win_length).to(z2.real),
                        win_length=win_length, normalized=True, length=None, center=True)
    else:
        w = hann_padded(win_length, n_fft, z2.real)
        fr = torch.fft.irfft(z2.transpose(1, 2) * (n_fft ** 0.5), n=n_fft, dim=-1) * w   # [N, T, n_fft]
        total = n_fft + hop * (frames - 1)
        y = z2.real.new_zeros(z2.shape[0], total)
        env = z2.real.new_zeros(total)
        for t in range(frames):
            y[:, t * hop:t * hop + n_fft] += fr[:, t]
            env[t * hop:t * hop + n_fft] += w * w
        lo, hi = n_fft // 2, total - n_fft // 2
        x = y[:, lo:hi] / env[lo:hi]
    return x.reshape(*lead, x.shape[-1])


# --------------------------------------------------------------------------- small pieces


def group_norm(x, groups, weight, bias, eps=1e-5, explicit=False):
    if not explicit:
        return F.group_norm(x, groups, weight, bias, eps)
    n, c = x.shape[:2]
    xg = x.reshape(n, groups, -1)
    mu = xg.mean(-1, keepdim=True)
    var = ((xg - mu) ** 2).mean(-1, keepdim=True)
    y = ((xg - mu) / torch.sqrt(var + eps)).reshape(x.shape)
    shape = [1, c] + [1] * (x.dim() - 2)
    return y * weight.view(shape) + bias.view(shape)


BN_TRAIN = False      # tests of the training path set this: BatchNorm then uses batch statistics (nn.BatchNorm in train mode)


def batch_norm_eval(x, sd, prefix, eps=1e-5):
    """BatchNorm of the FTB blocks, reference modules.py:287,293,300: running statistics (eval mode), or -- when the module
    flag BN_TRAIN is set -- the statistics of the batch (biased variance), as nn.BatchNorm normalises in train mode."""
    shape = [1, -1] + [1] * (x.dim() - 2)
    if BN_TRAIN:
        dims = [0] + list(range(2, x.dim()))
        mu = x.mean(dims, keepdim=True)
        var = ((x - mu) ** 2).mean(dims, keepdim=True)
        return (x - mu) * torch.rsqrt(var + eps) * sd[prefix + ".weight"].view(shape) + sd[prefix + ".bias"].view(shape)
    inv = torch.rsqrt(sd[prefix + ".running_var"] + eps) * sd[prefix + ".weight"]
    return (x - sd[prefix + ".running_mean"].view(shape)) * inv.view(shape) + sd[prefix + ".bias"].view(shape)


def snake(x, a):
    """reference snake.py:61-67 with ``a`` broadcast over the last axis."""
    return x + (1.0 / a) * torch.sin(x * a) ** 2


def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x * (2.0 ** -0.5)))


def glu(x, dim=1):
    a, b = x.chunk(2, dim)
    return a * torch.sigmoid(b)


# --------------------------------------------------------------------------- BLSTM


def _lstm_dir(x, w_ih, w_hh, b_ih, b_hh, reverse):
    """One direction of one LSTM layer, gate order i,f,g,o, zero initial state.  x [T, N, I]."""
    T, N, _ = x.shape
    H = w_hh.shape[1]
    gi = x @ w_ih.t() + (b_ih + b_hh)
    h = x.new_zeros(N, H)
    c = x.new_zeros(N, H)
    out = [None] * T
    order = range(T - 1, -1, -1) if reverse else range(T)
    for t in order:
        g = gi[t] + h @ w_hh.t()
        i, f, gg, o = g.chunk(4, -1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
        h = torch.sigmoid(o) * torch.tanh(c)
        out[t] = h
    return torch.stack(out)


def lstm_stack(x, sd, prefix, layers, explicit=False):
    """``nn.LSTM(bidirectional=True, num_layers=layers)`` on x [T, N, I] (reference modules.py:28,46)."""
    names = []
    for l in range(layers):
        for sfx in ("", "_reverse"):
            names += [f"{prefix}.weight_ih_l{l}{sfx}", f"{prefix}.weight_hh_l{l}{sfx}",
                      f"{prefix}.bias_ih_l{l}{sfx}", f"{prefix}.bias_hh_l{l}{sfx}"]
    if not explicit:
        H = sd[names[1]].shape[1]
        zeros = x.new_zeros(2 * layers, x.shape[1], H)
        out, _, _ = torch.lstm(x, (zeros, zeros), [sd[n] for n in names], True, layers, 0.0, BN_TRAIN, True, False)   # train flag: cuDNN needs it for backward; dropout is 0
        return out
    for l in range(layers):
        p = [sd[n] for n in names[8 * l:8 * l + 8]]
        x = torch.cat([_lstm_dir(x, *p[0:4], reverse=False), _lstm_dir(x, *p[4:8], reverse=True)], -1)
    return x


def blstm(x, sd, prefix, layers=2, max_steps=200, explicit=False):
    """reference modules.py:32-65 (+ ``unfold`` utils.py:22-35).  x [N, C, T] -> same, with skip."""
    N, C, T = x.shape
    y = x
    framed = max_steps is not None and T > max_steps
    if framed:
        width, stride = max_steps, max_steps // 2
        nframes = math.ceil(T / stride)
        xp = F.pad(x, (0, (nframes - 1) * stride + width - T))
        frames = xp.unfold(-1, width, stride)                   # [N, C, nframes, width]
        x = frames.permute(0, 2, 1, 3).reshape(-1, C, width)
    h = lstm_stack(x.permute(2, 0, 1), sd, prefix + ".lstm", layers, explicit)
    h = h @ sd[prefix + ".linear.weight"].t() + sd[prefix + ".linear.bias"]
    h = h.permute(1, 2, 0)
    if framed:
        fr = h.reshape(N, nframes, C, width)
        q = stride // 2
        keep = []
        for k in range(nframes):
            lo = 0 if k == 0 else q
            hi = width if k == nframes - 1 else width - q
            keep.append(fr[:, k, :, lo:hi])
        h = torch.cat(keep, -1)[..., :T]
    return h + y


# --------------------------------------------------------------------------- LocalState


def local_state(x, sd, prefix, heads=4, ndecay=4, explicit=False):
    """reference modules.py:94-127 (nfreqs=0).  x [N, C, T]."""
    N, C, T = x.shape

    def proj(name, inp=x):
        return F.conv1d(inp, sd[f"{prefix}.{name}.weight"], sd[f"{prefix}.{name}.bias"])

    q = proj("query").view(N, heads, -1, T)
    k = proj("key").view(N, heads, -1, T)
    v = proj("content").view(N, heads, -1, T)
    dq = torch.sigmoid(proj("query_decay").view(N, heads, ndecay, T)) / 2
    idx = torch.arange(T, dtype=x.dtype, device=x.device)
    dist = (idx[:, None] - idx[None, :]).abs()                    # [t(key), s(query)]
    if not explicit:
        dots = torch.einsum("bhct,bhcs->bhts", k, q) / k.shape[2] ** 0.5
        decays = torch.arange(1, ndecay + 1, dtype=x.dtype, device=x.device)
        kern = -decays.view(-1, 1, 1) * dist / ndecay ** 0.5
        dots = dots + torch.einsum("fts,bhfs->bhts", kern, dq)
        dots.masked_fill_(torch.eye(T, dtype=torch.bool, device=x.device), -100)
        w = torch.softmax(dots, dim=2)
        r = torch.einsum("bhts,bhct->bhcs", w, v)
    else:
        # closed form: the decay term is -|t-s| * slope[s], slope = sum_f f*dq_f / sqrt(ndecay)
        f = torch.arange(1, ndecay + 1, dtype=x.dtype, device=x.device).view(1, 1, -1, 1)
        slope = (f * dq).sum(2) / ndecay ** 0.5                   # [N, h, s]
        d = k.shape[2]
        r = torch.empty_like(v)
        for n in range(N):
            for hh in range(heads):
                s_ts = (k[n, hh].t() @ q[n, hh]) / d ** 0.5 - dist * slope[n, hh][None, :]
                s_ts.fill_diagonal_(-100.0)
                m = s_ts.max(0, keepdim=True).values
                e = torch.exp(s_ts - m)
                r[n, hh] = v[n, hh] @ (e / e.sum(0, keepdim=True))
    return x + proj("proj", r.reshape(N, C, T))


# --------------------------------------------------------------------------- blocks


def dconv(x, sd, prefix, depth, lstm, attn, explicit=False):
    """reference modules.py:221-249 with reshape=True, act_func='snake'.  x [B, C, F, T]."""
    B, C, Fr, T = x.shape
    x = x.permute(0, 2, 1, 3).reshape(-1, C, T)
    for d in range(depth):
        p = f"{prefix}.layers.{d}"
        skip = x
        w1 = sd[p + ".conv1.0.weight"]
        dil = 2 ** d
        h = F.conv1d(x, w1, sd[p + ".conv1.0.bias"], dilation=dil, padding=dil)
        h = group_norm(h, 1, sd[p + ".conv1.1.weight"], sd[p + ".conv1.1.bias"], explicit=explicit)
        hid = h.shape[1]
        h = snake(h.view(B, Fr, hid, T).permute(0, 2, 3, 1), sd[p + ".act.a"])
        h = h.permute(0, 3, 1, 2).reshape(-1, hid, T)
        if lstm:
            h = blstm(h, sd, p + ".lstm", explicit=explicit)
        if attn:
            h = local_state(h, sd, p + ".time_attn", explicit=explicit)
        u = F.conv1d(h, sd[p + ".conv2.0.weight"], sd[p + ".conv2.0.bias"])
        u = glu(group_norm(u, 1, sd[p + ".conv2.1.weight"], sd[p + ".conv2.1.bias"], explicit=explicit))
        x = skip + sd[p + ".conv2.3.scale"][:, None] * u
    return x.view(B, Fr, C, T).permute(0, 2, 1, 3)


def ftb(x, sd, prefix):
    """reference modules.py:304-325 (eval-mode BatchNorm).  x [B, C, F, T]."""
    B, C, D, T = x.shape
    r = torch.relu(batch_norm_eval(F.conv2d(x, sd[prefix + ".conv1.0.weight"], sd[prefix + ".conv1.0.bias"]),
                                   sd, prefix + ".conv1.1"))
    g = F.conv1d(r.reshape(B, -1, T), sd[prefix + ".conv1d.0.weight"], sd[prefix + ".conv1d.0.bias"], padding=4)
    g = torch.relu(batch_norm_eval(g, sd, prefix + ".conv1d.1")).reshape(B, C, 1, T)
    att = g * x
    att = (att.transpose(2, 3) @ sd[prefix + ".freq_fc.weight"].t()).transpose(2, 3)
    cat = torch.cat([att, x], 1)
    y = F.conv2d(cat, sd[prefix + ".conv2.0.weight"], sd[prefix + ".conv2.0.bias"])
    return torch.relu(batch_norm_eval(y, sd, prefix + ".conv2.1"))


def enc_layer(x, sd, g, kw, explicit=False, taps=None):
    """reference aero.py:108-135.  ``g`` is an aero_b200.model.LayerGeom-like object."""
    p = f"encoder.{g.index}"
    if g.index == 0:
        x = F.conv2d(x, sd[p + ".pre_conv.weight"], sd[p + ".pre_conv.bias"])
        if taps is not None:
            taps[p + ".pre_conv"] = x
    if g.ftb:
        x = ftb(x, sd, p + ".freq_attn_block")
        if taps is not None:
            taps[p + ".ftb"] = x
    x = F.conv2d(x, sd[p + ".conv.weight"], sd[p + ".conv.bias"], stride=(g.stride, 1), padding=(g.pad, 0))
    if g.norm:
        x = group_norm(x, kw["norm_groups"], sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], explicit=explicit)
    x = gelu(x)
    if taps is not None:
        taps[p + ".conv"] = x
    if g.dconv:
        x = dconv(x, sd, p + ".dconv", kw["dconv_depth"], g.lstm, g.attn, explicit)
        if taps is not None:
            taps[p + ".dconv"] = x
    x = F.conv2d(x, sd[p + ".rewrite.weight"], sd[p + ".rewrite.bias"])
    if g.norm:
        x = group_norm(x, kw["norm_groups"], sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], explicit=explicit)
    return glu(x)


def dec_layer(x, skip, sd, g, j, kw, last, explicit=False):
    """reference aero.py:189-215 (freq layer, no DConv)."""
    p = f"decoder.{j}"
    x = torch.cat([x, skip], 1)
    y = F.conv2d(x, sd[p + ".rewrite.weight"], sd[p + ".rewrite.bias"], padding=kw["context"])
    if g.norm:
        y = group_norm(y, kw["norm_groups"], sd[p + ".norm1.weight"], sd[p + ".norm1.bias"], explicit=explicit)
    y = glu(y)
    z = F.conv_transpose2d(y, sd[p + ".conv_tr.weight"], sd[p + ".conv_tr.bias"], stride=(g.stride, 1))
    if g.norm:   # statistics over the *uncropped* tensor, aero.py:206-209
        z = group_norm(z, kw["norm_groups"], sd[p + ".norm2.weight"], sd[p + ".norm2.bias"], explicit=explicit)
    if g.pad:
        z = z[..., g.pad:-g.pad, :]
    return z if last else gelu(z)


# --------------------------------------------------------------------------- whole model


def spec(x, geom, scale=False, explicit=False):
    """reference aero.py:409-421."""
    hop = geom.hop_in
    if x.shape[-1] % hop:
        x = F.pad(x, (0, hop - x.shape[-1] % hop))
    hl, win = hop, geom.win_in
    if scale:
        hl, win = int(hl * geom.scale), int(win * geom.scale)
    return stft(x, geom.nfft, hl, win, explicit)[..., :-1, :]


def ispec(z, geom, explicit=False):
    """reference aero.py:423-428."""
    z = F.pad(z, (0, 0, 0, 1))
    return istft(z, geom.hop_out, geom.win_out, explicit)


def aero_forward(sd, geom, mix, return_spec=False, return_lr_spec=False, explicit=False, taps=None):
    """reference aero.py:446-523.  ``sd``: state_dict (CPU tensors of mix.dtype); ``geom``:
    aero_b200.model.AeroGeometry (pure shape arithmetic, no kernels)."""
    kw = geom.kw
    length = mix.shape[-1]
    z = spec(mix, geom, explicit=explicit)
    B, C, Fq, T = z.shape
    x = torch.view_as_real(z).permute(0, 1, 4, 2, 3).reshape(B, 2 * C, Fq, T)
    mean = x.mean(dim=(1, 2, 3), keepdim=True)
    std = x.std(dim=(1, 2, 3), keepdim=True)
    x = (x - mean) / (1e-5 + std)
    if taps is not None:
        taps["input_norm"] = x
    saved = []
    for g in geom.layers:
        x = enc_layer(x, sd, g, kw, explicit, taps)
        if taps is not None:
            taps[f"encoder.{g.index}"] = x          # as seen by a forward hook: before the embedding add
        if g.index == 0 and kw["freq_emb"]:
            emb = sd["freq_emb.embedding.weight"] * kw["emb_scale"]          # [F, C]
            x = x + kw["freq_emb"] * emb.t()[None, :, :, None]
        saved.append(x)
    x = torch.zeros_like(x)
    for j, g in enumerate(reversed(geom.layers)):
        x = dec_layer(x, saved.pop(), sd, g, j, kw, last=(g.index == 0), explicit=explicit)
        if taps is not None:
            taps[f"decoder.{j}"] = x
    x = x.view(B, kw["out_channels"], -1, Fq, T)
    x = x * std[:, None] + mean[:, None]
    zc = torch.view_as_complex(x.permute(0, 1, 3, 4, 2).contiguous())
    out = ispec(zc, geom, explicit)[..., :int(length * geom.scale)]
    if return_spec:
        return (out, zc, z) if return_lr_spec else (out, zc)
    return out


# ------------------------------------------------------------------------------------------------
# Multi-resolution STFT loss (SURVEY.md section 8f rank 2), forward value
def mrstft_loss(x, y, fft_sizes=(1024, 2048, 512), hop_sizes=(120, 240, 50), win_lengths=(600, 1200, 240),
                factor_sc=0.1, factor_mag=0.1):
    """reference src/models/stft_loss.py:96-138 (`MultiResolutionSTFTLoss.forward`): per resolution, magnitudes
    sqrt(clamp(re^2 + im^2, 1e-7)) of the un-normalised centred STFT (`:11-27`), spectral convergence
    ||mag_y - mag_x||_F / ||mag_y||_F (`:30-45`) and L1 of the log magnitudes (`:48-63`); both averaged over the
    resolutions and scaled.  x = estimate, y = target, [B, T]."""
    sc, mag = 0.0, 0.0
    for n_fft, hop, win in zip(fft_sizes, hop_sizes, win_lengths):
        w = torch.hann_window(win, dtype=x.dtype, device=x.device)
        mx = torch.stft(x, n_fft, hop, win, w, return_complex=True).abs().square().clamp_min(1e-7).sqrt()
        my = torch.stft(y, n_fft, hop, win, w, return_complex=True).abs().square().clamp_min(1e-7).sqrt()
        sc = sc + torch.linalg.norm(my - mx) / torch.linalg.norm(my)
        mag = mag + (my.log() - mx.log()).abs().mean()
    k = len(fft_sizes)
    return factor_sc * sc / k, factor_mag * mag / k
