"""Host side of the AERO forward: weight packing and the kernel launch sequence.

Mirrors the control flow of reference ``src/models/aero.py:446-523`` (``Aero.forward``),
``:108-135`` (``HEncLayer.forward``), ``:189-215`` (``HDecLayer.forward``) and
``src/models/modules.py`` (``FTB`` 304-325, ``DConv`` 221-249, ``BLSTM`` 32-65, ``LocalState``
94-127), but every arithmetic step is a call into libaero_b200.so through the C ABI
(``include/aero_b200.h``).  PyTorch is used for device memory and the stream only.

Layout: activations are channels-last ``[B, F, T, C]``; see DESIGN.md.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import cabi
from .cabi import (ACT_GELU, ACT_NONE, ACT_RELU, NA_GELU, NA_GLU, NA_GLU_SCALE_RES, NA_SNAKE, TAPS_CONV,
                   TAPS_CONVT)

_LSTM_MAX_STEPS = 200      # reference modules.py:215 BLSTM(..., max_steps=200)
_ATTN_HEADS, _ATTN_NDECAY = 4, 4   # reference modules.py:154 DConv(heads=4, ndecay=4)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _pad4(n):
    return (n + 3) & ~3


def pack_taps(w_nkt):
    """[N, K, taps] -> contiguous [taps, K, pad4(N)] (N contiguous: the tap-GEMM weight layout)."""
    n, k, taps = w_nkt.shape
    out = w_nkt.new_zeros(taps, k, _pad4(n))
    out[:, :, :n] = w_nkt.permute(2, 1, 0)
    return out.contiguous()


def tf32_round(t):
    """Round-to-nearest (ties away) to TF32's 10-bit mantissa, as cvt.rna.tf32.f32 does on the device."""
    bits = t.contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def lstm_gate_reorder(H):
    """Row order of the tcgen05 LSTM recurrence (csrc/lstm_tc.cu): 4/GPT tiles of 128 rows per direction.
    GPT=1 (H > 64): tile g = gate g, lane = cell.  GPT=2 (H <= 64): tile t = gates (2t, 2t+1); in each 32-lane
    group lanes 0-15 carry gate 2t and lanes 16-31 gate 2t+1 of the same 16 cells.
    Returns (source row in PyTorch's [i|f|g|o] x H order, validity mask)."""
    gpt = 2 if H <= 64 else 1
    n_tiles = 4 // gpt
    idx = torch.arange(n_tiles * 128)
    m, r = idx // 128, idx % 128
    if gpt == 1:
        gate, cell = m, r
    else:
        q, lane = r // 32, r % 32
        gate, cell = 2 * m + lane // 16, 16 * q + lane % 16
    src = (gate * H + cell).clamp_max(4 * H - 1)
    return src, cell < H


def lstm_whh_fp16(whh_rows):
    """[rows, H] fp32 -> [rows, 64*ceil(H/64)] fp16 (zero padded): the A operand of the tcgen05 LSTM recurrence."""
    rows, H = whh_rows.shape
    out = torch.zeros(rows, 64 * ((H + 63) // 64), dtype=torch.float16, device=whh_rows.device)
    out[:, :H] = whh_rows.to(torch.float16)
    return out.contiguous()


def pack_kmajor_fp16(w_tkn):
    """[taps, K, pad4(N)] fp32 -> [taps, pad4(N), pad8(K)] fp16: the kind::f16 tcgen05 weight layout (16-byte rows for TMA)."""
    taps, k, n = w_tkn.shape
    out = torch.zeros(taps, n, (k + 7) & ~7, dtype=torch.float16, device=w_tkn.device)
    out[:, :, :k] = w_tkn.permute(0, 2, 1).to(torch.float16)
    return out.contiguous()


def glu_perm(n, device):
    """Column order that puts GLU partners (j, j + n/2) next to each other."""
    half = n // 2
    return torch.stack([torch.arange(half, device=device), torch.arange(half, device=device) + half], 1).reshape(-1)


class _Stats:
    """Bump allocator over one fp64 buffer of {sum, sumsq} pairs, zeroed once per forward."""

    def __init__(self, device, capacity=1 << 16):
        self.buf = torch.zeros(capacity, 2, dtype=torch.float64, device=device)
        self.used = 0

    def reset(self):
        self.buf.zero_()
        self.used = 0

    def take(self, slots):
        if self.used + slots > self.buf.shape[0]:
            raise RuntimeError("aero_b200: statistics workspace too small; raise _Stats capacity")
        view = self.buf[self.used:self.used + slots]
        self.used += slots
        return view


class AeroEngine:
    def __init__(self, model):
        self._init_state(model, cabi.load())

    def _init_state(self, model, lib):
        """All engine state (also used by the test / tooling subclasses that replace the kernel wrappers)."""
        self.model = model
        self.geom = model.geom
        self.lib = lib
        self._packed = None
        self._packed_key = None
        # workspaces live in "shape sets" (one per (input shape, precision)); only the most recently used few are kept,
        # so a loop over variable-length files (reference test.py / evaluate.py) cannot grow device memory without bound.
        # A CUDA graph holds raw pointers into its shape set: evicting a set drops its graph too.
        self._bufsets = {}
        self._bufs = {}
        self.max_shape_sets = 4
        self._plist = None
        self._windows = {}
        self._stats = None
        # 2 (default): FP16-stored activations / tcgen05 kind::f16 operands, fp32 accumulate, fp32 GroupNorm inputs and
        #    gate pre-activations -- TF32's 10-bit mantissa at half the HBM bytes and twice the tensor-core rate;
        # 1: fp32-stored activations rounded to TF32 / tcgen05 kind::tf32;  0: exact fp32 SIMT kernels everywhere.
        self.precision = 2
        # alternate the walk direction of consecutive tap-GEMM / norm_act launches (AERO_TG_REVERSE) so that a consumer starts
        # on what its producer wrote last; measured on B200: no gain for this model (12.19 ms either way), so off
        self.snake = False
        self._flip = False
        # precision 2 only: pre-normalisation GEMM outputs (GroupNorm inputs) are stored in FP16 as well; their statistics are
        # taken from the stored values.  Halves the bytes of every norm_act pass and of the GEMM writes that feed them
        # (tests/err_budget_emu.py: +6 % end-to-end error, paid for by keeping the last decoder layer's GLU output in fp32)
        self.raw16 = True
        # precision 2 + tcgen05 LSTM: optionally store the gate pre-activations (input projections, 8H columns per frame) in FP16
        # too.  Accuracy-neutral (tests/err_budget_emu.py) but measured SLOWER on B200: the recurrence reads them with scalar
        # loads (one gate of one cell per lane), and 2-byte loads cost 307 -> 336 us per H = 96 launch while the projection
        # GEMMs gain only ~0.05 ms per step (tools/kprof.py lstm96 / lstm48, round 2) -- off.
        self.gin16 = False
        self.lstm_tc = True         # tcgen05 LSTM recurrence (re-ordered gate layout) when precision >= 1
        self.fuse_pre_ftb = True    # encoder layer 0: evaluate FTB through the linear pre_conv (csrc/ftb_lin.cu)
        self.fp32_tags = ()         # tap-GEMM tags (prefix match) forced onto the exact-fp32 path even when precision == 1
        self._prof, self._prof_tags = None, set()
        self._wk, self._wh, self._wname = {}, {}, {}
        # CUDA-graph replay of the launch sequence, per input shape: "auto" captures a shape the third time it is seen
        # (steady-state serving / evaluation loops), True captures on first sight, False always launches eagerly.
        self.use_graph = "auto"
        self._graphs = {}
        self._seen = {}

    # ------------------------------------------------------------------ plumbing
    def invalidate(self):
        self._packed = None
        self._bufsets = {}
        self._bufs = {}
        self._graphs = {}
        self._seen = {}
        self._plist = None

    def _select_shape_set(self, key):
        """Make `key`'s workspace set current (LRU order = dict insertion order)."""
        cur = self._bufsets.pop(key, None)
        if cur is None:
            cur = {}
            while len(self._bufsets) >= self.max_shape_sets:
                old = next(iter(self._bufsets))
                del self._bufsets[old]
                for gk in [gk for gk in self._graphs if gk[0] == old[0] and gk[2] == old[1]]:
                    del self._graphs[gk]
        self._bufsets[key] = cur
        self._bufs = cur

    def _weights_version(self):
        """Cheap change detector for the model's tensors: in-place updates (optimizer steps, load_state_dict) bump
        `_version`, which only ever grows, so the sum changes whenever any tensor does.  An update that writes through raw
        pointers must bump it itself, as aero_b200.optim.FusedAdam.step does.  The tensor list is cached;
        `Aero._apply` / `load_state_dict` (device moves, re-materialised parameters) call invalidate()."""
        if self._plist is None:
            self._plist = list(self.model.parameters()) + list(self.model.buffers())
        return sum(t._version for t in self._plist)

    def _device(self):
        return next(self.model.parameters()).device

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self._device()).cuda_stream)

    def _on_device(self):
        """Context that makes the model's device current: every launch, event and allocation below it targets the
        device the weights live on, whatever the caller's current device is (the reference nn.Module works that way)."""
        return torch.cuda.device(self._device())

    def _require(self, x):
        dev = self._device()
        if dev.type != "cuda" or not x.is_cuda:
            raise RuntimeError(
                "aero_b200.Aero runs on CUDA only (sm_100a kernels in libaero_b200.so); there is no CPU path. "
                f"model on {dev}, input on {x.device}")
        if x.device != dev:
            raise RuntimeError(f"input on {x.device} but model on {dev}")
        if x.dtype != torch.float32:
            raise TypeError(f"aero_b200 computes in fp32; got {x.dtype}")

    def _buf(self, name, *shape, dtype=torch.float32, zero=False):
        """Cached workspace.  zero=True: zero-filled when created (row padding that no kernel writes must stay finite)."""
        key = (name, shape, dtype)
        t = self._bufs.get(key)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=self._device())
            self._bufs[key] = t
        return t

    def _adt(self, channels):
        """Storage type of an activation tensor that feeds a tensor-core GEMM: FP16 in precision 2 when its rows are
        16-byte multiples (TMA), else fp32 (rounded to TF32 by its producer when precision >= 1)."""
        return torch.float16 if (self.precision == 2 and channels % 8 == 0) else torch.float32

    def _rdt(self, channels):
        """Storage type of a pre-normalisation GEMM output (a GroupNorm input)."""
        return torch.float16 if (self.precision == 2 and self.raw16 and channels % 8 == 0) else torch.float32

    def _raw(self, like, name):
        """Buffer for a pre-normalisation GEMM output whose normalised form is `like`: `like` itself (norm_act runs in
        place) when the storage types agree, else a separate fp32 buffer."""
        return like if like.dtype == self._rdt(like.shape[-1]) else self._buf(name, *like.shape)

    def _window(self, win):
        key = (win, self._device())
        w = self._windows.get(key)
        if w is None:
            # computed on the host in fp32 exactly as reference spec.py:15 does, then moved
            w = torch.hann_window(win).to(self._device())
            self._windows[key] = w
        return w

    def _weights(self):
        key = self._weights_version()
        if self._packed is None or key != self._packed_key:
            self._packed = self._pack()
            self._packed_key = key
        return self._packed

    # ------------------------------------------------------------------ weight packing
    @torch.no_grad()
    def _pack(self):
        sd = {k: v.detach() for k, v in self.model.state_dict().items()}
        dev = self._device()
        kw = self.geom.kw
        W = {}

        def fold_bn(w_nk, b, bn):
            s = sd[bn + ".weight"] * torch.rsqrt(sd[bn + ".running_var"] + 1e-5)
            return w_nk * s.view(-1, *([1] * (w_nk.dim() - 1))), (b - sd[bn + ".running_mean"]) * s + sd[bn + ".bias"]

        for g in self.geom.layers:
            p = f"encoder.{g.index}"
            cin = g.enc_cin
            if g.index == 0:
                W[p + ".pre.w"] = pack_taps(sd[p + ".pre_conv.weight"][:, :, 0, 0][:, :, None])
                W[p + ".pre.b"] = sd[p + ".pre_conv.bias"].contiguous()
                cin = g.ch
            if g.ftb:
                q = p + ".freq_attn_block"
                Fi = g.f_in
                w, b = fold_bn(sd[q + ".conv1.0.weight"][:, :, 0, 0], sd[q + ".conv1.0.bias"], q + ".conv1.1")
                W[p + ".ftb1.w"], W[p + ".ftb1.b"] = pack_taps(w[:, :, None]), b.contiguous()
                r = w.shape[0]
                w1d = sd[q + ".conv1d.0.weight"]                              # [C, r*F, 9], channel = j*F + f
                w1d = w1d.view(cin, r, Fi, 9).permute(0, 2, 1, 3).reshape(cin, Fi * r, 9)   # -> f*r + j
                w, b = fold_bn(w1d, sd[q + ".conv1d.0.bias"], q + ".conv1d.1")
                W[p + ".ftb1d.w"], W[p + ".ftb1d.b"] = pack_taps(w), b.contiguous()
                W[p + ".ftbfc.w"] = sd[q + ".freq_fc.weight"].contiguous()
                w, b = fold_bn(sd[q + ".conv2.0.weight"][:, :, 0, 0], sd[q + ".conv2.0.bias"], q + ".conv2.1")
                W[p + ".ftb2.w"], W[p + ".ftb2.b"] = pack_taps(w[:, :, None]), b.contiguous()
                if g.index == 0:
                    # FTB through the linear pre_conv (include/aero_b200.h, aero_ftb_lin_out_fwd): x = Wp z + bp
                    Wp, bp = sd[p + ".pre_conv.weight"][:, :, 0, 0].double(), sd[p + ".pre_conv.bias"].double()
                    w1, b1 = fold_bn(sd[q + ".conv1.0.weight"][:, :, 0, 0], sd[q + ".conv1.0.bias"], q + ".conv1.1")
                    w1, b1 = w1.double(), b1.double()
                    W[p + ".ftb1p.w"] = (w1 @ Wp).float().contiguous()                  # [r, J]
                    W[p + ".ftb1p.b"] = (w1 @ bp + b1).float().contiguous()
                    w2, b2 = fold_bn(sd[q + ".conv2.0.weight"][:, :, 0, 0], sd[q + ".conv2.0.bias"], q + ".conv2.1")
                    w2, b2 = w2.double(), b2.double()
                    Cq, J = Wp.shape
                    w2a, w2b = w2[:, :Cq], w2[:, Cq:]                                   # cat([freq_fc out, x]) (modules.py:322)
                    ext = torch.cat([Wp, bp[:, None]], 1)                              # [C, J+1]
                    Q = (w2a.t()[:, :, None] * ext[:, None, :]).reshape(Cq, Cq * (J + 1))   # Q[c][n*(J+1)+j]
                    W[p + ".ftbQ.wf32"] = pack_taps(Q.t().float()[:, :, None])         # exact-fp32 GEMM (tiny): no tensor-core twin
                    W[p + ".ftbV"] = (w2b @ Wp).float().contiguous()
                    W[p + ".ftbd"] = (w2b @ bp + b2).float().contiguous()
                    W[p + ".ftbs"] = sd[q + ".freq_fc.weight"].double().sum(1).float().contiguous()
            W[p + ".conv.w"] = pack_taps(sd[p + ".conv.weight"][:, :, :, 0])
            W[p + ".conv.b"] = sd[p + ".conv.bias"].contiguous()
            wr, br = sd[p + ".rewrite.weight"][:, :, 0, 0], sd[p + ".rewrite.bias"]
            if g.norm:
                for nm in ("norm1", "norm2"):
                    W[f"{p}.{nm}.g"], W[f"{p}.{nm}.b"] = sd[f"{p}.{nm}.weight"].contiguous(), sd[f"{p}.{nm}.bias"].contiguous()
            else:
                perm = glu_perm(wr.shape[0], dev)
                wr, br = wr[perm], br[perm]
            W[p + ".rw.w"], W[p + ".rw.b"] = pack_taps(wr[:, :, None]), br.contiguous()
            if g.index == 0 and kw["freq_emb"]:
                W["emb"] = (sd["freq_emb.embedding.weight"] * (kw["emb_scale"] * kw["freq_emb"])).contiguous()
            if g.dconv:
                for d in range(abs(kw["dconv_depth"])):
                    q = f"{p}.dconv.layers.{d}"
                    o = f"{p}.dc{d}"
                    W[o + ".c1.w"], W[o + ".c1.b"] = pack_taps(sd[q + ".conv1.0.weight"]), sd[q + ".conv1.0.bias"].contiguous()
                    W[o + ".n1.g"], W[o + ".n1.b"] = sd[q + ".conv1.1.weight"].contiguous(), sd[q + ".conv1.1.bias"].contiguous()
                    W[o + ".a"] = sd[q + ".act.a"].reshape(-1).contiguous()
                    W[o + ".c2.w"], W[o + ".c2.b"] = pack_taps(sd[q + ".conv2.0.weight"]), sd[q + ".conv2.0.bias"].contiguous()
                    W[o + ".n2.g"], W[o + ".n2.b"] = sd[q + ".conv2.1.weight"].contiguous(), sd[q + ".conv2.1.bias"].contiguous()
                    W[o + ".ls"] = sd[q + ".conv2.3.scale"].contiguous()
                    if g.lstm:
                        for l in range(2):
                            wih = torch.cat([sd[f"{q}.lstm.lstm.weight_ih_l{l}"], sd[f"{q}.lstm.lstm.weight_ih_l{l}_reverse"]], 0)
                            W[f"{o}.lstm{l}.ih.w"] = pack_taps(wih[:, :, None])
                            W[f"{o}.lstm{l}.b"] = torch.cat([
                                sd[f"{q}.lstm.lstm.bias_ih_l{l}"] + sd[f"{q}.lstm.lstm.bias_hh_l{l}"],
                                sd[f"{q}.lstm.lstm.bias_ih_l{l}_reverse"] + sd[f"{q}.lstm.lstm.bias_hh_l{l}_reverse"]]).contiguous()
                            W[f"{o}.lstm{l}.whh"] = torch.stack([sd[f"{q}.lstm.lstm.weight_hh_l{l}"],
                                                                  sd[f"{q}.lstm.lstm.weight_hh_l{l}_reverse"]]).contiguous()
                        # tcgen05 recurrence: gate rows re-ordered / padded (include/aero_b200.h, aero_lstm_params.precision)
                        H_ = sd[f"{q}.lstm.lstm.weight_hh_l0"].shape[1]
                        src, ok = (t_.to(dev) for t_ in lstm_gate_reorder(H_))
                        for l in range(2):
                            def reord(t):
                                return torch.where(ok.view(-1, *([1] * (t.dim() - 1))), t[src], torch.zeros_like(t[src]))
                            whh = [reord(sd[f"{q}.lstm.lstm.weight_hh_l{l}{sfx}"]) for sfx in ("", "_reverse")]
                            W[f"{o}.lstm{l}r.whh"] = lstm_whh_fp16(torch.cat(whh, 0))
                        W[o + ".lin.w"] = pack_taps(sd[q + ".lstm.linear.weight"][:, :, None])
                        W[o + ".lin.b"] = sd[q + ".lstm.linear.bias"].contiguous()
                    if g.attn:
                        a = q + ".time_attn"
                        names = ("query", "key", "content", "query_decay")
                        W[o + ".qkvd.w"] = pack_taps(torch.cat([sd[f"{a}.{n}.weight"] for n in names], 0))
                        W[o + ".qkvd.b"] = torch.cat([sd[f"{a}.{n}.bias"] for n in names]).contiguous()
                        W[o + ".proj.w"] = pack_taps(sd[a + ".proj.weight"])
                        W[o + ".proj.b"] = sd[a + ".proj.bias"].contiguous()

        for j, g in enumerate(reversed(self.geom.layers)):
            p = f"decoder.{j}"
            wr, br = sd[p + ".rewrite.weight"], sd[p + ".rewrite.bias"]       # [4ch, 2ch, 3, 3]
            wr = wr.reshape(wr.shape[0], wr.shape[1], -1)
            if j == 0:
                wr = wr[:, g.ch:]          # decoder input starts at zero (aero.py:484): keep the skip half only
            if g.norm:
                for nm in ("norm1", "norm2"):
                    W[f"{p}.{nm}.g"], W[f"{p}.{nm}.b"] = sd[f"{p}.{nm}.weight"].contiguous(), sd[f"{p}.{nm}.bias"].contiguous()
            else:
                perm = glu_perm(wr.shape[0], dev)
                wr, br = wr[perm], br[perm]
            W[p + ".rw.w"], W[p + ".rw.b"] = pack_taps(wr), br.contiguous()
            W[p + ".ct.w"] = pack_taps(sd[p + ".conv_tr.weight"][:, :, :, 0].permute(1, 0, 2))
            W[p + ".ct.b"] = sd[p + ".conv_tr.bias"].contiguous()
        out = {k: (v.to(dev) if v.dtype == torch.float16 else v.to(device=dev, dtype=torch.float32)) for k, v in W.items()}
        # K-major TF32 twins of every tap-GEMM weight for the tcgen05 path: [taps, K, pad4(N)] -> [taps, pad4(N), K]
        # ... and FP16 twins [taps, pad4(N), pad8(K)] for kind::f16
        self._wk, self._wh, self._wname = {}, {}, {}
        for k in [k for k in out if k.endswith("ftbfc.w")]:
            out[k + "@k"] = tf32_round(out[k])          # [F', F] is already K-contiguous
            out[k + "@h"] = pack_kmajor_fp16(out[k].t()[None].contiguous())[0]
        for k in [k for k in out if k.endswith(".w") and out[k].dim() == 3]:
            out[k + "@k"] = tf32_round(out[k].permute(0, 2, 1).contiguous())
            out[k + "@h"] = pack_kmajor_fp16(out[k])
            self._wk[out[k].data_ptr()] = out[k + "@k"]
            self._wh[out[k].data_ptr()] = out[k + "@h"]
            self._wname[out[k].data_ptr()] = k[:-2]
        return out

    # ------------------------------------------------------------------ kernel wrappers
    def _gemm(self, out, w, *, B, F_out, T, N, C1, a1=None, a2=None, C2=0, F_in=None, T_in=None,
              a1_s=None, a2_s=None, o_s=None, mode=TAPS_CONV, kf=1, kt=1, stride_f=1, pad_f=0, dil_t=1, pad_t=0,
              f_off=0, bias=None, act=ACT_NONE, glu=0, stats=None, stats_mode=0, groups=1, addend=None,
              colscale=None, cs_s=(0, 0), residual=None, r_s=None, samp_affine=None, w_sb=0, tag=None, rnd=False):
        F_in = F_out if F_in is None else F_in
        T_in = T if T_in is None else T_in
        n_out = N // 2 if glu else N

        def cl(F, C_):
            return (F * T_in * C_, T_in * C_, C_)
        a1_s = a1_s or (cl(F_in, C1) if a1 is not None else (0, 0, 0))
        a2_s = a2_s or (cl(F_in, C2) if a2 is not None else (0, 0, 0))
        o_s = o_s or (F_out * T * n_out, T * n_out, n_out)
        r_s = r_s or (o_s if residual is not None else (0, 0, 0))
        tag = tag or self._wname.get(w.data_ptr())
        src = a1 if a1 is not None else a2
        a16 = src.dtype == torch.float16
        o16 = out.dtype == torch.float16
        if a1 is not None and a2 is not None and a1.dtype != a2.dtype:
            raise TypeError("aero_b200: the two sources of a tap-GEMM must share a storage type")
        if residual is not None and residual.dtype != out.dtype:
            raise TypeError("aero_b200: residual and output of a tap-GEMM must share a storage type")
        flags = (cabi.TG_ROUND_TF32 if (rnd and self.precision >= 1 and not o16) else 0) | (cabi.TG_A_F16 if a16 else 0) | \
                (cabi.TG_OUT_F16 if o16 else 0) | (cabi.TG_REVERSE if self._next_dir() else 0)
        p = cabi.TapGemmParams(B, F_out, T, N, F_in, T_in, C1, C2, mode, kf, kt, stride_f, pad_f, dil_t, pad_t, f_off,
                               act, glu, stats_mode, groups, *a1_s, *a2_s, w_sb, *o_s, *r_s, *cs_s, 0, flags)
        if mode == cabi.TAPS_MIX:
            p.precision = 2 if a16 else 1        # tcgen05-only mode; `w` is already the K-major twin of the right kind
        elif self.precision >= 1 and w_sb == 0 and not (tag and self.fp32_tags and tag.startswith(self.fp32_tags)):
            wk = (self._wh if a16 else self._wk).get(w.data_ptr())
            if wk is not None and self.lib.aero_tapgemm_tc_eligible(C.byref(p)):
                p.precision, w = (2 if a16 else 1), wk
        timed = self._prof is not None and tag in self._prof_tags
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        rc = self.lib.aero_tapgemm_fwd(_ptr(a1), _ptr(a2), _ptr(w), _ptr(bias), _ptr(addend), _ptr(colscale),
                                       _ptr(residual), _ptr(samp_affine), _ptr(out), _ptr(stats), C.byref(p),
                                       self._stream())
        cabi.check(rc, self.lib)
        if timed:
            e1.record()
            ntaps = kf * kt if mode == TAPS_CONV else kf // stride_f
            self._prof.append((tag, e0, e1, 2.0 * B * F_out * T * N * (C1 + C2) * ntaps))
        return out

    def _next_dir(self):
        """Walk direction of the next tap-GEMM / norm_act launch: alternating, so that a consumer starts where its producer
        just finished (that part of the tensor is still in L2)."""
        if not self.snake:
            return False
        self._flip = not self._flip
        return self._flip

    def start_profile(self, tags):
        """Time the tap-GEMM launches whose tag is in `tags` with CUDA events on the launch stream."""
        self._prof, self._prof_tags = [], set(tags)

    def stop_profile(self):
        torch.cuda.synchronize()
        out = {}
        for tag, e0, e1, flops in self._prof or []:
            d = out.setdefault(tag, {"ms": 0.0, "flops": 0.0, "launches": 0})
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += flops
            d["launches"] += 1
        self._prof = None
        return out

    def _gemm_flat(self, out, a, w, npix, K, N, **kw):
        """1x1 layer over `npix` independent pixels (any leading shape flattened)."""
        return self._gemm(out, w, a1=a, B=1, F_out=1, T=npix, N=N, C1=K, **kw)

    def _norm_act(self, x, stats, gamma, beta, y, *, B, F_in, T, C_, groups, scope, op, F_out=None, f_off=0,
                  snake_a=None, scale=None, residual=None, rnd=False):
        o16, i16 = y.dtype == torch.float16, x.dtype == torch.float16
        if (i16 and not o16) or (residual is not None and residual.dtype != y.dtype):
            raise TypeError("aero_b200: norm_act reads fp32 (or FP16 when it writes FP16) and its residual shares the output's storage type")
        p = cabi.NormActParams(B, F_in, F_in if F_out is None else F_out, f_off, T, C_, groups, scope, op, 1e-5,
                               (cabi.TG_ROUND_TF32 if (rnd and self.precision >= 1 and not o16) else 0) |
                               (cabi.TG_OUT_F16 if o16 else 0) | (cabi.TG_A_F16 if i16 else 0) |
                               (cabi.TG_REVERSE if self._next_dir() else 0))
        rc = self.lib.aero_norm_act_fwd(_ptr(x), _ptr(stats), _ptr(gamma), _ptr(beta), _ptr(snake_a), _ptr(scale),
                                        _ptr(residual), _ptr(y), C.byref(p), self._stream())
        cabi.check(rc, self.lib)
        return y

    def _lstm_rec(self, gin, bias_pad, whh, hout, *, rows, T, H, n_win, steps, stride, in_windowed, out_windowed,
                  tc=False):
        o16 = hout.dtype == torch.float16
        p = cabi.LstmParams(rows, T, H, n_win, steps, stride, in_windowed, out_windowed,
                            (cabi.TG_ROUND_TF32 if (self.precision >= 1 and not o16) else 0) | (cabi.TG_OUT_F16 if o16 else 0) |
                            (cabi.TG_A_F16 if gin.dtype == torch.float16 else 0), 1 if tc else 0)
        cabi.check(self.lib.aero_lstm_rec_fwd(_ptr(gin), _ptr(bias_pad), _ptr(whh), _ptr(hout), C.byref(p),
                                              self._stream()), self.lib)

    def _attn(self, qkvd, out, *, rows, T, H, heads, ndecay, ld):
        p = cabi.AttnParams(rows, T, H, heads, ndecay, ld, (cabi.TG_ROUND_TF32 if self.precision >= 1 else 0) |
                            (cabi.TG_OUT_F16 if out.dtype == torch.float16 else 0))
        cabi.check(self.lib.aero_local_attn_fwd(_ptr(qkvd), _ptr(out), C.byref(p), self._stream()), self.lib)

    def _sample_norm(self, x, stats, y, affine, B, per_sample, extent=None, rnd=False):
        cabi.check(self.lib.aero_sample_norm_fwd(_ptr(x), _ptr(stats), _ptr(y), _ptr(affine), B, per_sample,
                                                 extent or per_sample, 1 if rnd else 0, self._stream()), self.lib)

    def _freq_mix_small(self, x, Wfc, gate, out, *, B, F, M):
        flags = (cabi.TG_A_F16 | cabi.TG_OUT_F16) if x.dtype == torch.float16 else (cabi.TG_ROUND_TF32 if self.precision >= 1 else 0)
        cabi.check(self.lib.aero_freq_mix_small_fwd(_ptr(x), _ptr(Wfc), _ptr(gate), _ptr(out), B, F, M, flags, self._stream()),
                   self.lib)
        return out

    def _ftb_lin_squeeze(self, z, W1p, b1p, R, *, B, F, T, J, r, zrow):
        flags = cabi.TG_OUT_F16 if R.dtype == torch.float16 else (cabi.TG_ROUND_TF32 if self.precision >= 1 else 0)
        p = cabi.FtbLinParams(B, F, T, 0, J, flags, F * zrow, zrow, 0, 0)
        cabi.check(self.lib.aero_ftb_lin_squeeze_fwd(_ptr(z), _ptr(W1p), _ptr(b1p), _ptr(R), r, C.byref(p), self._stream()),
                   self.lib)
        return R

    def _ftb_lin_out(self, z, zm, M, s, V, d, out, *, B, F, T, N, J, zrow):
        flags = cabi.TG_OUT_F16 if out.dtype == torch.float16 else (cabi.TG_ROUND_TF32 if self.precision >= 1 else 0)
        p = cabi.FtbLinParams(B, F, T, N, J, flags, F * zrow, zrow, F * zrow, zrow)
        cabi.check(self.lib.aero_ftb_lin_out_fwd(_ptr(z), _ptr(zm), _ptr(M), _ptr(s), _ptr(V), _ptr(d), _ptr(out),
                                                 C.byref(p), self._stream()), self.lib)
        return out

    def stft_into(self, x, z, stats, *, n_fft, hop, win, channels, bins_out, strides):
        n_sig, length = x.shape[0], x.shape[1]
        frames = 1 + length // hop
        p = cabi.StftParams(n_fft, hop, win, n_sig, channels, length, frames, bins_out, *strides)
        rc = self.lib.aero_stft_fwd(_ptr(x), _ptr(self._window(win)), _ptr(z), _ptr(stats), C.byref(p), self._stream())
        cabi.check(rc, self.lib)

    def istft_into(self, z, y, *, n_fft, hop, win, channels, frames, bins_in, strides):
        n_sig, out_len = y.shape
        p = cabi.IstftParams(n_fft, hop, win, n_sig, channels, frames, bins_in, out_len, *strides)
        rc = self.lib.aero_istft_fwd(_ptr(z), _ptr(self._window(win)), _ptr(y), C.byref(p), self._stream())
        cabi.check(rc, self.lib)

    # ------------------------------------------------------------------ public pieces
    @torch.no_grad()
    def spec(self, x, scale=False):
        """reference aero.py:409-421 -> complex [..., nfft/2, frames]."""
        self._require(x)
        with self._on_device():
            return self._spec(x, scale)

    def _spec(self, x, scale):
        g = self.geom
        *lead, length = x.shape
        hop = g.hop_in
        if length % hop:
            x = torch.nn.functional.pad(x, (0, hop - length % hop))
        hl, win = (g.hop_out, g.win_out) if scale else (hop, g.win_in)
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        bins = g.nfft // 2
        frames = 1 + x2.shape[1] // hl
        z = torch.empty(x2.shape[0], bins, frames, 2, dtype=torch.float32, device=x.device)
        self.stft_into(x2, z, None, n_fft=g.nfft, hop=hl, win=win, channels=1, bins_out=bins,
                       strides=(bins * frames * 2, 0, frames * 2, 2))
        return torch.view_as_complex(z).view(*lead, bins, frames)

    @torch.no_grad()
    def ispec(self, zc):
        """reference aero.py:423-428: complex [..., nfft/2, frames] -> [..., hop_out*(frames-1)]."""
        g = self.geom
        *lead, bins, frames = zc.shape
        z = torch.view_as_real(zc.reshape(-1, bins, frames).contiguous())
        self._require(z)
        with self._on_device():
            return self._ispec(z, lead, bins, frames)

    def _ispec(self, z, lead, bins, frames):
        g = self.geom
        y = torch.empty(z.shape[0], g.hop_out * (frames - 1), dtype=torch.float32, device=z.device)
        self.istft_into(z, y, n_fft=g.nfft, hop=g.hop_out, win=g.win_out, channels=1, frames=frames, bins_in=bins,
                        strides=(bins * frames * 2, 0, frames * 2, 2))
        return y.view(*lead, y.shape[-1])

    # ------------------------------------------------------------------ blocks
    def _ftb(self, x, W, p, B, Fq, T, Cc, tag):
        """reference modules.py:304-325 (eval BatchNorm folded into the convs at pack time)."""
        r = 5
        R = self._buf(tag + ".R", B, T, Fq * r, dtype=self._adt(Fq * r))
        self._gemm(R, W[p + ".ftb1.w"], a1=x, B=B, F_out=Fq, T=T, N=r, C1=Cc, bias=W[p + ".ftb1.b"], act=ACT_RELU,
                   o_s=(T * Fq * r, r, Fq * r), rnd=True)
        G = self._buf(tag + ".G", B, T, Cc)
        self._gemm(G, W[p + ".ftb1d.w"], a1=R, B=B, F_out=1, T=T, N=Cc, C1=Fq * r, kt=9, pad_t=4,
                   bias=W[p + ".ftb1d.b"], act=ACT_RELU, a1_s=(T * Fq * r, 0, Fq * r), o_s=(T * Cc, 0, Cc))
        Y = self._buf(tag + ".Y", B, Fq, T, Cc, dtype=x.dtype)
        x16 = x.dtype == torch.float16
        q = 8 if x16 else 4
        if self.precision >= 1 and Fq in (8, 16) and (T * Cc) % 4 == 0:
            # deep layers: too few rows for tensor-core tiles -- one pass at copy bandwidth (csrc/ftb_lin.cu)
            self._freq_mix_small(x, W[p + ".ftbfc.w"], G, Y, B=B, F=Fq, M=T * Cc)
        elif self.precision >= 1 and Fq % q == 0 and Fq >= 8 and (T * Cc) % q == 0 and \
                not (self.fp32_tags and (p + ".ftbfc").startswith(self.fp32_tags)):
            # frequency mixing on the tensor cores: contraction over the row axis, activations as the MN-major operand
            self._gemm(Y, W[p + (".ftbfc.w@h" if x16 else ".ftbfc.w@k")], a1=x, mode=cabi.TAPS_MIX, B=B, F_out=1, T=T * Cc,
                       N=Fq, C1=Fq, a1_s=(Fq * T * Cc, 0, T * Cc), o_s=(Fq * T * Cc, 0, T * Cc), colscale=G, cs_s=(T * Cc, 0),
                       rnd=True, tag=p + ".ftbfc")
        else:
            # fp32 path: a GEMM whose "weights" are the activations: out[f'] = sum_f Wfc[f',f] x[f], times the gate
            self._gemm(Y, x.float() if x16 else x, a1=W[p + ".ftbfc.w"], B=B, F_out=1, T=Fq, T_in=Fq, N=T * Cc, C1=Fq,
                       a1_s=(0, 0, Fq), w_sb=Fq * T * Cc, o_s=(Fq * T * Cc, 0, T * Cc), colscale=G, cs_s=(T * Cc, 0), rnd=True,
                       tag=p + ".ftbfc")
        out = self._buf(tag + ".out", B, Fq, T, Cc, dtype=x.dtype)
        self._gemm(out, W[p + ".ftb2.w"], a1=Y, a2=x, B=1, F_out=1, T=B * Fq * T, N=Cc, C1=Cc, C2=Cc,
                   bias=W[p + ".ftb2.b"], act=ACT_RELU, rnd=True)
        return out

    def _pre_ftb(self, xn, xr, W, p, B, Fq, T, J, Cc, tag, zrow):
        """Encoder layer 0: pre_conv (aero.py:112) + FTB (modules.py:304-325) evaluated through the linearity of pre_conv
        (include/aero_b200.h, aero_ftb_lin_out_fwd): the C-channel tensors pre_conv(z), freq_fc(..), cat(..) never exist.
        xn: normalised spectrogram [B, Fq, zrow] (rows padded to 16 bytes); xr: its TF32-rounded copy for the tensor cores."""
        r = 5
        R = self._buf(tag + ".R", B, T, Fq * r, dtype=self._adt(Fq * r))
        self._ftb_lin_squeeze(xn, W[p + ".ftb1p.w"], W[p + ".ftb1p.b"], R, B=B, F=Fq, T=T, J=J, r=r, zrow=zrow)
        G = self._buf(tag + ".G", B, T, Cc)
        self._gemm(G, W[p + ".ftb1d.w"], a1=R, B=B, F_out=1, T=T, N=Cc, C1=Fq * r, kt=9, pad_t=4,
                   bias=W[p + ".ftb1d.b"], act=ACT_RELU, a1_s=(T * Fq * r, 0, Fq * r), o_s=(T * Cc, 0, Cc))
        Zm = self._buf(tag + ".Zm", B, Fq, zrow, zero=True)
        if xr is not None and Fq % 4 == 0 and Fq >= 8:
            self._gemm(Zm, W[p + ".ftbfc.w@k"], a1=xr, mode=cabi.TAPS_MIX, B=B, F_out=1, T=T * J, N=Fq, C1=Fq,
                       a1_s=(Fq * zrow, 0, zrow), o_s=(Fq * zrow, 0, zrow), tag=p + ".ftbfc")
        else:
            self._gemm(Zm, xn, a1=W[p + ".ftbfc.w"], B=B, F_out=1, T=Fq, T_in=Fq, N=T * J, C1=Fq, a1_s=(0, 0, Fq),
                       w_sb=Fq * zrow, o_s=(Fq * zrow, 0, zrow), tag=p + ".ftbfc")
        M = self._buf(tag + ".M", B * T, Cc * (J + 1))
        self._gemm_flat(M, G, W[p + ".ftbQ.wf32"], B * T, Cc, Cc * (J + 1), tag=p + ".ftbQ")
        out = self._buf(tag + ".out", B, Fq, T, Cc, dtype=self._adt(Cc))
        return self._ftb_lin_out(xn, Zm, M, W[p + ".ftbs"], W[p + ".ftbV"], W[p + ".ftbd"], out, B=B, F=Fq, T=T, N=Cc,
                                 J=J, zrow=zrow)

    def _blstm(self, h, W, o, rows, T, H, tag):
        """reference modules.py:32-65: framing, 2-layer BiLSTM, Linear, central-crop reassembly, skip."""
        if T > _LSTM_MAX_STEPS:
            steps, stride = _LSTM_MAX_STEPS, _LSTM_MAX_STEPS // 2
            n_win = math.ceil(T / stride)
        else:
            steps, stride, n_win = T, 0, 1
        n_seq = rows * n_win
        tc = self.lstm_tc and self.precision >= 1 and H % 4 == 0 and 32 < H <= 96
        # the input projections use PyTorch's own [dir][i,f,g,o][H] column order on both paths; only W_hh is re-ordered
        # (tile / lane order, FP16) for the tcgen05 recurrence
        G = 8 * H
        whh0, whh1 = (W[f"{o}.lstm0r.whh"], W[f"{o}.lstm1r.whh"]) if tc else (W[f"{o}.lstm0.whh"], W[f"{o}.lstm1.whh"])
        gdt = torch.float16 if (tc and self.precision == 2 and self.gin16 and h.dtype == torch.float16) else torch.float32
        gin1 = self._buf(tag + ".gin1", rows * T, G, dtype=gdt)
        self._gemm_flat(gin1, h, W[f"{o}.lstm0.ih.w"], rows * T, H, G, bias=W[f"{o}.lstm0.b"])
        h1 = self._buf(tag + ".h1", n_seq * steps, 2 * H, dtype=self._adt(2 * H))
        self._lstm_rec(gin1, W[f"{o}.lstm0.b"], whh0, h1, rows=rows, T=T, H=H, n_win=n_win, steps=steps,
                       stride=stride, in_windowed=0, out_windowed=1, tc=tc)
        gin2 = self._buf(tag + ".gin2", n_seq * steps, G, dtype=gdt if h1.dtype == torch.float16 else torch.float32)
        self._gemm_flat(gin2, h1, W[f"{o}.lstm1.ih.w"], n_seq * steps, 2 * H, G, bias=W[f"{o}.lstm1.b"])
        h2 = self._buf(tag + ".h2", rows * T, 2 * H, dtype=self._adt(2 * H))
        self._lstm_rec(gin2, W[f"{o}.lstm1.b"], whh1, h2, rows=rows, T=T, H=H, n_win=n_win, steps=steps,
                       stride=stride, in_windowed=1, out_windowed=0, tc=tc)
        self._gemm_flat(h, h2, W[o + ".lin.w"], rows * T, 2 * H, H, bias=W[o + ".lin.b"], residual=h, rnd=True)
        return h

    def _local_attn(self, h, W, o, rows, T, H, tag):
        """reference modules.py:94-127."""
        ld = 3 * H + _ATTN_HEADS * _ATTN_NDECAY
        qkvd = self._buf(tag + ".qkvd", rows * T, ld)
        # (fp32 output rounded to TF32 by the epilogue: the attention kernel feeds q/k/v to mma.sync without converting)
        self._gemm_flat(qkvd, h, W[o + ".qkvd.w"], rows * T, H, ld, bias=W[o + ".qkvd.b"], rnd=True)
        r = self._buf(tag + ".attn", rows * T, H, dtype=self._adt(H))
        self._attn(qkvd, r, rows=rows, T=T, H=H, heads=_ATTN_HEADS, ndecay=_ATTN_NDECAY, ld=ld)
        self._gemm_flat(h, r, W[o + ".proj.w"], rows * T, H, H, bias=W[o + ".proj.b"], residual=h, rnd=True)
        return h

    def _dconv(self, y, W, g, B, T, tag):
        """reference modules.py:221-249; rows are (b, f) pairs, which is just our memory order."""
        kw = self.geom.kw
        Fq, Cc = g.f_out, g.ch
        hid = int(Cc / kw["dconv_comp"])
        rows = B * Fq
        for d in range(abs(kw["dconv_depth"])):
            o = f"encoder.{g.index}.dc{d}"
            dil = 2 ** d if kw["dconv_depth"] > 0 else 1      # negative depth = no dilation (reference modules.py:176-177,201)
            st1 = self._stats.take(rows)
            h = self._buf(f"{tag}.h", B, Fq, T, hid, dtype=self._adt(hid))
            h_raw = self._raw(h, f"{tag}.h32")
            self._gemm(h_raw, W[o + ".c1.w"], a1=y, B=B, F_out=Fq, T=T, N=hid, C1=Cc, kt=3, dil_t=dil, pad_t=dil,
                       bias=W[o + ".c1.b"], stats=st1, stats_mode=2)
            self._norm_act(h_raw, st1, W[o + ".n1.g"], W[o + ".n1.b"], h, B=B, F_in=Fq, T=T, C_=hid, groups=1, scope=2,
                           op=NA_SNAKE, snake_a=W[o + ".a"], rnd=True)
            if g.lstm:
                self._blstm(h, W, o, rows, T, hid, f"{tag}.lstm")
            if g.attn:
                self._local_attn(h, W, o, rows, T, hid, f"{tag}.attn")
            st2 = self._stats.take(rows)
            u = self._buf(f"{tag}.u", B, Fq, T, 2 * Cc, dtype=self._rdt(2 * Cc))
            self._gemm(u, W[o + ".c2.w"], a1=h, B=B, F_out=Fq, T=T, N=2 * Cc, C1=hid, bias=W[o + ".c2.b"],
                       stats=st2, stats_mode=2)
            self._norm_act(u, st2, W[o + ".n2.g"], W[o + ".n2.b"], y, B=B, F_in=Fq, T=T, C_=2 * Cc, groups=1, scope=2,
                           op=NA_GLU_SCALE_RES, scale=W[o + ".ls"], residual=y, rnd=True)
        return y

    def _encode(self, x, W, g, B, T, xr=None):
        """reference aero.py:108-135 (+ the frequency-embedding add aero.py:475-480 for layer 0)."""
        kw = self.geom.kw
        p = f"encoder.{g.index}"
        tag = f"e{g.index}"
        Fi, Fo, Cc = g.f_in, g.f_out, g.ch
        cin = g.enc_cin
        fused = False
        if g.index == 0:
            zrow = x.shape[-1]                   # spectrogram rows [B, Fi, zrow]: T*cin floats padded to 16 bytes
            fused = g.ftb and self.fuse_pre_ftb and cin in (2, 4) and Cc % 8 == 0 and Cc <= 64
            if fused:
                x = self._pre_ftb(x, xr, W, p, B, Fi, T, cin, Cc, tag + ".ftb", zrow)
            else:
                pre = self._buf(tag + ".pre", B, Fi, T, Cc, dtype=self._adt(Cc))
                self._gemm(pre, W[p + ".pre.w"], a1=x, B=B, F_out=Fi, T=T, N=Cc, C1=cin, a1_s=(Fi * zrow, zrow, cin),
                           bias=W[p + ".pre.b"], rnd=True)
                x = pre
            cin = Cc
        if g.ftb and not fused:
            x = self._ftb(x, W, p, B, Fi, T, cin, tag + ".ftb")
        y = self._buf(tag + ".conv", B, Fo, T, Cc, dtype=self._adt(Cc))
        if g.norm:
            st = self._stats.take(B * kw["norm_groups"])
            y_raw = self._raw(y, tag + ".conv32")
            self._gemm(y_raw, W[p + ".conv.w"], a1=x, B=B, F_out=Fo, F_in=Fi, T=T, N=Cc, C1=cin, kf=g.kernel,
                       stride_f=g.stride, pad_f=g.pad, bias=W[p + ".conv.b"], stats=st, stats_mode=1,
                       groups=kw["norm_groups"])
            self._norm_act(y_raw, st, W[p + ".norm1.g"], W[p + ".norm1.b"], y, B=B, F_in=Fo, T=T, C_=Cc,
                           groups=kw["norm_groups"], scope=1, op=NA_GELU, rnd=True)
        else:
            self._gemm(y, W[p + ".conv.w"], a1=x, B=B, F_out=Fo, F_in=Fi, T=T, N=Cc, C1=cin, kf=g.kernel,
                       stride_f=g.stride, pad_f=g.pad, bias=W[p + ".conv.b"], act=ACT_GELU, rnd=True)
        if g.dconv:
            y = self._dconv(y, W, g, B, T, tag + ".dc")
        out = self._buf(tag + ".out", B, Fo, T, Cc, dtype=self._adt(Cc))
        if g.norm:
            st = self._stats.take(B * kw["norm_groups"])
            raw = self._buf(tag + ".rw", B, Fo, T, 2 * Cc, dtype=self._rdt(2 * Cc))
            self._gemm(raw, W[p + ".rw.w"], a1=y, B=B, F_out=Fo, T=T, N=2 * Cc, C1=Cc, bias=W[p + ".rw.b"],
                       stats=st, stats_mode=1, groups=kw["norm_groups"])
            self._norm_act(raw, st, W[p + ".norm2.g"], W[p + ".norm2.b"], out, B=B, F_in=Fo, T=T, C_=2 * Cc,
                           groups=kw["norm_groups"], scope=1, op=NA_GLU, rnd=True)
        else:
            self._gemm(out, W[p + ".rw.w"], a1=y, B=B, F_out=Fo, T=T, N=2 * Cc, C1=Cc, bias=W[p + ".rw.b"], glu=1,
                       addend=W.get("emb") if g.index == 0 else None, rnd=True)
        return out

    def _decode(self, x, skip, W, g, j, B, T, last, samp_affine):
        """reference aero.py:189-215."""
        kw = self.geom.kw
        p = f"decoder.{j}"
        tag = f"d{j}"
        Fq, Cc = g.f_out, g.ch
        c1 = 0 if x is None else Cc
        # the last layer's GLU output feeds the exact-fp32 final transposed conv: kept in fp32 (-15 % end-to-end error for 75 MB)
        y = self._buf(tag + ".glu", B, Fq, T, 2 * Cc, dtype=torch.float32 if last else self._adt(2 * Cc))
        common = dict(a1=x, a2=skip, B=B, F_out=Fq, T=T, N=4 * Cc, C1=c1, C2=Cc, kf=3, kt=3, pad_f=1, pad_t=1,
                      bias=W[p + ".rw.b"])
        if g.norm:
            st = self._stats.take(B * kw["norm_groups"])
            raw = self._buf(tag + ".rw", B, Fq, T, 4 * Cc, dtype=self._rdt(4 * Cc))
            self._gemm(raw, W[p + ".rw.w"], stats=st, stats_mode=1, groups=kw["norm_groups"], **common)
            self._norm_act(raw, st, W[p + ".norm1.g"], W[p + ".norm1.b"], y, B=B, F_in=Fq, T=T, C_=4 * Cc,
                           groups=kw["norm_groups"], scope=1, op=NA_GLU, rnd=True)
        else:
            # the last layer's transposed conv runs on the exact-fp32 thin kernel: do not round its input
            self._gemm(y, W[p + ".rw.w"], glu=1, rnd=not last, **common)
        cout = g.dec_cout
        f_full = (Fq - 1) * g.stride + g.kernel
        f_keep = f_full - 2 * g.pad
        z = self._buf(tag + ".out", B, f_keep, T, cout, dtype=torch.float32 if last else self._adt(cout))
        if g.norm:
            st = self._stats.take(B * kw["norm_groups"])
            raw = self._buf(tag + ".ct", B, f_full, T, cout, dtype=self._rdt(cout))
            self._gemm(raw, W[p + ".ct.w"], a1=y, B=B, F_out=f_full, F_in=Fq, T=T, N=cout, C1=2 * Cc, mode=TAPS_CONVT,
                       kf=g.kernel, stride_f=g.stride, bias=W[p + ".ct.b"], stats=st, stats_mode=1,
                       groups=kw["norm_groups"])
            self._norm_act(raw, st, W[p + ".norm2.g"], W[p + ".norm2.b"], z, B=B, F_in=f_full, F_out=f_keep,
                           f_off=g.pad, T=T, C_=cout, groups=kw["norm_groups"], scope=1,
                           op=cabi.NA_NONE if last else NA_GELU, rnd=not last)
            if last and samp_affine is not None:
                raise NotImplementedError("GroupNorm on the last decoder layer (norm_starts=0) is not supported")
        else:
            self._gemm(z, W[p + ".ct.w"], a1=y, B=B, F_out=f_keep, F_in=Fq, T=T, N=cout, C1=2 * Cc, mode=TAPS_CONVT,
                       kf=g.kernel, stride_f=g.stride, f_off=g.pad, bias=W[p + ".ct.b"],
                       act=ACT_NONE if last else ACT_GELU, samp_affine=samp_affine if last else None, rnd=not last)
        return z

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, mix, return_spec=False, return_lr_spec=False):
        """Public entry (behind Aero.forward).  With ``use_graph`` the ~110 launches of one forward are captured once per
        input shape into a CUDA graph and replayed: identical kernels and results, no per-launch host cost (this is what
        matters at batch 1, where the eager path is host-bound)."""
        self._require(mix)
        self._check_mode()
        with self._on_device():
            if not self.use_graph or return_spec or self._prof is not None or mix.shape[0] == 0 or \
                    torch.cuda.is_current_stream_capturing():
                return self._forward(mix, return_spec, return_lr_spec)
            key = (tuple(mix.shape), self._weights_version(), self.precision, self.fp32_tags, self.lstm_tc, self.fuse_pre_ftb,
                   self.snake, self.raw16, self.gin16)
            entry = self._graphs.get(key)
            if entry is None and self.use_graph == "auto":
                n = self._seen.get(key, 0)
                if n < 2:
                    if len(self._seen) >= 64:
                        self._seen.clear()
                    self._seen[key] = n + 1
                    return self._forward(mix, return_spec, return_lr_spec)
            if entry is None:
                static_in = mix.contiguous().clone()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(2):                   # allocate workspaces / pack weights / encode tensor maps outside capture
                        self._forward(static_in, False, False)
                torch.cuda.current_stream().wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    static_out = self._forward(static_in, False, False)
                for gk in [gk for gk in self._graphs if gk[1] != key[1]]:     # graphs of superseded weights
                    del self._graphs[gk]
                entry = self._graphs[key] = (graph, static_in, static_out)
            else:
                self._select_shape_set((key[0], self.precision))   # keep the replayed shape's workspaces most recently used
            graph, static_in, static_out = entry
            static_in.copy_(mix)
            graph.replay()
            return static_out.clone()

    def _check_mode(self):
        if self.model.training:
            raise NotImplementedError(
                "aero_b200: the CUDA path implements the inference forward (eval-mode BatchNorm, no autograd); "
                "call model.eval().  Training kernels are SURVEY.md section 8f 'next'.")

    @torch.no_grad()
    def _forward(self, mix, return_spec=False, return_lr_spec=False):
        self._require(mix)
        self._check_mode()
        g = self.geom
        kw = g.kw
        if mix.dim() != 3 or mix.shape[1] != kw["in_channels"]:
            raise ValueError(f"expected input [B, {kw['in_channels']}, L], got {tuple(mix.shape)}")
        if mix.shape[0] == 0:
            # an empty batch maps to an empty batch (clips are independent); nothing to launch
            hop = g.hop_in
            Lp = mix.shape[2] + (-mix.shape[2]) % hop
            Tn, Fq0 = 1 + Lp // hop, g.nfft // 2
            y0 = mix.new_zeros(0, kw["out_channels"], min(int(mix.shape[2] * g.scale), g.hop_out * (Tn - 1)))
            if not return_spec:
                return y0
            zc0 = torch.zeros(0, kw["out_channels"], Fq0, Tn, dtype=torch.complex64, device=mix.device)
            if not return_lr_spec:
                return y0, zc0
            return y0, zc0, torch.zeros(0, kw["in_channels"], Fq0, Tn, dtype=torch.complex64, device=mix.device)
        W = self._weights()
        self._select_shape_set((tuple(mix.shape), self.precision))
        B_ = mix.shape[0]
        need = B_ + sum((2 * B_ * kw["norm_groups"] if lg.norm else 0) * 2 +
                        (2 * abs(kw["dconv_depth"]) * B_ * lg.f_out if lg.dconv else 0) for lg in g.layers) + 64
        if self._stats is None or self._stats.buf.device != mix.device or self._stats.buf.shape[0] < need:
            self._stats = _Stats(mix.device, capacity=max(1 << 16, need))
            self._graphs.clear()             # captured graphs point into the statistics buffer that was just replaced
            self._seen.clear()
        self._stats.reset()

        B, Cin, length = mix.shape
        x = mix.contiguous()
        if length % g.hop_in:
            x = torch.nn.functional.pad(x, (0, g.hop_in - length % g.hop_in))
        Lp = x.shape[-1]
        T = 1 + Lp // g.hop_in
        Fq = g.nfft // 2
        C2 = 2 * Cin

        # STFT straight into channels-last [B, F, T, 2*Cin]; channel 2c+{0,1} = {re,im} (aero.py:430-434)
        # (rows of T*C2 floats padded to 16 bytes so that TMA can address them: the pad is zero and never read as data)
        zrow = _pad4(T * C2)
        z = self._buf("z", B, Fq, zrow, zero=True)
        st_in = self._stats.take(B)
        self.stft_into(x.view(B * Cin, Lp), z, st_in, n_fft=g.nfft, hop=g.hop_in, win=g.win_in, channels=Cin,
                       bins_out=Fq, strides=(Fq * zrow, 2, zrow, C2))
        xn = self._buf("xn", B, Fq, zrow)
        affine = self._buf("affine", B, 2)
        self._sample_norm(z, st_in, xn, affine, B, Fq * T * C2, extent=Fq * zrow)
        xr = None
        l0 = g.layers[0]
        if self.precision >= 1 and l0.ftb and self.fuse_pre_ftb:
            xr = self._buf("xnr", B, Fq, zrow)        # TF32-rounded copy: the tensor-core operand of the frequency mix
            self._sample_norm(z, st_in, xr, affine, B, Fq * T * C2, extent=Fq * zrow, rnd=True)
        h = xn
        saved = []
        for lg in g.layers:
            h = self._encode(h, W, lg, B, T, xr=xr if lg.index == 0 else None)
            saved.append(h)
        h = None
        for j, lg in enumerate(reversed(g.layers)):
            last = lg.index == 0
            h = self._decode(h, saved.pop(), W, lg, j, B, T, last, affine)
        Cout = kw["out_channels"]
        assert h.shape == (B, Fq, T, 2 * Cout), (h.shape, (B, Fq, T, 2 * Cout))

        out_len = min(int(length * g.scale), g.hop_out * (T - 1))
        y = torch.empty(B * Cout, out_len, dtype=torch.float32, device=mix.device)
        self.istft_into(h, y, n_fft=g.nfft, hop=g.hop_out, win=g.win_out, channels=Cout, frames=T, bins_in=Fq,
                        strides=(Fq * T * 2 * Cout, 2, T * 2 * Cout, 2 * Cout))
        y = y.view(B, Cout, out_len)
        if not return_spec:
            return y
        zc = torch.view_as_complex(h.clone().view(B, Fq, T, Cout, 2)).permute(0, 3, 1, 2)
        if not return_lr_spec:
            return y, zc
        zl = torch.view_as_complex(z[:, :, :T * C2].reshape(B, Fq, T, Cin, 2)).permute(0, 3, 1, 2)
        return y, zc, zl
