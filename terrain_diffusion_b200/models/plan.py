"""Launch planner: turns an EDMUnet2D (reference: terrain_diffusion/models/edm_unet.py:67-184) into a libtdx Program.

The reference evaluates ~6 500 ATen ops per forward (weight re-normalisation, pixel-norm, mp_silu, mp_sum, mp_concat,
resample, clip around 96 convolutions).  Here every UNetBlock (models/unet_block.py:116-156) becomes two launches of the
tcgen05 implicit-GEMM kernel (three for encoder blocks with a 1x1 skip) whose epilogues carry all of that:

  enc block   [K1: 1x1 skip -> pixel-norm -> (x_n, mp_silu(x_n))]                         (only if Cin != Cout)
              res0: conv3x3(a) -> mp_silu(y * c)                                          (c = embedding modulation)
              res1: conv3x3(h)*t/n + (1-t)/n * pixelnorm(x) -> clip -> outputs
  dec block   res0: conv3x3 over K-slabs [mp_silu(s1*x) | mp_silu(s2*skip)] -> mp_silu(y * c)
              res1: one GEMM over K-slabs [h (3x3) | x (1x1 skip) | skip (1x1 skip)] with mp_sum / mp_concat constants
                    folded into the weights -> clip -> outputs          (or residual add when there is no skip conv)

"outputs" = what the consumers need, written by the producer's epilogue: the raw block output (skip connection /
residual / 1x1 K-slab), the next block's activated input (mp_silu, or pixel-norm + mp_silu, optionally stride-2
sub-sampled or nearest-x2 up-sampled) and the decoder-side activated skip.  Weights are normalised/folded ONCE here
(the reference redoes it every forward, mp_layers.py:203-213).
"""
from __future__ import annotations

import ctypes as C
import os
import math

import numpy as np
import torch

from .. import _lib as L
from ..layout import pack_weight_segments


_TUNED = None
_TUNED_NEW: dict = {}      # shapes measured in this process (TDX_AUTOTUNE=1); tools/tune_igemm.py writes them out
_TUNE_CANDIDATES: dict = {}   # TDX_AUTOTUNE=2: valid (N, k_split) per shape key, in program order
TUNED_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tuned_shapes.json")


def tuned_shapes() -> dict:
    """{"cout|n|h|w|segments|norm": [n_per_item, k_split]} measured on a B200 (tools/tune_igemm.py)."""
    global _TUNED
    if _TUNED is None:
        _TUNED = {}
        if os.environ.get("TDX_TUNED_TABLE", "1") != "0":
            try:
                import json
                with open(TUNED_PATH) as f:
                    _TUNED = dict(json.load(f).get("shapes", {}))
            except Exception:
                _TUNED = {}
    return _TUNED


def effective_weight(w: torch.Tensor, gain=1.0) -> torch.Tensor:
    """fp32 weight MPConv.forward convolves with (mp_layers.py:203-213): global-RMS normalise, gain / sqrt(fan_in)."""
    w = w.detach().to(torch.float32)
    norm = torch.linalg.vector_norm(w)
    norm = torch.add(1e-4, norm, alpha=np.sqrt(1.0 / w.numel()))
    w = w / norm
    if isinstance(gain, torch.Tensor):
        gain = gain.detach().to(torch.float32)
    return w * (gain / np.sqrt(w[0].numel()))


def mp_concat_scales(n_a: int, n_b: int, t: float) -> tuple[float, float]:
    """Per-tensor scalars of mp_concat (mp_layers.py:65-86)."""
    c = math.sqrt((n_a + n_b) / ((1 - t) ** 2 + t ** 2))
    return c / math.sqrt(n_a) * (1 - t), c / math.sqrt(n_b) * t


def block_plan(cfg: dict) -> tuple[list, list]:
    """Module order / shapes of EDMUnet2D.__init__ (edm_unet.py:105-137)."""
    mults = cfg.get("model_channel_mults") or [1, 2, 3, 4]
    mc = cfg.get("model_channels", 128)
    lpb = cfg.get("layers_per_block", 2)
    if isinstance(lpb, int):
        lpb = [lpb] * len(mults)
    attn_res = cfg.get("attn_resolutions") or []
    image_size = cfg["image_size"]
    chans = [mc * m for m in mults]
    enc, dec = [], []
    cout = cfg["in_channels"] + 1
    for level, (ch, nb) in enumerate(zip(chans, lpb)):
        res = image_size // 2 ** level
        if level == 0:
            enc.append(dict(name=f"{res}x{res}_conv", kind="conv", cin=cout, cout=ch))
            cout = ch
        else:
            enc.append(dict(name=f"{res}x{res}_down", kind="block", mode="enc", resample="down", cin=cout, cout=cout,
                            attention=False))
        for idx in range(nb):
            enc.append(dict(name=f"{res}x{res}_block{idx}", kind="block", mode="enc", resample="keep", cin=cout,
                            cout=ch, attention=(res in attn_res)))
            cout = ch
    skips = [b["cout"] for b in enc]
    if not cfg.get("encode_only", False):
        for level, (ch, nb) in reversed(list(enumerate(zip(chans, lpb)))):
            res = image_size // 2 ** level
            if level == len(chans) - 1:
                dec.append(dict(name=f"{res}x{res}_in0", kind="block", mode="dec", resample="keep", cin=cout,
                                cout=cout, attention=bool(cfg.get("midblock_attention", True)), concat=False))
                dec.append(dict(name=f"{res}x{res}_in1", kind="block", mode="dec", resample="keep", cin=cout,
                                cout=cout, attention=False, concat=False))
            else:
                dec.append(dict(name=f"{res}x{res}_up", kind="block", mode="dec", resample="up", cin=cout, cout=cout,
                                attention=False, concat=False))
            for idx in range(nb + 1):
                sk = skips.pop()
                dec.append(dict(name=f"{res}x{res}_block{idx}", kind="block", mode="dec", resample="keep",
                                cin=cout + sk, cout=ch, attention=(res in attn_res), concat=True, skip_channels=sk))
                cout = ch
    return enc, dec


class FoldedWeights:
    """Device-resident effective weights of one model (fp32 small tensors + packed bf16 GEMM operands).

    The fold itself (normalise, gains, mp_sum / mp_concat constants, bf16 rounding, B-stage packing) is host arithmetic
    on the fp32 master weights, done once: the results are uploaded with plain copies, so creating a model puts no
    kernel on the device (the reference re-normalises 130 tensors with ~7 launches each on EVERY forward)."""

    def __init__(self, model, device):
        cfg = dict(model.config)
        sd = {k: v.detach().cpu().to(torch.float32) for k, v in model.state_dict().items()}
        dev_arg, device = device, torch.device("cpu")      # fold on the host; upload at the end of __init__
        self.cfg = cfg
        self.device = device
        enc, dec = block_plan(cfg)
        bk = cfg.get("block_kwargs") or {}
        for bad in ("conv_type", "resample_type", "activation", "no_padding", "expansion_factor"):
            if bk.get(bad) not in (None, "default", "pooling", "silu", False, 1):
                raise NotImplementedError(f"block_kwargs[{bad!r}]={bk[bad]!r} is not used by any shipped model and is "
                                          "not implemented by the B200 path")
        self.t_res = float(bk.get("res_balance", 0.3))
        self.clip = float(bk.get("clip_act", 256.0) or 0.0)
        self.cb = float(cfg.get("concat_balance", 0.3))
        self.enc, self.dec = enc, dec
        self.cph = int(bk.get("channels_per_head", 64))
        self.t_attn = float(bk.get("attn_balance", 0.3))
        for b in enc + dec:
            b["heads"] = (b["cout"] // self.cph) if b.get("attention") else 0
            if b["heads"] and self.cph != 64:
                raise NotImplementedError(f"attention block {b['name']}: channels_per_head={self.cph}; the B200 path "
                                          "implements the shipped value 64")
        self.mc = cfg.get("model_channels", 128)
        mults = cfg.get("model_channel_mults") or [1, 2, 3, 4]
        self.emb_channels = cfg.get("emb_channels") or self.mc * max(mults)
        self.noise_dims = self.mc if cfg.get("noise_emb_dims") is None else cfg["noise_emb_dims"]
        self.has_cond = bool(cfg.get("conditional_inputs"))
        self.pos_emb = cfg.get("fourier_scale", 1) == "pos"
        self.in_channels = cfg["in_channels"]
        self.out_channels = cfg.get("out_channels") or cfg["in_channels"]

        t = self.t_res
        nrm = math.sqrt((1 - t) ** 2 + t ** 2)
        self.w_res = t / nrm
        self.w_skip = (1 - t) / nrm

        # map each encoder output to the decoder block that consumes it as a skip
        idx = list(range(len(enc)))
        self.skip_consumer = {}
        for d in dec:
            if d.get("concat"):
                self.skip_consumer[idx.pop()] = d

        g: dict = {}
        self.g = g
        self.segs: dict = {}
        self._packed: dict = {}
        if self.noise_dims > 0:
            g["noise_linear"] = effective_weight(sd["noise_linear.weight"]).t().contiguous()  # [in][out]
            if self.pos_emb:
                g["noise_freqs"] = sd["noise_fourier.freqs"].contiguous()
        # conditional-input layers of compute_embeddings (edm_unet.py:145-159): folded once like everything else
        for i, (kind, _dim, _wgt) in enumerate(cfg.get("conditional_inputs") or []):
            if kind == "float":
                g[f"cond{i}"] = effective_weight(sd[f"conditional_layers.{i}.1.weight"]).t().contiguous()
            elif kind == "tensor":
                g[f"cond{i}"] = effective_weight(sd[f"conditional_layers.{i}.weight"]).t().contiguous()
            else:
                g[f"cond{i}"] = sd[f"conditional_layers.{i}.weight"].contiguous()      # MPEmbedding: un-normalised table
        first = enc[0]
        w_in = effective_weight(sd[f"enc.{first['name']}.weight"])               # [cout][ci][3][3]
        g["conv_in"] = w_in.permute(2, 3, 1, 0).reshape(9, w_in.shape[1], w_in.shape[0]).contiguous()  # [tap][ci][cout]
        # the same weights as the [cout][k_pad] matrix of the tensor-core path (tdx_im2col_run + 1x1 igemm):
        # k = tap * ci + c, zero-padded to a multiple of 64
        ci = w_in.shape[1]
        self.conv_in_kpad = ((9 * ci + 63) // 64) * 64
        w_mat = torch.zeros((w_in.shape[0], self.conv_in_kpad, 1, 1), dtype=torch.float32, device=device)
        w_mat[:, :9 * ci, 0, 0] = w_in.permute(0, 2, 3, 1).reshape(w_in.shape[0], 9 * ci)
        self.segs["conv_in.im2col"] = [w_mat]
        out_gain = sd["out_gain"] if "out_gain" in sd else 1.0
        w_out = effective_weight(sd["out_conv.weight"], gain=out_gain)                  # [cout<=8][c][3][3]
        wpad = 1 if w_out.shape[0] == 1 else 8
        w_out8 = torch.zeros((wpad, w_out.shape[1], 3, 3), dtype=torch.float32, device=device)
        w_out8[:w_out.shape[0]] = w_out
        g["conv_out"] = w_out8.permute(2, 3, 1, 0).reshape(9, w_out.shape[1], wpad).contiguous()    # [tap][c][1|8]
        for side, blocks in (("enc", enc), ("dec", dec)):
            for b in blocks:
                if b["kind"] != "block":
                    continue
                p = f"{side}.{b['name']}."
                if (p + "emb_linear.weight") in sd:
                    g[p + "emb"] = effective_weight(sd[p + "emb_linear.weight"],
                                                    gain=sd[p + "emb_gain"]).t().contiguous()  # [E][cout]
                w0 = effective_weight(sd[p + "conv_res0.weight"])
                w1 = effective_weight(sd[p + "conv_res1.weight"]) * self.w_res
                ws = effective_weight(sd[p + "conv_skip.weight"]) if (p + "conv_skip.weight") in sd else None
                # effective GEMM operands as bf16 segment lists; packed per launch shape by packed()
                seg = self.segs
                if b["heads"]:
                    # UNetBlock.attn (unet_block.py:102-108): qkv rows are (head, d, {q,k,v}) interleaved -> split into
                    # three [C, C] projections with channel = head*64 + d; mp_sum(attn_balance) folded into proj.
                    c = b["cout"]
                    wqkv = effective_weight(sd[p + "attn_qkv.weight"]).reshape(b["heads"], self.cph, 3, c, 1, 1)
                    for wi, nm in enumerate(("q", "k", "v")):
                        seg[p + nm] = [wqkv[:, :, wi].reshape(c, c, 1, 1).contiguous().bfloat16()]
                    ta = self.t_attn
                    na = math.sqrt((1 - ta) ** 2 + ta ** 2)
                    seg[p + "proj"] = [(effective_weight(sd[p + "attn_proj.weight"]) * (ta / na)).bfloat16()]
                if b["mode"] == "enc":
                    if ws is not None:
                        seg[p + "k1"] = [ws.bfloat16()]
                    seg[p + "res0"] = [w0.bfloat16()]
                    seg[p + "res1"] = [w1.bfloat16()]
                else:
                    if b.get("concat"):
                        cs = b["skip_channels"]
                        cx = b["cin"] - cs
                        s1, s2 = mp_concat_scales(cx, cs, self.cb)
                        seg[p + "res0"] = [w0[:, :cx].contiguous().bfloat16(), w0[:, cx:].contiguous().bfloat16()]
                        assert ws is not None
                        seg[p + "res1"] = [w1.bfloat16(), (ws[:, :cx] * (s1 * self.w_skip)).contiguous().bfloat16(),
                                           (ws[:, cx:] * (s2 * self.w_skip)).contiguous().bfloat16()]
                    else:
                        assert ws is None, "decoder block without concat but with a skip conv is not planned"
                        seg[p + "res0"] = [w0.bfloat16()]
                        seg[p + "res1"] = [w1.bfloat16()]
        self.device = dev_arg
        for k in list(g):
            g[k] = g[k].to(dev_arg)

    def packed(self, key: str, n_per_item: int) -> torch.Tensor:
        """bf16 B operand of GEMM `key` packed for work items of `n_per_item` output channels (cached)."""
        ck = (key, n_per_item)
        if ck not in self._packed:
            self._packed[ck] = pack_weight_segments([w.float() for w in self.segs[key]], n_per_item).to(self.device)
        return self._packed[ck]


class UNetProgram:
    """One compiled launch list (single forward, or a whole N-step solve) + the buffers it owns."""

    def __init__(self, device=None):
        import torch as _t
        self.device = _t.device("cuda", _t.cuda.current_device()) if device is None else _t.device(device)
        self.handle = C.c_void_p()
        L.check(L.lib().tdx_program_create(C.byref(self.handle)))
        self.keep: list = []
        self.arena: dict = {}
        self.n_igemm = 0
        self.n_launch = 0

    def run(self, use_graph: bool = True):
        L.call(L.lib().tdx_program_run, self.device, self.handle, 1 if use_graph else 0)

    def instantiate(self):
        L.call(L.lib().tdx_program_instantiate, self.device, self.handle)

    def profile(self):
        """Eager run with per-launch CUDA events: returns (ms list, kind list) in program order."""
        n = L.lib().tdx_program_num_launches(self.handle)
        ms = (C.c_float * n)()
        kinds = (C.c_int32 * n)()
        L.call(L.lib().tdx_program_profile, self.device, self.handle, ms, kinds)
        return list(ms), list(kinds)

    def __del__(self):
        try:
            if self.handle:
                L.lib().tdx_program_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass


class UNetEmitter:
    """Allocates the activation arena for (n, h, w) and appends the launches of one U-Net evaluation to a program."""

    def __init__(self, fw: FoldedWeights, n: int, h: int, w: int, cvec_sets: int = 1):
        """cvec_sets: how many independent label sets (e.g. solver steps) share this arena; the modulation vectors of
        all of them are produced by ONE embed launch (emit_embed) and selected per evaluation with `cvec_set`."""
        self.cvec_sets = cvec_sets
        levels = len(fw.cfg.get("model_channel_mults") or [1, 2, 3, 4])
        need = 8 * 2 ** (levels - 1)
        if h % need or w % need:
            raise ValueError(f"spatial size {h}x{w} must be a multiple of {need} for this model")
        self.fw, self.n, self.h, self.w = fw, n, h, w
        self.dev = fw.device
        # TDX_CONV_IN_DIRECT=1 selects the CUDA-core first convolution (fp32 inputs / weights) instead of im2col + igemm
        self.conv_in_direct = os.environ.get("TDX_CONV_IN_DIRECT") == "1"
        self.arena: dict = {}
        self.cvecs: dict = {}
        self.igemm_flops = 0          # sum of 2*M*N*K over the igemm launches this emitter has appended

    def act(self, key, c, h, w):
        if key not in self.arena:
            self.arena[key] = torch.empty((self.n, c // 8, h, w, 8), dtype=torch.bfloat16, device=self.dev)
        return self.arena[key]

    def cvec(self, key, c):
        if key not in self.cvecs:
            self.cvecs[key] = torch.ones((self.cvec_sets * self.n, c), dtype=torch.float32, device=self.dev)
        return self.cvecs[key]

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def _set_out(desc, i, tensor, kind, spatial=L.SP_SAME, scale=1.0):
        desc.out[i].ptr = tensor.data_ptr()
        desc.out[i].kind = kind
        desc.out[i].spatial = spatial
        desc.out[i].scale = scale

    def _next_spec(self, nxt, cur_c):
        """(kind, spatial, scale) of the activated tensor the next stage reads, or None if it only reads RAW."""
        if nxt is None:
            return None
        if nxt["mode"] == "enc":
            if nxt["cin"] != nxt["cout"]:
                return None
            return (L.OUT_PNORM_SILU, L.SP_DOWN2 if nxt["resample"] == "down" else L.SP_SAME, 1.0)
        if nxt.get("concat"):
            s1, _ = mp_concat_scales(cur_c, nxt["skip_channels"], self.fw.cb)
            return (L.OUT_SILU, L.SP_SAME, s1)
        return (L.OUT_SILU, L.SP_UP2 if nxt["resample"] == "up" else L.SP_SAME, 1.0)

    def _emit_outputs(self, desc, stage_key, c, h, w, nxt, enc_index):
        """Fill desc.out[] for a block output; returns dict(raw=, act=, skip_act=)."""
        res = {}
        res["raw"] = self.act(stage_key + ".raw", c, h, w)
        self._set_out(desc, 0, res["raw"], L.OUT_RAW)
        slot = 1
        spec = self._next_spec(nxt, c)
        if spec is not None:
            kind, spatial, scale = spec
            hh, ww = (h // 2, w // 2) if spatial == L.SP_DOWN2 else ((h * 2, w * 2) if spatial == L.SP_UP2 else (h, w))
            res["act"] = self.act(stage_key + ".act", c, hh, ww)
            self._set_out(desc, slot, res["act"], kind, spatial, scale)
            slot += 1
            if kind == L.OUT_PNORM_SILU and hasattr(desc, "rms_out"):
                # the consumer block adds pixelnorm(raw) as its residual: leave it the per-pixel factor (fp32 plane)
                key = stage_key + ".inv"
                if key not in self.arena:
                    self.arena[key] = torch.empty((self.n, h, w), dtype=torch.float32, device=self.dev)
                res["inv"] = self.arena[key]
                desc.rms_out = res["inv"].data_ptr()
        if enc_index is not None and enc_index in self.fw.skip_consumer:
            d = self.fw.skip_consumer[enc_index]
            cx = d["cin"] - d["skip_channels"]
            _, s2 = mp_concat_scales(cx, d["skip_channels"], self.fw.cb)
            res["skip_act"] = self.act(stage_key + ".skip_act", c, h, w)
            self._set_out(desc, slot, res["skip_act"], L.OUT_SILU, L.SP_SAME, s2)
            slot += 1
        return res

    def _igemm(self, prog, segs, wkey, cout, h, w):
        d = L.TdxIgemmDesc()
        for i, (tensor, ch, taps) in enumerate(segs):
            d.a_ptr[i] = tensor.data_ptr()
            d.a_channels[i] = ch
            d.a_taps[i] = taps
        d.n_seg = len(segs)
        n_item = L.igemm_choose_n(cout, self.n, h, w, [(ch, taps) for _, ch, taps in segs])
        d.n_per_item = n_item
        d.b_packed = self.fw.packed(wkey, n_item).data_ptr()
        d.c_out = cout
        d.n_img, d.height, d.width = self.n, h, w
        d._wkey = wkey          # (python-side attribute) lets _add_igemm re-pack for the tuned work-item width
        return d

    def _finish_block(self, prog, d, b, key, cout, h, w, nxt, enc_index):
        """Tail of UNetBlock.forward after conv_res1 (`d` = its launch, residual already configured):
        [x = mp_sum(x, attn(x))] ; clip ; write what the consumers need (unet_block.py:147-156)."""
        fw = self.fw
        if not b["heads"]:
            d.clip = fw.clip
            cur = self._emit_outputs(d, key, cout, h, w, nxt, enc_index)
            self._add_igemm(prog, d)
            return cur
        # ---- attention: x1 = mp_sum(x, y) un-clipped -> q, k, v (1x1) -> softmax core -> proj (1x1) + mp_sum + clip
        x1 = self.act(key + "x1", cout, h, w)
        d.clip = 0.0
        self._set_out(d, 0, x1, L.OUT_RAW)
        self._add_igemm(prog, d)
        qkv = []
        for nm in ("q", "k", "v"):
            t = self.act(key + nm, cout, h, w)
            dq = self._igemm(prog, [(x1, cout, 1)], key + nm, cout, h, w)
            self._set_out(dq, 0, t, L.OUT_RAW)
            self._add_igemm(prog, dq)
            qkv.append(t)
        yat = self.act(key + "attn_y", cout, h, w)
        ad = L.TdxAttnDesc()
        ad.q, ad.k, ad.v, ad.out = qkv[0].data_ptr(), qkv[1].data_ptr(), qkv[2].data_ptr(), yat.data_ptr()
        ad.n_img, ad.heads, ad.head_dim, ad.tokens = self.n, b["heads"], fw.cph, h * w
        L.check(L.lib().tdx_program_add_attn(prog.handle, C.byref(ad)))
        prog.n_launch += 1
        dp = self._igemm(prog, [(yat, cout, 1)], key + "proj", cout, h, w)
        ta = fw.t_attn
        dp.epi_flags = L.EPI_RESID
        dp.resid = x1.data_ptr()
        dp.resid_spatial = L.SP_SAME
        dp.resid_scale = (1 - ta) / math.sqrt((1 - ta) ** 2 + ta ** 2)
        dp.clip = fw.clip
        cur = self._emit_outputs(dp, key, cout, h, w, nxt, enc_index)
        self._add_igemm(prog, dp)
        return cur

    def _add_igemm(self, prog, d):
        self._apply_tuned_shape(d)
        L.check(L.lib().tdx_program_add_igemm(prog.handle, C.byref(d)))
        k = sum(d.a_channels[i] * d.a_taps[i] for i in range(d.n_seg))
        self.igemm_flops += 2 * d.n_img * d.height * d.width * d.c_out * k
        prog.n_igemm += 1
        prog.n_launch += 1

    # ------------------------------------------------------------------ measured (n_per_item, k_split) per launch shape
    @staticmethod
    def _shape_key(d) -> str:
        norm = bool(d.epi_flags & L.EPI_PNORM) or bool(d.rms_out) or any(d.out[o].kind == L.OUT_PNORM_SILU
                                                                        for o in range(3))
        segs = ";".join(f"{d.a_channels[i]}x{d.a_taps[i]}" for i in range(d.n_seg))
        return f"{d.c_out}|{d.n_img}|{d.height}|{d.width}|{segs}|{int(norm)}"

    def _apply_tuned_shape(self, d):
        """Work-item width N and split-K factor of this launch: from the measured table (tuned_shapes.json, produced on
        a B200 by tools/tune_igemm.py: the library's cost model is only the fallback), or measured now when
        TDX_AUTOTUNE=1.  The table is a file, not a run-time search, so every process / rank makes the same choice and
        multi-GPU results stay bit-identical to single-GPU ones."""
        wkey = getattr(d, "_wkey", None)
        if wkey is None:
            return
        key = self._shape_key(d)
        choice = tuned_shapes().get(key)
        if os.environ.get("TDX_AUTOTUNE") == "2" and key not in _TUNE_CANDIDATES:
            _TUNE_CANDIDATES[key] = self._valid_shapes(d, wkey)       # tools/tune_igemm.py graph mode
        if choice is None and os.environ.get("TDX_AUTOTUNE") == "1":
            choice = self._measure_shape(d, wkey)
            if choice is not None:
                tuned_shapes()[key] = choice
                _TUNED_NEW[key] = choice
        if choice is None:
            return
        n_item, ks = int(choice[0]), int(choice[1])
        if d.c_out % n_item:
            return
        d.n_per_item = n_item
        d.b_packed = self.fw.packed(wkey, n_item).data_ptr()
        d.k_split = ks

    def _valid_shapes(self, d, wkey):
        """Every (N, k_split) this launch accepts (one trial launch each)."""
        lib = L.lib()
        out = []
        keep = (d.n_per_item, d.b_packed, d.k_split)
        with torch.cuda.device(self.dev):
            stream = L.current_stream_ptr(self.dev)
            for n_item in (64, 128, 192, 256):
                if d.c_out % n_item or n_item > d.c_out:
                    continue
                d.n_per_item = n_item
                d.b_packed = self.fw.packed(wkey, n_item).data_ptr()
                for ks in (1, 2, 3, 4, 6, 8):
                    d.k_split = ks
                    if lib.tdx_igemm_run(C.byref(d), stream) == 0:
                        out.append([n_item, ks])
            torch.cuda.synchronize()
        d.n_per_item, d.b_packed, d.k_split = keep
        return out

    def _measure_shape(self, d, wkey):
        """Time every valid (N, k_split) of this launch: median of 5 x 12 back-to-back dependent launches each."""
        lib = L.lib()
        best, best_t = None, float("inf")
        keep = (d.n_per_item, d.b_packed, d.k_split)
        with torch.cuda.device(self.dev):
            stream = L.current_stream_ptr(self.dev)
            for n_item in (64, 128, 192, 256):
                if d.c_out % n_item or n_item > d.c_out:
                    continue
                d.n_per_item = n_item
                d.b_packed = self.fw.packed(wkey, n_item).data_ptr()
                for ks in (1, 2, 3, 4, 6, 8):
                    d.k_split = ks
                    if lib.tdx_igemm_run(C.byref(d), stream) != 0:
                        continue
                    ts = []
                    for _ in range(5):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(12):
                            lib.tdx_igemm_run(C.byref(d), stream)
                        e1.record()
                        torch.cuda.synchronize()
                        ts.append(e0.elapsed_time(e1))
                    t = sorted(ts)[len(ts) // 2]
                    if t < best_t:
                        best, best_t = (n_item, ks), t
        d.n_per_item, d.b_packed, d.k_split = keep
        return list(best) if best else None

    # ------------------------------------------------------------------ embedding / modulation vectors
    def emit_embed(self, prog: UNetProgram, labels=None, emb_in=None):
        # (planning allocates per-device library scratch and asks per-device questions: the model's device is current)
        with torch.cuda.device(self.dev):
            return self._emit_embed(prog, labels, emb_in)

    def _emit_embed(self, prog: UNetProgram, labels=None, emb_in=None):
        """One launch producing the modulation vectors c_b of every block for `cvec_sets * n` label rows.
        labels: fp32 [cvec_sets * n] device tensor, or emb_in: fp32 [cvec_sets * n, E] (host-computed embedding)."""
        fw = self.fw
        g = fw.g
        seq = [("enc", b) for b in fw.enc] + [("dec", b) for b in fw.dec]
        blocks = [(side, b) for side, b in seq if b["kind"] == "block" and f"{side}.{b['name']}.emb" in g]
        if not blocks:
            return
        rows = self.cvec_sets * self.n
        ed = L.TdxEmbedDesc()
        arr = (L.TdxEmbedBlock * len(blocks))()
        for i, (side, b) in enumerate(blocks):
            key = f"{side}.{b['name']}."
            arr[i].weight = g[key + "emb"].data_ptr()
            arr[i].cvec = self.cvec(key, b["cout"]).data_ptr()
            arr[i].c_out = b["cout"]
        if emb_in is not None:
            ed.emb_in = emb_in.data_ptr()
        else:
            if not (fw.pos_emb and fw.noise_dims > 0):
                raise ValueError("this model needs a host-computed embedding (emb_in)")
            assert labels.numel() == rows, (labels.shape, rows)
            ed.noise_labels = labels.data_ptr()
            ed.noise_weight = g["noise_linear"].data_ptr()
            ed.noise_freqs = g["noise_freqs"].data_ptr()
            ed.noise_dims = fw.noise_dims
        ed.emb_channels = fw.emb_channels
        ed.n_img = rows
        ed.n_blocks = len(blocks)
        ed.blocks = arr
        L.check(L.lib().tdx_program_add_embed(prog.handle, C.byref(ed)))
        prog.n_launch += 1
        prog.keep.append((labels, emb_in))

    def _cvec_ptr(self, key, c, cvec_set):
        return self.cvec(key, c).data_ptr() + cvec_set * self.n * c * 4

    # ------------------------------------------------------------------ one U-Net evaluation
    def emit(self, prog: UNetProgram, srcs, model_out=None, sched=None, cvec_set: int = 0):
        with torch.cuda.device(self.dev):
            return self._emit(prog, srcs, model_out, sched, cvec_set)

    def _emit(self, prog: UNetProgram, srcs, model_out=None, sched=None, cvec_set: int = 0):
        """srcs: [(tensor NCHW fp32/bf16, channels, scale_ptr_tensor or None)] (1 or 2 sources);
        model_out: fp32 [n, Cout, h, w] or None; sched: None or dict(coef=tensor[4], sample=tensor, x0_prev=tensor)
        or, for two-model guidance, dict(coef=tensor[5] {.., s}, sample=, x0_prev=, guide_out=fp32 [n, Cout, h, w]);
        cvec_set: which label set's modulation vectors (see emit_embed) this evaluation uses."""
        fw = self.fw
        g = fw.g
        n, dev = self.n, self.dev
        seq = [("enc", i, b) for i, b in enumerate(fw.enc)] + [("dec", i, b) for i, b in enumerate(fw.dec)]

        h, w = self.h, self.w
        cur = None
        skips = []
        for si, (side, idx, b) in enumerate(seq):
            nxt = seq[si + 1][2] if si + 1 < len(seq) else None
            key = f"{side}.{b['name']}."
            enc_index = idx if side == "enc" else None
            cout = b["cout"]
            if b["kind"] == "conv":
                cd = L.TdxConvInDesc()
                tot = 0
                for i, (tensor, ch, scale) in enumerate(srcs):
                    cd.src[i] = tensor.data_ptr()
                    cd.src_channels[i] = ch
                    cd.src_dtype[i] = 0 if tensor.dtype == torch.float32 else 1
                    cd.src_scale[i] = scale.data_ptr() if scale is not None else None
                    tot += ch
                assert tot + 1 == b["cin"], (tot, b["cin"])
                if self.conv_in_direct:
                    # CUDA-core first convolution (fp32 inputs and weights): kept for parity experiments
                    cd.weight = g["conv_in"].data_ptr()
                    cd.c_out = cout
                    cd.n_img, cd.height, cd.width = n, h, w
                    cur = self._emit_outputs(cd, key, cout, h, w, nxt, enc_index)
                    L.check(L.lib().tdx_program_add_conv_in(prog.handle, C.byref(cd)))
                    prog.n_launch += 1
                else:
                    # tensor-core first convolution: gather the 3x3 neighbourhoods (tdx_im2col_run), then a 1x1 igemm
                    im = L.TdxIm2colDesc()
                    for i in range(2):
                        im.src[i], im.src_channels[i] = cd.src[i], cd.src_channels[i]
                        im.src_dtype[i], im.src_scale[i] = cd.src_dtype[i], cd.src_scale[i]
                    kpad = fw.conv_in_kpad
                    cols = self.act(key + "im2col", kpad, h, w)
                    im.out = cols.data_ptr()
                    im.k_pad = kpad
                    im.n_img, im.height, im.width = n, h, w
                    L.check(L.lib().tdx_program_add_im2col(prog.handle, C.byref(im)))
                    prog.n_launch += 1
                    d = self._igemm(prog, [(cols, kpad, 1)], "conv_in.im2col", cout, h, w)
                    cur = self._emit_outputs(d, key, cout, h, w, nxt, enc_index)
                    self._add_igemm(prog, d)
            elif b["mode"] == "enc":
                resid_sp = L.SP_SAME
                if b["resample"] == "down":
                    h, w = h // 2, w // 2
                    resid_sp = L.SP_DOWN2
                if (key + "k1") in fw.segs:
                    d = self._igemm(prog, [(cur["raw"], b["cin"], 1)], key + "k1", cout, h, w)
                    d.epi_flags = L.EPI_PNORM
                    xn = self.act(key + "xn", cout, h, w)
                    a_in = self.act(key + "a0", cout, h, w)
                    self._set_out(d, 0, xn, L.OUT_RAW)
                    self._set_out(d, 1, a_in, L.OUT_SILU, L.SP_SAME, 1.0)
                    self._add_igemm(prog, d)
                    resid, resid_pn, resid_inv = xn, 0, None
                else:
                    a_in, resid, resid_pn = cur["act"], cur["raw"], 1
                    resid_inv = cur.get("inv")
                    if resid_inv is not None:
                        resid_pn = 0
                hbuf = self.act(key + "h", cout, h, w)
                d = self._igemm(prog, [(a_in, cout, 9)], key + "res0", cout, h, w)
                d.epi_flags = L.EPI_EMB_SILU
                d.cvec = self._cvec_ptr(key, cout, cvec_set)
                self._set_out(d, 0, hbuf, L.OUT_RAW)
                self._add_igemm(prog, d)
                d = self._igemm(prog, [(hbuf, cout, 9)], key + "res1", cout, h, w)
                d.epi_flags = L.EPI_RESID
                d.resid = resid.data_ptr()
                d.resid_spatial = resid_sp
                d.resid_pnorm = resid_pn
                if resid_inv is not None:
                    d.resid_inv = resid_inv.data_ptr()
                d.resid_scale = fw.w_skip
                cur = self._finish_block(prog, d, b, key, cout, h, w, nxt, enc_index)
            else:
                resid_sp = L.SP_SAME
                if b["resample"] == "up":
                    h, w = h * 2, w * 2
                    resid_sp = L.SP_UP2
                hbuf = self.act(key + "h", cout, h, w)
                if b.get("concat"):
                    sk = skips.pop()
                    cs = b["skip_channels"]
                    cx = b["cin"] - cs
                    segs0 = [(cur["act"], cx, 9), (sk["skip_act"], cs, 9)]
                else:
                    segs0 = [(cur["act"], b["cin"], 9)]
                d = self._igemm(prog, segs0, key + "res0", cout, h, w)
                d.epi_flags = L.EPI_EMB_SILU
                d.cvec = self._cvec_ptr(key, cout, cvec_set)
                self._set_out(d, 0, hbuf, L.OUT_RAW)
                self._add_igemm(prog, d)
                if b.get("concat"):
                    d = self._igemm(prog, [(hbuf, cout, 9), (cur["raw"], cx, 1), (sk["raw"], cs, 1)], key + "res1",
                                    cout, h, w)
                else:
                    d = self._igemm(prog, [(hbuf, cout, 9)], key + "res1", cout, h, w)
                    d.epi_flags = L.EPI_RESID
                    d.resid = cur["raw"].data_ptr()
                    d.resid_spatial = resid_sp
                    d.resid_scale = fw.w_skip
                cur = self._finish_block(prog, d, b, key, cout, h, w, nxt, None)
            if side == "enc":
                skips.append(cur)

        od = L.TdxConvOutDesc()
        od.x = cur["raw"].data_ptr()
        od.c_in = seq[-1][2]["cout"]
        od.weight = g["conv_out"].data_ptr()
        od.c_out = fw.out_channels
        od.n_img, od.height, od.width = n, h, w
        if model_out is not None:
            od.model_out = model_out.data_ptr()
        if sched is not None:
            od.sched_coef = sched["coef"].data_ptr()
            od.sample = sched["sample"].data_ptr()
            od.x0_prev = sched["x0_prev"].data_ptr()
        if sched is not None and sched.get("guide_out") is not None:
            gd = L.TdxConvOutGuidedDesc()
            gd.base = od
            gd.guide_out = sched["guide_out"].data_ptr()
            L.check(L.lib().tdx_program_add_conv_out_guided(prog.handle, C.byref(gd)))
        else:
            L.check(L.lib().tdx_program_add_conv_out(prog.handle, C.byref(od)))
        prog.n_launch += 1
        prog.keep.append((self.arena, self.cvecs, fw, srcs, model_out, sched))
        prog.arena = self.arena
