"""One-time repack of a reference ``state_dict`` into the device layouts libdvd_b200 expects.

Key names are the reference's own (SURVEY.md §8(b)); DiT blocks 0..10 are accepted and ignored
(dead compute, cross_model.py:614-616).  Repacking is load-time plumbing done with torch ops on
the target device; nothing here runs per step.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

LIVE_BLOCK = 11
BN_EPS = 1e-5      # torch BatchNorm2d default used by mmcv ConvModule (cross_attn.py:24-50)

PYR_KEYS = ["pyramid.level_0.0", "pyramid.level_1.0", "pyramid.level_2.0", "pyramid.level_2.2",
            "pyramid.level_3.0", "pyramid.level_3.2", "pyramid.level_3.4"]
EMB_KEYS = ["obs", "r", "c", "m", "l"]


def required_keys():
    """Keys the live path needs (a subset of the reference state dict)."""
    ks = ["noised_obs_pos_embed"]
    for p in PYR_KEYS:
        ks += [p + ".weight", p + ".bias"]
    for e in EMB_KEYS:
        ks += [f"{e}_embedder.proj.weight", f"{e}_embedder.proj.bias"]
    ks += [f"t_embedder.mlp.{i}.{x}" for i in (0, 2) for x in ("weight", "bias")]
    b = f"blocks.{LIVE_BLOCK}."
    ks += [b + s for s in ("attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias", "mlp.fc1.weight",
                           "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias", "adaLN_modulation.1.weight",
                           "adaLN_modulation.1.bias", "cross_attn.in_proj_weight", "cross_attn.in_proj_bias",
                           "cross_attn.out_proj.weight", "cross_attn.out_proj.bias")]
    pd = "decoder.position_dec."
    ks += [pd + "h_position_encoder", pd + "w_position_encoder"]
    ks += [pd + f"{hw}_scale.{i}.{x}" for hw in "hw" for i in (0, 2) for x in ("weight", "bias")]
    for i in range(6):
        p = f"decoder.layer_stack.{i}."
        ks += [p + s for s in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "attn.linear_q.weight",
                               "attn.linear_k.weight", "attn.linear_v.weight", "attn.fc.weight")]
        for n in ("conv1", "depthwise_conv", "conv2"):
            ks += [p + f"feed_forward.{n}.conv.weight"] + [p + f"feed_forward.{n}.bn.{x}" for x in
                                                           ("weight", "bias", "running_mean", "running_var")]
    ks += ["decoder.layer_norm.weight", "decoder.layer_norm.bias", "final_layer2.linear.weight", "final_layer2.linear.bias",
           "final_layer2.adaLN_modulation.1.weight", "final_layer2.adaLN_modulation.1.bias"]
    return ks


def split_bf16(w: torch.Tensor):
    """fp32 -> (hi, lo) bf16 pair with hi = bf16(w), lo = bf16(w - hi): the operands of the 3-pass split-precision GEMM."""
    hi = w.to(torch.bfloat16)
    lo = (w - hi.float()).to(torch.bfloat16)
    return hi.contiguous(), lo.contiguous()


def split_f16(w: torch.Tensor):
    """fp32 -> (hi, lo) IEEE fp16 pair (weights of the GEMMs whose activation operand is a single fp16 value)."""
    if float(w.abs().max()) >= 65504.0:
        raise ValueError("weight magnitude exceeds the fp16 range")
    hi = w.to(torch.float16)
    lo = (w - hi.float()).to(torch.float16)
    return hi.contiguous(), lo.contiguous()


class PackedWeights:
    """Owns the packed device tensors and the ``dvd_weights_t`` table that points into them."""

    def __init__(self, sd: dict, device: torch.device, with_bf16: bool = True):
        self.device = device
        self.keep = []                      # keeps every packed tensor alive
        self.table = _lib.Weights()
        self.with_bf16 = with_bf16
        self.tables_cache = {}              # conditioning tables per step plan: they depend on these weights and die with them
        missing = [k for k in required_keys() if k not in sd]
        if missing:
            raise KeyError(f"state_dict is missing {len(missing)} live keys, e.g. {missing[:4]}")
        self._pack(sd)

    # -- helpers
    def _dev(self, t: torch.Tensor) -> torch.Tensor:
        t = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
        self.keep.append(t)
        return t

    def _vec(self, t):
        return C.c_void_p(self._dev(t).data_ptr())

    def _mat(self, w2d: torch.Tensor, bf16: bool = True, lo: bool = True) -> _lib.Mat:
        """fp32 W, plus bf16(W) for the tensor modes when ``bf16``, plus bf16(W - bf16(W)) when ``lo`` (the matrices bf16x3 runs on
        bf16 pairs)."""
        w = self._dev(w2d)
        m = _lib.Mat()
        m.f32 = w.data_ptr()
        m.n, m.k = int(w.shape[0]), int(w.shape[1])
        if bf16 and self.with_bf16:
            h, l = split_bf16(w)
            self.keep += [h, l] if lo else [h]
            m.bf16, m.bf16_lo = h.data_ptr(), (l.data_ptr() if lo else None)
        return m

    def _ln_fold(self, w64: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, f16: bool = False):
        """W' = W * gamma as a 16-bit pair (bf16, or IEEE fp16 for the two-pass q|k|v GEMM), the column sums of the ROUNDED pair, W beta."""
        wp = (w64 * gamma.double()[None, :]).float()
        m = self._mat(wp, bf16=not f16)
        if f16:
            h16, l16 = split_f16(self.keep[-1])                    # (the fp32 copy _mat just made)
            self.keep += [h16, l16]
            m.bf16, m.bf16_lo = h16.data_ptr(), l16.data_ptr()
        hi, lo = self.keep[-2], self.keep[-1]                      # the pair that is used
        colsum = (hi.double() + lo.double()).sum(1).float()
        cvec = (w64 @ beta.double()).float()
        return m, self._vec(colsum), self._vec(cvec)

    def _bn(self, sd, prefix):
        w, b = sd[prefix + "bn.weight"].float(), sd[prefix + "bn.bias"].float()
        mu, var = sd[prefix + "bn.running_mean"].float(), sd[prefix + "bn.running_var"].float()
        scale = w / torch.sqrt(var + BN_EPS)
        return self._vec(scale), self._vec(b - mu * scale)

    def _pack(self, sd):
        T = self.table
        T.pos = self._vec(sd["noised_obs_pos_embed"].reshape(1024, 384))
        for i, p in enumerate(PYR_KEYS):
            w = sd[p + ".weight"].float()
            wk = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(self.device)    # [Cout, Cin, 3, 3] -> [Cout, ky, kx, Cin]
            T.pyr[i] = self._mat(wk, bf16=(i > 0), lo=False)                # bf16 reads the hi; bf16x3 reads pyr_h
            if self.with_bf16:
                w2 = wk
                if i == 0:                                                  # level_0: K = 36 zero-padded to 64 for the tcgen05 im2col GEMM
                    w2 = torch.nn.functional.pad(wk, (0, 64 - wk.shape[1]))
                    h = w2.to(torch.bfloat16).contiguous()
                    self.keep.append(h)
                    T.pyr[0].bf16 = h.data_ptr()
                h16, l16 = split_f16(w2)                                    # the same matrices as fp16 pairs (two-pass pyramid of bf16x3)
                self.keep += [h16, l16]
                T.pyr_h[i].f32, T.pyr_h[i].bf16, T.pyr_h[i].bf16_lo = T.pyr[i].f32, h16.data_ptr(), l16.data_ptr()
                T.pyr_h[i].n, T.pyr_h[i].k = int(w2.shape[0]), int(w2.shape[1])
            T.pyr_b[i] = self._vec(sd[p + ".bias"])
        for i, e in enumerate(EMB_KEYS):
            w = sd[f"{e}_embedder.proj.weight"].float()
            T.emb[i] = self._mat(w.reshape(w.shape[0], -1), bf16=(i > 0))   # k = c*4 + p*2 + q (conv weight order)
            T.emb_b[i] = self._vec(sd[f"{e}_embedder.proj.bias"])
        T.t_mlp0 = self._mat(sd["t_embedder.mlp.0.weight"], bf16=False); T.t_mlp0_b = self._vec(sd["t_embedder.mlp.0.bias"])
        T.t_mlp2 = self._mat(sd["t_embedder.mlp.2.weight"], bf16=False); T.t_mlp2_b = self._vec(sd["t_embedder.mlp.2.bias"])
        b = f"blocks.{LIVE_BLOCK}."
        T.blk_ada = self._mat(sd[b + "adaLN_modulation.1.weight"], bf16=False); T.blk_ada_b = self._vec(sd[b + "adaLN_modulation.1.bias"])
        T.xattn_in = self._mat(sd[b + "cross_attn.in_proj_weight"]); T.xattn_in_b = self._vec(sd[b + "cross_attn.in_proj_bias"])
        T.xattn_out = self._mat(sd[b + "cross_attn.out_proj.weight"]); T.xattn_out_b = self._vec(sd[b + "cross_attn.out_proj.bias"])
        T.blk_qkv = self._mat(sd[b + "attn.qkv.weight"]); T.blk_qkv_b = self._vec(sd[b + "attn.qkv.bias"])
        T.blk_proj = self._mat(sd[b + "attn.proj.weight"]); T.blk_proj_b = self._vec(sd[b + "attn.proj.bias"])
        T.blk_fc1 = self._mat(sd[b + "mlp.fc1.weight"]); T.blk_fc1_b = self._vec(sd[b + "mlp.fc1.bias"])
        T.blk_fc2 = self._mat(sd[b + "mlp.fc2.weight"]); T.blk_fc2_b = self._vec(sd[b + "mlp.fc2.bias"])
        pd = "decoder.position_dec."
        T.dec_hpe = self._vec(sd[pd + "h_position_encoder"].reshape(1536, 32).t())     # -> [32, 1536]
        T.dec_wpe = self._vec(sd[pd + "w_position_encoder"].reshape(1536, 32).t())
        for hw in "hw":
            for j in (0, 2):
                setattr(T, f"{hw}_scale{j}", self._mat(sd[pd + f"{hw}_scale.{j}.weight"].reshape(1536, 1536), bf16=False))
                setattr(T, f"{hw}_scale{j}_b", self._vec(sd[pd + f"{hw}_scale.{j}.bias"]))
        for i in range(6):
            p = f"decoder.layer_stack.{i}."
            L = T.dec[i]
            L.n1_w, L.n1_b = self._vec(sd[p + "norm1.weight"]), self._vec(sd[p + "norm1.bias"])
            L.n2_w, L.n2_b = self._vec(sd[p + "norm2.weight"]), self._vec(sd[p + "norm2.bias"])
            L.qkv = self._mat(torch.cat([sd[p + "attn.linear_q.weight"], sd[p + "attn.linear_k.weight"],
                                         sd[p + "attn.linear_v.weight"]], 0), lo=False)          # bf16x3 reads qkv_ln
            L.fc = self._mat(sd[p + "attn.fc.weight"])
            f = p + "feed_forward."
            L.conv1 = self._mat(sd[f + "conv1.conv.weight"].reshape(2048, 1536), lo=False)         # bf16x3 reads conv1_ln
            L.bn1_scale, L.bn1_shift = self._bn(sd, f + "conv1.")
            L.dw_w = self._vec(sd[f + "depthwise_conv.conv.weight"].reshape(2048, 9).t())   # tap-major [9, 2048]
            L.bn2_scale, L.bn2_shift = self._bn(sd, f + "depthwise_conv.")
            L.conv2 = self._mat(sd[f + "conv2.conv.weight"].reshape(1536, 2048))
            L.bn3_scale, L.bn3_shift = self._bn(sd, f + "conv2.")
            if self.with_bf16:
                # LayerNorm folded into the consumer GEMMs (fused-LN epilogue, csrc/gemm_pair.cu): W' = W * gamma, colsum of the ROUNDED
                # pair, cvec = W beta (float64 sums)
                wq = torch.cat([sd[p + "attn.linear_q.weight"], sd[p + "attn.linear_k.weight"], sd[p + "attn.linear_v.weight"]], 0).double()
                L.qkv_ln, L.qkv_colsum, L.qkv_cvec = self._ln_fold(wq, sd[p + "norm1.weight"], sd[p + "norm1.bias"], f16=True)
                wc = sd[f + "conv1.conv.weight"].reshape(2048, 1536).double()
                L.conv1_ln, L.conv1_colsum, L.conv1_cvec = self._ln_fold(wc, sd[p + "norm2.weight"], sd[p + "norm2.bias"])
        T.dec_ln_w, T.dec_ln_b = self._vec(sd["decoder.layer_norm.weight"]), self._vec(sd["decoder.layer_norm.bias"])
        T.fin = self._mat(sd["final_layer2.linear.weight"], bf16=False); T.fin_b = self._vec(sd["final_layer2.linear.bias"])
        T.fin_ada = self._mat(sd["final_layer2.adaLN_modulation.1.weight"], bf16=False)
        T.fin_ada_b = self._vec(sd["final_layer2.adaLN_modulation.1.bias"])

    def ref(self):
        return C.byref(self.table)
