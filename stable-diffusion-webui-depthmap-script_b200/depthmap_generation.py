"""Depth estimation on B200 — drop-in for the hot-path part of the reference's ``src/depthmap_generation.py``.

``ModelHolder`` keeps the reference's public methods and attributes (src/depthmap_generation.py:40-403):
``update_settings``, ``ensure_models``, ``load_models``, ``get_default_net_size``, ``offload``, ``reload``,
``unload_models``, ``get_raw_prediction(input, net_width, net_height) -> (float32 [H,W], invert)``, plus the additive
``get_raw_prediction_batch`` (uint8 CUDA batch in, float32 CUDA batch out, no host sync) used by the batched funnel and
the bench.  The network forward is a sequence of C-ABI calls (tcgen05 GEMM / implicit-GEMM conv / fused attention /
LayerNorm / resize kernels, include/depthmap_b200.h); PyTorch only owns device memory and the stream.

Implemented model types: 0 (LeReS res101), 1, 2 (MiDaS 3.1 DPT-BEiT-L 512 / 384), 3 (MiDaS 3.0 DPT-Large 384), 7, 8, 9
(ZoeDepth-N, -K, -NK) and 12, 13, 14 (Depth-Anything-V2 S/B/L).  Others raise NotImplementedError naming the type.
Weights: a state_dict in the upstream checkpoint layout (``depth_anything_v2_vit{s,b,l}.pth``), packed once at load
into the kernels' layout (fp16 GEMM operands, (ky,kx,cin)-ordered conv filters, ConvTranspose as GEMM + pixel shuffle).
"""
from __future__ import annotations

import ctypes
import gc
import math
import os
import sys

import numpy as np

from . import _lib

DAV2_CONFIGS = {
    'vits': dict(embed_dim=384, depth=12, heads=6, features=64, out_channels=[48, 96, 192, 384], layers=[2, 5, 8, 11]),
    'vitb': dict(embed_dim=768, depth=12, heads=12, features=128, out_channels=[96, 192, 384, 768], layers=[2, 5, 8, 11]),
    'vitl': dict(embed_dim=1024, depth=24, heads=16, features=256, out_channels=[256, 512, 1024, 1024], layers=[4, 11, 17, 23]),
}


def _ru(x, m):
    return (x + m - 1) // m * m


def _constrain_to_multiple_of(x, multiple_of, min_val=0, max_val=None):
    y = int(np.round(x / multiple_of) * multiple_of)
    if max_val is not None and y > max_val:
        y = int(np.floor(x / multiple_of) * multiple_of)
    if y < min_val:
        y = int(np.ceil(x / multiple_of) * multiple_of)
    return y


def dav2_net_size(width, height, target, multiple_of=14):
    """Resize(keep_aspect_ratio, lower_bound, multiple of 14) of the reference (util/transform.py:61-104)."""
    sh, sw = target / height, target / width
    if sw > sh:
        sh = sw
    else:
        sw = sh
    return (_constrain_to_multiple_of(sw * width, multiple_of, min_val=target),
            _constrain_to_multiple_of(sh * height, multiple_of, min_val=target))


class _Ops:
    """Thin typed wrappers over the C-ABI; every method is asynchronous on the current torch stream."""

    def __init__(self):
        self.L = _lib.load()
        for name in ("dm_gemm_ex", "dm_conv3x3_ex", "dm_attention_f16", "dm_layernorm_f16"):
            if not hasattr(self.L, name):
                raise RuntimeError(f"depthmap_b200: native library lacks {name}; rebuild csrc (no fallback exists)")
        self.launches = 0

    def gemm(self, A, lda, W, ldw, M, N, K, epi=_lib.EPI_STORE_F16, act=_lib.ACT_NONE, bias=None, C=None, ldc=0, C2=None,
             R=None, ldr=0, R2=None, ldr2=0, X=None, ldx=0, gamma=None, head_b2=0.0, ps=None):
        d = _lib.GemmDesc()
        d.M, d.N, d.K, d.epi, d.act = M, N, K, epi, act
        d.bias = bias.data_ptr() if bias is not None else None
        d.C = C.data_ptr() if C is not None else None
        d.ldc = ldc
        d.C2 = C2.data_ptr() if C2 is not None else None
        d.R = R.data_ptr() if R is not None else None
        d.ldr = ldr
        d.R2 = R2.data_ptr() if R2 is not None else None
        d.ldr2 = ldr2
        d.X = X.data_ptr() if X is not None else None
        d.ldx = ldx
        d.gamma = gamma.data_ptr() if gamma is not None else None
        d.head_b2 = head_b2
        if ps is not None:
            d.ps_s, d.ps_cout, d.ps_h, d.ps_w = ps
        _lib.check(self.L.dm_gemm_ex(A.data_ptr(), lda, W.data_ptr(), ldw, ctypes.byref(d), _lib.stream_ptr()), "dm_gemm_ex")
        self.launches += 1

    def conv3x3(self, act_t, B, H, W_, Cin, Wt, Cout, epi=_lib.EPI_STORE_F16, act=_lib.ACT_NONE, bias=None, C=None, C2=None,
                R=None, R2=None, X=None, gamma=None, head_b2=0.0, ldx=1):
        d = _lib.GemmDesc()
        d.N, d.epi, d.act = Cout, epi, act
        d.bias = bias.data_ptr() if bias is not None else None
        d.C = C.data_ptr() if C is not None else None
        d.ldc = Cout
        d.C2 = C2.data_ptr() if C2 is not None else None
        d.R = R.data_ptr() if R is not None else None
        d.ldr = Cout
        d.R2 = R2.data_ptr() if R2 is not None else None
        d.ldr2 = Cout
        d.X = X.data_ptr() if X is not None else None
        d.ldx = ldx
        d.gamma = gamma.data_ptr() if gamma is not None else None
        d.head_b2 = head_b2
        _lib.check(self.L.dm_conv3x3_ex(act_t.data_ptr(), B, H, W_, Cin, Wt.data_ptr(), ctypes.byref(d), _lib.stream_ptr()), "dm_conv3x3_ex")
        self.launches += 1

    def attention(self, qkv, B, N, H, scale, out, bias=None, bias_ld=0):
        _lib.check(self.L.dm_attention_f16(qkv.data_ptr(), B, N, H, float(scale), bias.data_ptr() if bias is not None else None,
                                           bias_ld, out.data_ptr(), _lib.stream_ptr()), "dm_attention_f16")
        self.launches += 1

    def attention_relpos(self, qkv, B, gh, gw, H, scale, table, rowmax, nrd, out):
        _lib.check(self.L.dm_attention_relpos_f16(qkv.data_ptr(), B, gh, gw, H, float(scale), table.data_ptr(), rowmax.data_ptr(), nrd,
                                                  out.data_ptr(), _lib.stream_ptr()), "dm_attention_relpos_f16")
        self.launches += 1

    def layernorm(self, x, rows, C, w, b, out, tokens_per_img=1, drop_first=0, eps=1e-6):
        _lib.check(self.L.dm_layernorm_f16(x.data_ptr(), rows, C, w.data_ptr(), b.data_ptr(), eps, out.data_ptr(), tokens_per_img,
                                           drop_first, _lib.stream_ptr()), "dm_layernorm_f16")
        self.launches += 1

    def patchify(self, rgb, B, H, W, nh, nw, patch, mean, std, cmap, out, kpad):
        m = (ctypes.c_float * 3)(*mean)
        s = (ctypes.c_float * 3)(*std)
        c = (ctypes.c_int * 3)(*cmap)
        _lib.check(self.L.dm_preprocess_patchify(rgb.data_ptr(), B, H, W, nh, nw, patch, m, s, c, out.data_ptr(), kpad, _lib.stream_ptr()),
                   "dm_preprocess_patchify")
        self.launches += 2 if kpad > 3 * patch * patch else 1

    def tokens(self, pe, cls, pos, X, B, Np, C):
        _lib.check(self.L.dm_assemble_tokens(pe.data_ptr(), cls.data_ptr(), pos.data_ptr() if pos is not None else None, X.data_ptr(),
                                             B, Np, C, _lib.stream_ptr()), "dm_assemble_tokens")
        self.launches += 1

    def resize_nhwc(self, x, B, Hin, Win, C, out, Hout, Wout):
        _lib.check(self.L.dm_resize_bilinear_nhwc_f16(x.data_ptr(), B, Hin, Win, C, out.data_ptr(), Hout, Wout, _lib.stream_ptr()),
                   "dm_resize_bilinear_nhwc_f16")
        self.launches += 1

    def resize_f32(self, x, B, Hin, Win, out, Hout, Wout, mode):
        _lib.check(self.L.dm_resize_f32(x.data_ptr(), B, Hin, Win, out.data_ptr(), Hout, Wout, mode, _lib.stream_ptr()), "dm_resize_f32")
        self.launches += 1

    def im2col_s2(self, x, B, H, W, C, out):
        _lib.check(self.L.dm_im2col_s2_f16(x.data_ptr(), B, H, W, C, out.data_ptr(), _lib.stream_ptr()), "dm_im2col_s2_f16")
        self.launches += 1


def _conv_w(w, cin_pad, cout_pad):
    """[Cout, Cin, 3, 3] -> fp16 [cout_pad, 9*cin_pad], K ordered (ky, kx, cin)."""
    import torch
    co, ci = w.shape[:2]
    t = torch.zeros(cout_pad, 3, 3, cin_pad, dtype=torch.float16, device=w.device)
    t[:co, :, :, :ci] = w.permute(0, 2, 3, 1).to(torch.float16)
    return t.reshape(cout_pad, 9 * cin_pad).contiguous()


def _pad_vec(b, n):
    import torch
    t = torch.zeros(n, dtype=torch.float32, device=b.device)
    t[:b.numel()] = b.float().reshape(-1)
    return t


class DepthAnythingV2Engine:
    """Depth-Anything-V2 (DINOv2 ViT + DPT head) forward on the sm_100a kernels.

    Mirrors DepthAnythingV2.forward / DPTHead.forward / DINOv2.get_intermediate_layers of the reference
    (ddepth_anything_v2/depth_anything_v2/dpt.py:117-184, dinov2.py:297-321) plus image2tensor (dpt.py:196-221) and the
    final resize of estimatedepthanything_v2 (src/depthmap_generation.py:548-559).  Also the base of DptBeitEngine: the
    two families share the ViT block sequence and the whole DPT decoder and differ only in the hooks below."""

    PATCH = 14
    MEAN = (0.485, 0.456, 0.406)
    STD = (0.229, 0.224, 0.225)
    # the reference swaps R/B three times before the network sees the image (src/depthmap_generation.py:381,550; dpt.py:213):
    # network channel c carries source channel 2-c
    CHAN_MAP = (2, 1, 0)
    FINAL_RESIZE_MODE = 0  # bilinear, align_corners=True (src/depthmap_generation.py:558)
    CONFIGS = DAV2_CONFIGS

    def __init__(self, state_dict, encoder, device):
        import torch
        self.cfg = self.CONFIGS[encoder]
        self.encoder = encoder
        self.device = device
        self.ops = _Ops()
        self._buf_key = None
        self._bufs = {}
        self._pos_cache = {}
        self.probe = None  # bench hook: {'fc1': (start_event, end_event)} records the block-0 fc1 GEMM launch
        self._pack(state_dict)

    # ---- weight packing --------------------------------------------------------------------------------------------
    def _pack(self, sd):
        import torch
        dev = self.device
        cfg = self.cfg
        C, Fch, oc = cfg['embed_dim'], cfg['features'], cfg['out_channels']
        f16 = lambda t: t.detach().to(dev, torch.float16).contiguous()
        f32 = lambda t: t.detach().to(dev, torch.float32).contiguous()
        w = {}
        pw = sd['pretrained.patch_embed.proj.weight'].detach().to(dev).reshape(C, -1)
        self.kpad = _ru(pw.shape[1], 64)
        t = torch.zeros(C, self.kpad, dtype=torch.float16, device=dev)
        t[:, :pw.shape[1]] = pw.to(torch.float16)
        w['pe_w'], w['pe_b'] = t, f32(sd['pretrained.patch_embed.proj.bias'])
        w['cls'] = f32(sd['pretrained.cls_token']).reshape(C)
        self._pos_embed = f32(sd['pretrained.pos_embed'])
        blocks = []
        for i in range(cfg['depth']):
            p = f'pretrained.blocks.{i}.'
            blocks.append(dict(
                ln1_w=f32(sd[p + 'norm1.weight']), ln1_b=f32(sd[p + 'norm1.bias']),
                qkv_w=f16(sd[p + 'attn.qkv.weight']), qkv_b=f32(sd[p + 'attn.qkv.bias']),
                proj_w=f16(sd[p + 'attn.proj.weight']), proj_b=f32(sd[p + 'attn.proj.bias']), ls1=f32(sd[p + 'ls1.gamma']),
                ln2_w=f32(sd[p + 'norm2.weight']), ln2_b=f32(sd[p + 'norm2.bias']),
                fc1_w=f16(sd[p + 'mlp.fc1.weight']), fc1_b=f32(sd[p + 'mlp.fc1.bias']),
                fc2_w=f16(sd[p + 'mlp.fc2.weight']), fc2_b=f32(sd[p + 'mlp.fc2.bias']), ls2=f32(sd[p + 'ls2.gamma'])))
        w['blocks'] = blocks
        w['norm_w'], w['norm_b'] = f32(sd['pretrained.norm.weight']), f32(sd['pretrained.norm.bias'])
        # ---- DPT head; channel counts padded to multiples of 64 with zero weights (ViT-S/B have 48/96-wide maps) ----
        self.ocp = [_ru(c, 64) for c in oc]
        self.Fp = _ru(Fch, 64)
        self.F2p = _ru(Fch // 2, 64)
        h = 'depth_head.'
        for i in range(4):
            t = torch.zeros(self.ocp[i], C, dtype=torch.float16, device=dev)
            t[:oc[i]] = sd[h + f'projects.{i}.weight'].detach().to(dev).reshape(oc[i], C).to(torch.float16)
            w[f'proj{i}_w'], w[f'proj{i}_b'] = t, _pad_vec(sd[h + f'projects.{i}.bias'].detach().to(dev), self.ocp[i])
        for i, s in ((0, 4), (1, 2)):  # ConvTranspose2d(k = s): W[(i,j,co), ci] = w[ci, co, i, j]
            wt = sd[h + f'resize_layers.{i}.weight'].detach().to(dev)  # [ci, co, s, s]
            t = torch.zeros(s, s, self.ocp[i], self.ocp[i], dtype=torch.float16, device=dev)
            t[:, :, :oc[i], :oc[i]] = wt.permute(2, 3, 1, 0).to(torch.float16)
            w[f'up{i}_w'] = t.reshape(s * s * self.ocp[i], self.ocp[i]).contiguous()
            w[f'up{i}_b'] = _pad_vec(sd[h + f'resize_layers.{i}.bias'].detach().to(dev), self.ocp[i]).repeat(s * s).contiguous()
        w['down3_w'] = _conv_w(sd[h + 'resize_layers.3.weight'].detach().to(dev), self.ocp[3], self.ocp[3])
        w['down3_b'] = _pad_vec(sd[h + 'resize_layers.3.bias'].detach().to(dev), self.ocp[3])
        for i in range(4):
            w[f'rn{i}_w'] = _conv_w(sd[h + f'scratch.layer{i + 1}_rn.weight'].detach().to(dev), self.ocp[i], self.Fp)
        for i in range(1, 5):
            r = h + f'scratch.refinenet{i}.'
            t = torch.zeros(self.Fp, self.Fp, dtype=torch.float16, device=dev)
            t[:Fch, :Fch] = sd[r + 'out_conv.weight'].detach().to(dev).reshape(Fch, Fch).to(torch.float16)
            w[f'rf{i}_out_w'], w[f'rf{i}_out_b'] = t, _pad_vec(sd[r + 'out_conv.bias'].detach().to(dev), self.Fp)
            for u in (1, 2):
                for cv in (1, 2):
                    k = r + f'resConfUnit{u}.conv{cv}.'
                    if k + 'weight' in sd:
                        w[f'rf{i}_u{u}c{cv}_w'] = _conv_w(sd[k + 'weight'].detach().to(dev), self.Fp, self.Fp)
                        w[f'rf{i}_u{u}c{cv}_b'] = _pad_vec(sd[k + 'bias'].detach().to(dev), self.Fp)
        w['oc1_w'] = _conv_w(sd[h + 'scratch.output_conv1.weight'].detach().to(dev), self.Fp, self.F2p)
        w['oc1_b'] = _pad_vec(sd[h + 'scratch.output_conv1.bias'].detach().to(dev), self.F2p)
        w['oc2_w'] = _conv_w(sd[h + 'scratch.output_conv2.0.weight'].detach().to(dev), self.F2p, 32)
        w['oc2_b'] = f32(sd[h + 'scratch.output_conv2.0.bias'])
        w['oc3_w'] = f32(sd[h + 'scratch.output_conv2.2.weight']).reshape(32)
        self.oc3_b = float(sd[h + 'scratch.output_conv2.2.bias'].detach().float().reshape(-1)[0])
        self.w = w

    def _pos(self, gh, gw):
        """interpolate_pos_encoding (dinov2.py:179-210); identity for the native 37x37 grid.  Setup-time, cached."""
        import torch
        import torch.nn.functional as F
        key = (gh, gw)
        if key in self._pos_cache:
            return self._pos_cache[key]
        pe = self._pos_embed
        C = pe.shape[-1]
        N = pe.shape[1] - 1
        n = int(round(math.sqrt(N)))
        # host arithmetic shared with the model-level C-ABI (csrc/model.cu), so both paths use bit-identical tables
        src = np.ascontiguousarray(pe.reshape(N + 1, C).cpu().numpy(), dtype=np.float32)
        dst = np.empty((gh * gw + 1, C), dtype=np.float32)
        _lib.check(self.ops.L.dm_dinov2_pos_embed(src.ctypes.data, n, C, gh, gw, dst.ctypes.data), "dm_dinov2_pos_embed")
        out = torch.from_numpy(dst).to(self.device)
        self._pos_cache[key] = out
        return out

    # ---- activation buffers ----------------------------------------------------------------------------------------
    def _buffers(self, B, nh, nw):
        import torch
        key = (B, nh, nw)
        if self._buf_key == key:
            return self._bufs
        self._bufs = {}
        self._buf_key = None
        dev = self.device
        C, Fp = self.cfg['embed_dim'], self.Fp
        gh, gw = nh // self.PATCH, nw // self.PATCH
        Np, N = gh * gw, gh * gw + 1
        h16 = lambda *s: torch.empty(*s, dtype=torch.float16, device=dev)
        b = {}
        b['patches'] = h16(B * Np, self.kpad)
        b['pe'] = h16(B * Np, C)
        b['x'] = torch.empty(B * N, C, dtype=torch.float32, device=dev)
        b['h'] = h16(B * N, C)
        b['qkv'] = h16(B * N, 3 * C)
        b['att'] = h16(B * N, C)
        b['mlp'] = h16(B * N, 4 * C)
        b['feat'] = [h16(B * Np, C) for _ in range(4)]
        b['cat'] = h16(B * Np, 2 * C) if getattr(self, 'NEEDS_READOUT', False) else None
        sizes = [(gh * 4, gw * 4), (gh * 2, gw * 2), (gh, gw), ((gh - 1) // 2 + 1, (gw - 1) // 2 + 1)]
        b['sizes'] = sizes
        b['p'] = [h16(B * Np, self.ocp[i]) for i in range(4)]
        b['r'] = [h16(B, sizes[0][0], sizes[0][1], self.ocp[0]), h16(B, sizes[1][0], sizes[1][1], self.ocp[1]), None,
                  h16(B, sizes[3][0], sizes[3][1], self.ocp[3])]
        b['cols3'] = h16(B * sizes[3][0] * sizes[3][1], 9 * self.ocp[3])
        b['l'] = [h16(B, s[0], s[1], Fp) for s in sizes]
        b['lr'] = [h16(B, s[0], s[1], Fp) for s in sizes]
        for i in range(4):
            s = sizes[i]
            b[f't{i}'] = h16(B, s[0], s[1], Fp)      # relu(conv1(.)) scratch
            b[f'o{i}'] = h16(B, s[0], s[1], Fp)      # fused sum
            b[f'or{i}'] = h16(B, s[0], s[1], Fp)     # relu copy
            b[f'u{i}'] = h16(B, s[0], s[1], Fp)      # RCU2 output
        up = [sizes[2], sizes[1], sizes[0], (sizes[0][0] * 2, sizes[0][1] * 2)]  # target size of refinenet4..1
        b['up_sizes'] = up
        b['v'] = [h16(B, s[0], s[1], Fp) for s in (sizes[3], sizes[2], sizes[1], sizes[0])]   # out_conv output, before the up-sample
        b['path'] = [h16(B, s[0], s[1], Fp) for s in up]   # refinenet output (up-sampled)
        b['oc1'] = h16(B, up[3][0], up[3][1], self.F2p)
        b['oc1u'] = h16(B, nh, nw, self.F2p)
        b['d'] = torch.empty(B, nh, nw, dtype=torch.float32, device=dev)
        self._bufs, self._buf_key = b, key
        return b

    # ---- model-family hooks ------------------------------------------------------------------------------------------
    def net_size(self, W, H, net_w, net_h):
        return dav2_net_size(W, H, net_w)  # estimatedepthanything_v2 passes w as input_size (:552)

    def attention(self, i, b, B, N, heads, C, gh, gw):
        self.ops.attention(b['qkv'], B, N, heads, (C // heads) ** -0.5, b['att'])

    def _probed_attention(self, i, b, B, N, heads, C, gh, gw):
        """bench hook: probe['attn'] collects one (start, end) CUDA event pair per attention launch"""
        if self.probe is not None and 'attn' in self.probe:
            import torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.attention(i, b, B, N, heads, C, gh, gw)
            e1.record()
            self.probe['attn'].append((e0, e1))
        else:
            self.attention(i, b, B, N, heads, C, gh, gw)

    def emit_feature(self, b, fi, B, N, C):
        """get_intermediate_layers(norm=True) without the class token (dinov2.py:297-321)."""
        self.ops.layernorm(b['x'], B * N, C, self.w['norm_w'], self.w['norm_b'], b['feat'][fi], tokens_per_img=N, drop_first=1)

    # ---- forward ---------------------------------------------------------------------------------------------------
    def forward_batch(self, rgb, net_w, net_h=None, out_hw=None):
        """rgb: uint8 CUDA [B,H,W,3] -> float32 CUDA [B,H,W] raw prediction (what the reference's estimate* returns)."""
        import torch
        ops, w, cfg = self.ops, self.w, self.cfg
        B, H, W, _ = rgb.shape
        nw, nh = self.net_size(W, H, net_w, net_h if net_h is not None else net_w)
        C, heads, Fp = cfg['embed_dim'], cfg['heads'], self.Fp
        P_ = self.PATCH
        gh, gw = nh // P_, nw // P_
        Np, N = gh * gw, gh * gw + 1
        b = self._buffers(B, nh, nw)
        # image2tensor
        ops.patchify(rgb, B, H, W, nh, nw, P_, self.MEAN, self.STD, self.CHAN_MAP, b['patches'], self.kpad)
        self.run_network(b, B, nh, nw)
        return self.run_head(b, B, H, W, nh, nw, out_hw)

    def run_network(self, b, B, nh, nw):
        """patch embedding -> transformer blocks -> reassemble -> fusion blocks; leaves refinenet1's output in b['path'][3]
        (and layer4_rn / refinenet4..2 in b['l'][3] / b['path'][0..2], which the ZoeDepth head reads)."""
        ops, w, cfg = self.ops, self.w, self.cfg
        C, heads, Fp = cfg['embed_dim'], cfg['heads'], self.Fp
        P_ = self.PATCH
        gh, gw = nh // P_, nw // P_
        Np, N = gh * gw, gh * gw + 1
        E, A = _lib, _lib
        # patch embedding + tokens
        ops.gemm(b['patches'], self.kpad, w['pe_w'], self.kpad, B * Np, C, self.kpad, bias=w['pe_b'], C=b['pe'], ldc=C)
        ops.tokens(b['pe'], w['cls'], self._pos(gh, gw) if self._pos_embed is not None else None, b['x'], B, Np, C)
        rows = B * N
        fi = 0
        for i, blk in enumerate(w['blocks']):
            ops.layernorm(b['x'], rows, C, blk['ln1_w'], blk['ln1_b'], b['h'])
            ops.gemm(b['h'], C, blk['qkv_w'], C, rows, 3 * C, C, bias=blk['qkv_b'], C=b['qkv'], ldc=3 * C)
            self._probed_attention(i, b, B, N, heads, C, gh, gw)
            ops.gemm(b['att'], C, blk['proj_w'], C, rows, C, C, epi=E.EPI_RESID_F32, bias=blk['proj_b'], X=b['x'], ldx=C, gamma=blk['ls1'])
            ops.layernorm(b['x'], rows, C, blk['ln2_w'], blk['ln2_b'], b['h'])
            if self.probe is not None and 'fc1' in self.probe and i == 0:
                self.probe['fc1'][0].record()
            ops.gemm(b['h'], C, blk['fc1_w'], C, rows, 4 * C, C, act=A.ACT_GELU, bias=blk['fc1_b'], C=b['mlp'], ldc=4 * C)
            if self.probe is not None and 'fc1' in self.probe and i == 0:
                self.probe['fc1'][1].record()
            ops.gemm(b['mlp'], 4 * C, blk['fc2_w'], 4 * C, rows, C, 4 * C, epi=E.EPI_RESID_F32, bias=blk['fc2_b'], X=b['x'], ldx=C, gamma=blk['ls2'])
            if i in cfg['layers']:
                self.emit_feature(b, fi, B, N, C)
                fi += 1
        # ---- DPT head (dpt.py:117-150) ----
        sizes = b['sizes']
        for i in range(4):
            ops.gemm(b['feat'][i], C, w[f'proj{i}_w'], C, B * Np, self.ocp[i], C, bias=w[f'proj{i}_b'], C=b['p'][i], ldc=self.ocp[i])
        ops.gemm(b['p'][0], self.ocp[0], w['up0_w'], self.ocp[0], B * Np, 16 * self.ocp[0], self.ocp[0], epi=E.EPI_PIXSHUF, bias=w['up0_b'],
                 C=b['r'][0], ps=(4, self.ocp[0], gh, gw))
        ops.gemm(b['p'][1], self.ocp[1], w['up1_w'], self.ocp[1], B * Np, 4 * self.ocp[1], self.ocp[1], epi=E.EPI_PIXSHUF, bias=w['up1_b'],
                 C=b['r'][1], ps=(2, self.ocp[1], gh, gw))
        r2 = b['p'][2]
        ops.im2col_s2(b['p'][3], B, gh, gw, self.ocp[3], b['cols3'])
        ops.gemm(b['cols3'], 9 * self.ocp[3], w['down3_w'], 9 * self.ocp[3], B * sizes[3][0] * sizes[3][1], self.ocp[3], 9 * self.ocp[3],
                 bias=w['down3_b'], C=b['r'][3], ldc=self.ocp[3])
        rs = [b['r'][0], b['r'][1], r2, b['r'][3]]
        for i in range(4):  # layer{i}_rn (no bias) -> l_i and relu(l_i)
            ops.conv3x3(rs[i], B, sizes[i][0], sizes[i][1], self.ocp[i], w[f'rn{i}_w'], Fp, C=b['l'][i], C2=b['lr'][i])
        # refinenet4: resConfUnit2(l4) -> resize -> out_conv.  The 1x1 out_conv (+ bias) commutes with the bilinear
        # interpolation (a per-pixel channel mix against per-channel spatial weights that sum to one), so it runs BEFORE the
        # up-sample: a quarter of the MACs and no full-resolution intermediate (dmidas/blocks.py:425-437 has it after).
        s3 = sizes[3]
        ops.conv3x3(b['lr'][3], B, s3[0], s3[1], Fp, w['rf4_u2c1_w'], Fp, act=A.ACT_RELU, bias=w['rf4_u2c1_b'], C=b['t3'])
        ops.conv3x3(b['t3'], B, s3[0], s3[1], Fp, w['rf4_u2c2_w'], Fp, bias=w['rf4_u2c2_b'], C=b['u3'], R=b['l'][3])
        up = b['up_sizes']
        ops.gemm(b['u3'], Fp, w['rf4_out_w'], Fp, B * s3[0] * s3[1], Fp, Fp, bias=w['rf4_out_b'], C=b['v'][0], ldc=Fp)
        ops.resize_nhwc(b['v'][0], B, s3[0], s3[1], Fp, b['path'][0], up[0][0], up[0][1])
        # refinenet3, 2, 1: output = path + RCU1(l_i); output = RCU2(output); out_conv; resize (commuted, see above)
        for step, (li, rf) in enumerate(((2, 3), (1, 2), (0, 1))):
            s = sizes[li]
            path = b['path'][step]
            ops.conv3x3(b['lr'][li], B, s[0], s[1], Fp, w[f'rf{rf}_u1c1_w'], Fp, act=A.ACT_RELU, bias=w[f'rf{rf}_u1c1_b'], C=b[f't{li}'])
            ops.conv3x3(b[f't{li}'], B, s[0], s[1], Fp, w[f'rf{rf}_u1c2_w'], Fp, bias=w[f'rf{rf}_u1c2_b'], C=b[f'o{li}'], C2=b[f'or{li}'],
                        R=b['l'][li], R2=path)
            ops.conv3x3(b[f'or{li}'], B, s[0], s[1], Fp, w[f'rf{rf}_u2c1_w'], Fp, act=A.ACT_RELU, bias=w[f'rf{rf}_u2c1_b'], C=b[f't{li}'])
            ops.conv3x3(b[f't{li}'], B, s[0], s[1], Fp, w[f'rf{rf}_u2c2_w'], Fp, bias=w[f'rf{rf}_u2c2_b'], C=b[f'u{li}'], R=b[f'o{li}'])
            t = up[step + 1]
            ops.gemm(b[f'u{li}'], Fp, w[f'rf{rf}_out_w'], Fp, B * s[0] * s[1], Fp, Fp, bias=w[f'rf{rf}_out_b'], C=b['v'][step + 1], ldc=Fp)
            ops.resize_nhwc(b['v'][step + 1], B, s[0], s[1], Fp, b['path'][step + 1], t[0], t[1])

    def run_head(self, b, B, H, W, nh, nw, out_hw=None):
        """output_conv (dpt.py:139-150 / dpt_depth.py:150-158) + the final resize to the image size."""
        import torch
        ops, w = self.ops, self.w
        Fp = self.Fp
        E, A = _lib, _lib
        t = b['up_sizes'][3]
        ops.conv3x3(b['path'][3], B, t[0], t[1], Fp, w['oc1_w'], self.F2p, bias=w['oc1_b'], C=b['oc1'])
        ops.resize_nhwc(b['oc1'], B, t[0], t[1], self.F2p, b['oc1u'], nh, nw)
        # conv3x3 -> ReLU -> conv1x1 -> ReLU (+ the outer F.relu, idempotent) fused into one epilogue
        ops.conv3x3(b['oc1u'], B, nh, nw, self.F2p, w['oc2_w'], 32, epi=E.EPI_HEAD, act=A.ACT_RELU, bias=w['oc2_b'], X=b['d'], gamma=w['oc3_w'],
                    head_b2=self.oc3_b)
        oh, ow = out_hw if out_hw is not None else (H, W)
        out = torch.empty(B, oh, ow, dtype=torch.float32, device=self.device)
        ops.resize_f32(b['d'], B, nh, nw, out, oh, ow, self.FINAL_RESIZE_MODE)
        return out

    def to(self, device):
        return self

BEIT_CONFIGS = {
    'beitl16_512': dict(embed_dim=1024, depth=24, heads=16, features=256, out_channels=[256, 512, 1024, 1024],
                        layers=[5, 11, 17, 23], window=32),
    'beitl16_384': dict(embed_dim=1024, depth=24, heads=16, features=256, out_channels=[256, 512, 1024, 1024],
                        layers=[5, 11, 17, 23], window=24),
    'beit_tiny': dict(embed_dim=128, depth=4, heads=2, features=64, out_channels=[64, 64, 128, 128],
                      layers=[0, 1, 2, 3], window=4),  # structural test configuration
}


def midas_net_size(width, height, net_w, net_h, multiple_of=32):
    """Resize(keep_aspect_ratio, 'minimal', multiple of 32) of the reference (dmidas/transforms.py:61-104)."""
    sh, sw = net_h / height, net_w / width
    if abs(1 - sw) < abs(1 - sh):
        sh = sw
    else:
        sw = sh
    return _constrain_to_multiple_of(sw * width, multiple_of), _constrain_to_multiple_of(sh * height, multiple_of)


def _gen_relative_position_index(wh, ww):
    """timm 0.9 gen_relative_position_index (restated): cls rows / cols use the three extra table entries."""
    import torch
    nrd = (2 * wh - 1) * (2 * ww - 1) + 3
    coords = torch.stack(torch.meshgrid([torch.arange(wh), torch.arange(ww)], indexing='ij')).flatten(1)
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += wh - 1
    rel[:, :, 1] += ww - 1
    rel[:, :, 0] *= 2 * ww - 1
    idx = torch.zeros((wh * ww + 1,) * 2, dtype=rel.dtype)
    idx[1:, 1:] = rel.sum(-1)
    idx[0, 0:] = nrd - 3
    idx[0:, 0] = nrd - 2
    idx[0, 0] = nrd - 1
    return idx


class DptBeitEngine(DepthAnythingV2Engine):
    """MiDaS 3.1 DPT-BEiT (dpt_beit_large_512 / _384) on the sm_100a kernels.

    Mirrors the reference's overriding forwards (dmidas/backbones/beit.py:18-129), the reassemble stage
    (dmidas/backbones/utils.py:28-39,83-124,144-249), DPT / DPTDepthModel (dmidas/dpt_depth.py:110-166) and estimatemidas
    (src/depthmap_generation.py:455-499).  The relative-position bias, which the reference rebuilds (bilinear table
    resize + gather) in every block of every forward, is expanded once per resolution into a [heads, N, N] fp16 table
    per block and added inside the fused attention kernel."""

    PATCH = 16
    MEAN = (0.5, 0.5, 0.5)
    STD = (0.5, 0.5, 0.5)
    CHAN_MAP = (2, 1, 0)        # estimatemidas receives the BGR-swapped image of get_raw_prediction (:381) unchanged
    FINAL_RESIZE_MODE = 1       # bicubic, align_corners=False (:487-497)
    CONFIGS = BEIT_CONFIGS
    NEEDS_READOUT = True

    def net_size(self, W, H, net_w, net_h):
        return midas_net_size(W, H, net_w, net_h)

    def _pack(self, sd):
        import torch
        dev = self.device
        cfg = self.cfg
        C = cfg['embed_dim']
        f16 = lambda t: t.detach().to(dev, torch.float16).contiguous()
        f32 = lambda t: t.detach().to(dev, torch.float32).contiguous()
        # re-key the MiDaS checkpoint into the layout the shared packer understands
        m = {}
        p = 'pretrained.model.'
        m['pretrained.patch_embed.proj.weight'] = sd[p + 'patch_embed.proj.weight']
        m['pretrained.patch_embed.proj.bias'] = sd[p + 'patch_embed.proj.bias']
        m['pretrained.cls_token'] = sd[p + 'cls_token']
        m['pretrained.pos_embed'] = torch.zeros(1, 1, C)
        for i in range(cfg['depth']):
            b, d = p + f'blocks.{i}.', f'pretrained.blocks.{i}.'
            for k in ('norm1.weight', 'norm1.bias', 'attn.qkv.weight', 'attn.proj.weight', 'attn.proj.bias', 'norm2.weight', 'norm2.bias',
                      'mlp.fc1.weight', 'mlp.fc1.bias', 'mlp.fc2.weight', 'mlp.fc2.bias'):
                m[d + k] = sd[b + k]
            m[d + 'attn.qkv.bias'] = torch.cat((sd[b + 'attn.q_bias'].float(), torch.zeros(C), sd[b + 'attn.v_bias'].float()))
            m[d + 'ls1.gamma'] = sd[b + 'gamma_1']
            m[d + 'ls2.gamma'] = sd[b + 'gamma_2']
        m['pretrained.norm.weight'] = torch.ones(C)
        m['pretrained.norm.bias'] = torch.zeros(C)
        for j in range(4):
            a = f'pretrained.act_postprocess{j + 1}.'
            m[f'depth_head.projects.{j}.weight'] = sd[a + '3.weight']
            m[f'depth_head.projects.{j}.bias'] = sd[a + '3.bias']
        for j in (0, 1, 3):
            a = f'pretrained.act_postprocess{j + 1}.4.'
            m[f'depth_head.resize_layers.{j}.weight'] = sd[a + 'weight']
            m[f'depth_head.resize_layers.{j}.bias'] = sd[a + 'bias']
        for k, v in sd.items():
            if k.startswith('scratch.layer') or k.startswith('scratch.refinenet'):
                m['depth_head.' + k] = v
        m['depth_head.scratch.output_conv1.weight'] = sd['scratch.output_conv.0.weight']
        m['depth_head.scratch.output_conv1.bias'] = sd['scratch.output_conv.0.bias']
        m['depth_head.scratch.output_conv2.0.weight'] = sd['scratch.output_conv.2.weight']
        m['depth_head.scratch.output_conv2.0.bias'] = sd['scratch.output_conv.2.bias']
        m['depth_head.scratch.output_conv2.2.weight'] = sd['scratch.output_conv.4.weight']
        m['depth_head.scratch.output_conv2.2.bias'] = sd['scratch.output_conv.4.bias']
        super()._pack(m)
        self._pos_embed = None  # BEiT uses no absolute position embedding (use_abs_pos_emb=False)
        self.w['readout'] = [(f16(sd[f'pretrained.act_postprocess{j + 1}.0.project.0.weight']),
                              f32(sd[f'pretrained.act_postprocess{j + 1}.0.project.0.bias'])) for j in range(4)]
        self._tables = [f32(sd[p + f'blocks.{i}.attn.relative_position_bias_table']) for i in range(cfg['depth'])]
        self._bias_cache = {}

    def rel_tables(self, gh, gw):
        """Table half of _get_rel_pos_bias (dmidas/backbones/beit.py:29-50): per block, the [nrd, heads] table resized
        (bilinear) to the current window, laid out [heads, nrd] in fp32 and multiplied by log2(e).  Once per resolution.
        The gather half (:52-62, relative_position_index) happens inside the attention kernel."""
        import torch
        import torch.nn.functional as F
        key = (gh, gw)
        if key not in self._bias_cache:
            win = self.cfg['window']
            old_h = old_w = 2 * win - 1
            new_h, new_w = 2 * gh - 1, 2 * gw - 1
            out = []
            idx = _gen_relative_position_index(gh, gw).to(self.device)       # [N, N]
            nrd_new = new_h * new_w + 3
            heads = self.cfg['heads']
            for t in self._tables:
                # host arithmetic shared with the model-level C-ABI (csrc/model.cu: beit_rel_table_host)
                src = np.ascontiguousarray(t.cpu().numpy(), dtype=np.float32)
                dst = np.empty((heads, nrd_new), dtype=np.float32)
                _lib.check(self.ops.L.dm_beit_rel_table(src.ctypes.data, win, heads, gh, gw, dst.ctypes.data), "dm_beit_rel_table")
                tab = torch.from_numpy(dst).to(self.device)
                # per (head, query) maximum of the bias over all keys: the round-1 kernel's row-max upper bound
                rowmax = torch.stack([tab[hh][idx].max(dim=1).values for hh in range(tab.shape[0])]).contiguous()
                out.append((tab, rowmax))
            self._bias_cache = {key: (out, new_h * new_w + 3)}  # keep one resolution resident (drops dense tables too)
        return self._bias_cache[key]

    @staticmethod
    def table_fits_on_chip(gh, gw):
        """The table attention modes keep one head's bias table (twice, reversed, for 16-aligned grids) and the per-key
        offsets in the 60.75 KB of shared memory the kernel has left (csrc/attention_tcgen05.cu, A4_TAB_MAX)."""
        nrd, N = (2 * gh - 1) * (2 * gw - 1) + 3, gh * gw + 1
        if gw % 16 == 0:
            nrd_pad = ((nrd + 16) & ~31) + 16                 # csrc/attention_tcgen05.cu: attn4_nrd_pad
            need = 8 * nrd_pad + 2 * (((N + 126) // 128) * 8 + 8) + 16
        else:
            need = 4 * ((nrd + 3) & ~3) + 2 * ((N + 127) // 128) * 128 + 16
        return need <= 227 * 1024 - 170240

    def dense_bias(self, gh, gw):
        """Fallback for windows whose table does not fit on chip (e.g. a 3:2 image on dpt_beit_large_512: net 768x512,
        nrd = 5988): the gather half of _get_rel_pos_bias (beit.py:52-62) done once per resolution into a dense fp16
        [heads, N, ld] tensor per block (ld = N rounded up to whole 128-key tiles), added inside the attention kernel."""
        import torch
        key = ('dense', gh, gw)
        if key not in self._bias_cache:
            tabs, nrd = self.rel_tables(gh, gw)
            idx = _gen_relative_position_index(gh, gw).to(self.device)
            N = gh * gw + 1
            ld = _ru(N, 128)
            out = []
            for tab, _ in tabs:
                d = torch.zeros(tab.shape[0], N, ld, dtype=torch.float16, device=self.device)
                d[:, :, :N] = (tab / 1.4426950408889634)[:, idx.view(-1)].view(-1, N, N).to(torch.float16)
                out.append(d)
            self._bias_cache[key] = (out, ld)
        return self._bias_cache[key]

    def attention(self, i, b, B, N, heads, C, gh, gw):
        tabs, nrd = self.rel_tables(gh, gw)
        if not self.table_fits_on_chip(gh, gw):
            dense, ld = self.dense_bias(gh, gw)
            self.ops.attention(b['qkv'], B, N, heads, (C // heads) ** -0.5, b['att'], bias=dense[i], bias_ld=ld)
            return
        self.ops.attention_relpos(b['qkv'], B, gh, gw, heads, (C // heads) ** -0.5, tabs[i][0], tabs[i][1], nrd, b['att'])

    def emit_feature(self, b, fi, B, N, C):
        """forward hook on the raw block output + ProjectReadout: GELU(Linear(cat(tokens, cls)))."""
        rw, rb = self.w['readout'][fi]
        _lib.check(self.ops.L.dm_concat_readout_f16(b['x'].data_ptr(), B, N, C, b['cat'].data_ptr(), _lib.stream_ptr()), "dm_concat_readout_f16")
        self.ops.launches += 1
        self.ops.gemm(b['cat'], 2 * C, rw, 2 * C, B * (N - 1), C, 2 * C, act=_lib.ACT_GELU, bias=rb, C=b['feat'][fi], ldc=C)


class DptVitEngine(DptBeitEngine):
    """MiDaS 3.0 dpt_large_384 (model type 3) on the sm_100a kernels, op-level path: timm's vit_large_patch16_384 driven by
    the reference's forward_flex (dmidas/backbones/vit.py:12-79,107-118) — absolute position embedding resized bilinearly to
    the current grid, plain (un-biased) attention, no LayerScale — with the hooks, ProjectReadout, reassemble stage and DPT
    decoder it shares with the BEiT models (dmidas/dpt_depth.py:31-166)."""

    CONFIGS = {
        'vitl16_384': dict(embed_dim=1024, depth=24, heads=16, features=256, out_channels=[256, 512, 1024, 1024], layers=[5, 11, 17, 23], window=24),
        'vit_tiny': dict(embed_dim=128, depth=4, heads=2, features=64, out_channels=[64, 64, 128, 128], layers=[0, 1, 2, 3], window=4),
    }

    def _pack(self, sd):
        import torch
        C = self.cfg['embed_dim']
        p = 'pretrained.model.'
        m = dict(sd)
        for i in range(self.cfg['depth']):      # present the ViT block in the layout the BEiT packer reads
            b = p + f'blocks.{i}.'
            qb = sd[b + 'attn.qkv.bias'].float()
            m[b + 'attn.q_bias'], m[b + 'attn.v_bias'] = qb[:C], qb[2 * C:]
            m[b + 'gamma_1'] = torch.ones(C)
            m[b + 'gamma_2'] = torch.ones(C)
            m[b + 'attn.relative_position_bias_table'] = torch.zeros(1, self.cfg['heads'])
        super()._pack(m)
        # the key projection DOES have a bias here: restore the full qkv bias the BEiT packer zeroed
        for i, blk in enumerate(self.w['blocks']):
            blk['qkv_b'] = sd[p + f'blocks.{i}.attn.qkv.bias'].detach().to(self.device, torch.float32).contiguous()
        self._pos_embed = sd[p + 'pos_embed'].detach().to(self.device, torch.float32).contiguous()

    def _pos(self, gh, gw):
        """_resize_pos_embed (vit.py:16-31) through the host routine the model-level C-ABI uses (bit-identical tables)."""
        import torch
        key = (gh, gw)
        if key not in self._pos_cache:
            pe = self._pos_embed
            C = pe.shape[-1]
            N = pe.shape[1] - 1
            n = int(round(math.sqrt(N)))
            src = np.ascontiguousarray(pe.reshape(N + 1, C).cpu().numpy(), dtype=np.float32)
            dst = np.empty((gh * gw + 1, C), dtype=np.float32)
            _lib.check(self.ops.L.dm_vit_pos_embed(src.ctypes.data, n, C, gh, gw, dst.ctypes.data), "dm_vit_pos_embed")
            self._pos_cache[key] = torch.from_numpy(dst).to(self.device)
        return self._pos_cache[key]

    def attention(self, i, b, B, N, heads, C, gh, gw):
        self.ops.attention(b['qkv'], B, N, heads, (C // heads) ** -0.5, b['att'])


class LeresEngine:
    """LeReS / res101 (model type 0) on the sm_100a kernels: estimateleres (src/depthmap_generation.py:406-440) around
    RelDepthModel('resnext101') (lib/multi_depth_model_woauxi.py:6-32, lib/Resnext_torch.py:60-220, lib/network_auxi.py:15-215).
    NHWC fp16 activations, fp32 accumulation.  1x1 convolutions are GEMMs, 3x3 ones the implicit-GEMM conv; the 32-group 3x3
    convolutions use block-diagonal dense filters (exact: the extra products are zeros), the three stride-2 ones go through the
    strided im2col; BatchNorm (running statistics, eps 1e-5) is folded into filters and biases when the checkpoint is packed; the
    bottleneck's `relu(out + identity)` and FTB's `relu(x + branch)` come out of the GEMM epilogue's relu copy (C2)."""

    LAYERS = (3, 4, 23, 3)
    GROUPS = 32
    ENC = "depth_model.encoder_modules.encoder."
    DEC = "depth_model.decoder_modules."
    MEAN = (0.485, 0.456, 0.406)
    STD = (0.229, 0.224, 0.225)

    def __init__(self, state_dict, device):
        self.device = device
        self.ops = _Ops()
        self._bufs, self._buf_key = {}, None
        self._graphs, self._graph_calls = {}, {}
        self._pooled_bytes, self._pool_limit = 0, None
        self._use_graph = os.environ.get("DEPTHMAP_B200_LERES_GRAPH", "1") != "0"
        self._pack(state_dict)

    # ---- weights -------------------------------------------------------------------------------------------------------
    def _fold(self, sd, conv, bn):
        """conv weight [Co, Ci/g, kh, kw] (+ optional bias) followed by BatchNorm (inference) -> (weight, bias) in fp32"""
        import torch
        w = sd[conv + '.weight'].detach().float()
        b = sd[conv + '.bias'].detach().float() if conv + '.bias' in sd else torch.zeros(w.shape[0])
        if bn is not None:
            scale = sd[bn + '.weight'].detach().float() / torch.sqrt(sd[bn + '.running_var'].detach().float() + 1e-5)
            w = w * scale.view(-1, 1, 1, 1)
            b = (b - sd[bn + '.running_mean'].detach().float()) * scale + sd[bn + '.bias'].detach().float()
        return w, b

    def _mat(self, w, b, kpad=None, npad=None):
        import torch
        co = w.shape[0]
        m = w.reshape(co, -1)
        k, n = kpad or m.shape[1], npad or co
        t = torch.zeros(n, k, dtype=torch.float16)
        t[:co, :m.shape[1]] = m.to(torch.float16)
        bb = torch.zeros(n, dtype=torch.float32)
        bb[:co] = b
        return t.to(self.device).contiguous(), bb.to(self.device).contiguous()

    def _conv3(self, w, b, groups=1, npad=None):
        """[Co, Ci/g, 3, 3] -> dense fp16 [Co(pad), 9 * Ci], K ordered (ky, kx, ci); groups become diagonal blocks"""
        import torch
        co, cig = w.shape[:2]
        ci = cig * groups
        n = npad or co
        t = torch.zeros(n, 3, 3, ci, dtype=torch.float16)
        wp = w.permute(0, 2, 3, 1).to(torch.float16)             # [Co, ky, kx, Ci/g]
        cog = co // groups
        for g in range(groups):
            t[g * cog:(g + 1) * cog, :, :, g * cig:(g + 1) * cig] = wp[g * cog:(g + 1) * cog]
        bb = torch.zeros(n, dtype=torch.float32)
        bb[:co] = b
        return t.reshape(n, 9 * ci).to(self.device).contiguous(), bb.to(self.device).contiguous()

    def _pack(self, sd):
        import torch
        E, D = self.ENC, self.DEC
        w = {}
        sw, sb = self._fold(sd, E + 'conv1', E + 'bn1')            # [64, 3, 7, 7] -> [64, (ky, kx, c)] padded to 192
        w['stem'] = self._mat(sw.permute(0, 2, 3, 1).contiguous(), sb, kpad=192)
        blocks = []
        for li, nb in enumerate(self.LAYERS, start=1):
            for bi in range(nb):
                p = f"{E}layer{li}.{bi}"
                blk = dict(stride=2 if (bi == 0 and li > 1) else 1)
                blk['c1'] = self._mat(*self._fold(sd, p + '.conv1', p + '.bn1'))
                blk['c2'] = self._conv3(*self._fold(sd, p + '.conv2', p + '.bn2'), groups=self.GROUPS)
                blk['c3'] = self._mat(*self._fold(sd, p + '.conv3', p + '.bn3'))
                blk['down'] = self._mat(*self._fold(sd, p + '.downsample.0', p + '.downsample.1')) if bi == 0 else None
                blk['width'], blk['cout'] = blk['c1'][0].shape[0], blk['c3'][0].shape[0]
                blocks.append(blk)
        w['blocks'] = blocks

        def ftb(p):
            return dict(c1=self._conv3(*self._fold(sd, p + '.conv1', None)),
                        b1=self._conv3(*self._fold(sd, p + '.conv_branch.1', p + '.conv_branch.2')),
                        b4=self._conv3(*self._fold(sd, p + '.conv_branch.4', None)))
        w['conv'] = ftb(D + 'conv')
        w['conv1'] = self._conv3(*self._fold(sd, D + 'conv1', None))
        for k in ('ffm2', 'ffm1', 'ffm0'):
            w[k] = (ftb(D + k + '.ftb1'), ftb(D + k + '.ftb2'))
        a = D + 'outconv.adapt_conv'
        w['ao0'] = self._conv3(*self._fold(sd, a + '.0', a + '.1'))
        w['ao3'] = self._conv3(*self._fold(sd, a + '.3', None), npad=32)
        self.w = w

    # ---- buffers: a simple keyed pool (every tensor of a forward has its own name) ---------------------------------
    def _buf(self, name, shape, dtype=None):
        import torch
        dtype = dtype or torch.float16
        key = (name, tuple(shape), dtype)          # one set of buffers per net size: BOOST alternates 448 / 896 / whole-image nets, and the
        t = self._bufs.get(key)                    # captured graphs below need stable addresses
        if t is None:
            t = torch.empty(*shape, dtype=dtype, device=self.device)
            self._bufs[key] = t
            self._pooled_bytes += t.numel() * t.element_size()
        return t

    def _trim_pools(self):
        """Called at the start of a forward, never inside one: BOOST's whole-image net size depends on the image, so a long run would
        otherwise collect one buffer set (and one graph) per size.  Past half of the device memory everything pooled is dropped and
        rebuilt lazily."""
        import torch
        if self._pool_limit is None:
            self._pool_limit = torch.cuda.get_device_properties(self.device).total_memory // 2
        if self._pooled_bytes > self._pool_limit and not torch.cuda.is_current_stream_capturing():
            torch.cuda.synchronize(self.device)
            self._graphs.clear()
            self._graph_calls.clear()
            self._bufs.clear()
            self._pooled_bytes = 0
            torch.cuda.empty_cache()

    # ---- forward ---------------------------------------------------------------------------------------------------
    def _network(self, B, net_h, net_w, cols):
        """stem GEMM .. decoder output [B, net_h, net_w] fp32 (a pooled buffer).  From the second call on at a given (B, net size) the
        ~500 launches replay from a CUDA graph (DEPTHMAP_B200_LERES_GRAPH=0: eager)."""
        import torch
        key = (B, net_h, net_w)
        capturing = torch.cuda.is_current_stream_capturing()       # inside somebody else's capture: plain launches
        g = self._graphs.get(key)
        if g is not None and not capturing:
            g[0].replay()
            self.ops.launches += g[2]                                # the kernels inside the graph still launch
            return g[1]
        n = self._graph_calls.get(key, 0) + 1
        self._graph_calls[key] = n
        if self._use_graph and g is None and n >= 2 and not capturing:
            try:
                graph = torch.cuda.CUDAGraph()
                n0 = self.ops.launches
                with torch.cuda.graph(graph):
                    dn = self._network_eager(B, net_h, net_w, cols)
                self._graphs[key] = (graph, dn, self.ops.launches - n0)
                graph.replay()
                return dn
            except Exception as e:  # noqa: BLE001 — an optimisation only: same kernels eagerly
                sys.stderr.write(f"[depthmap_b200] LeReS graph capture failed ({e}); running eagerly\n")
                torch.cuda.synchronize()
                self._use_graph = False
        return self._network_eager(B, net_h, net_w, cols)

    def forward_batch(self, rgb, net_w, net_h=None, out_hw=None, planar=None):
        """rgb: uint8 CUDA [B,H,W,3] -> float32 CUDA [B,H,W] (what estimateleres returns; invert = True).
        planar = (fp32 CUDA [3,Hi,Wi] image in network channel order, (x0, y0, w, h)) instead of `rgb`: estimateleres on a float
        crop, as BOOST calls it (src/depthmap_generation.py:1053-1056) — one image, result [1, h, w]."""
        import torch
        ops, w, L = self.ops, self.w, self.ops.L
        st = _lib.stream_ptr
        A = _lib
        if planar is None:
            B, H, W, _ = rgb.shape
        else:
            pl_img, rect = planar
            pl_hi, pl_wi = int(pl_img.shape[1]), int(pl_img.shape[2])
            B, H, W = 1, int(rect[3]), int(rect[2])
        net_h = net_h if net_h is not None else net_w
        if net_w % 32 or net_h % 32:
            raise ValueError("LeReS needs a net size that is a multiple of 32")
        self._trim_pools()
        # stem: pre-processing + im2col of the 7x7 / 2 conv, folded BN + ReLU in the GEMM, max-pool
        h1, w1 = (net_h + 6 - 7) // 2 + 1, (net_w + 6 - 7) // 2 + 1
        cols = self._buf('stem_cols', (B * h1 * w1, 192))
        m = (ctypes.c_float * 3)(*self.MEAN)
        s = (ctypes.c_float * 3)(*self.STD)
        if planar is None:
            _lib.check(L.dm_leres_stem_im2col(rgb.data_ptr(), B, H, W, net_h, net_w, m, s, cols.data_ptr(), st()), "dm_leres_stem_im2col")
        else:
            _lib.check(L.dm_leres_stem_im2col_f32(pl_img.data_ptr(), pl_hi, pl_wi, rect[0], rect[1], rect[2], rect[3], net_h, net_w, m, s, cols.data_ptr(),
                                                  st()), "dm_leres_stem_im2col_f32")
        dn = self._network(B, net_h, net_w, cols)
        hh, ww = net_h // 2, net_w // 2
        oh, ow = out_hw if out_hw is not None else (H, W)
        out = torch.empty(B, oh, ow, dtype=torch.float32, device=self.device)
        if (oh, ow) == (2 * hh, 2 * ww):
            out.copy_(dn)                                      # cv2.resize to the same size is a copy
        else:
            ops.resize_f32(dn, B, 2 * hh, 2 * ww, out, oh, ow, 1)   # cv2.INTER_CUBIC (A = -0.75, replicated borders)
        ops.launches += 1
        return out

    def forward_crops(self, planar, rects, net):
        """BOOST's patch batch: estimateleres' network on B crops of one planar fp32 image ([3, Hi, Wi], rects = [(x0, y0, w, h)]), all at the
        same square net size -> fp32 [B, net, net] (a pooled buffer, valid until the next call at this (B, net)); the caller does the
        per-crop resize back (each crop has its own size)."""
        import torch
        if net % 32:
            raise ValueError("LeReS needs a net size that is a multiple of 32")
        B = len(rects)
        self._trim_pools()
        hi, wi = int(planar.shape[1]), int(planar.shape[2])
        for x0, y0, w, h in rects:
            if x0 < 0 or y0 < 0 or w <= 0 or h <= 0 or x0 + w > wi or y0 + h > hi:
                raise ValueError(f"crop {(x0, y0, w, h)} outside the {wi}x{hi} image")
        r = torch.tensor([list(map(int, q)) for q in rects], dtype=torch.int32).to(self.device)
        h1 = (net + 6 - 7) // 2 + 1
        cols = self._buf('stem_cols', (B * h1 * h1, 192))
        m = (ctypes.c_float * 3)(*self.MEAN)
        sdev = (ctypes.c_float * 3)(*self.STD)
        _lib.check(self.ops.L.dm_leres_stem_im2col_f32_batch(planar.data_ptr(), hi, wi, r.data_ptr(), B, net, net, m, sdev, cols.data_ptr(), _lib.stream_ptr()),
                   "dm_leres_stem_im2col_f32_batch")
        self.ops.launches += 1
        return self._network(B, net, net, cols)

    def _network_eager(self, B, net_h, net_w, cols):
        import torch
        ops, w, L = self.ops, self.w, self.ops.L
        st = _lib.stream_ptr
        A = _lib
        h1, w1 = (net_h + 6 - 7) // 2 + 1, (net_w + 6 - 7) // 2 + 1
        x = self._buf('stem', (B, h1, w1, 64))
        ops.gemm(cols, 192, w['stem'][0], 192, B * h1 * w1, 64, 192, act=A.ACT_RELU, bias=w['stem'][1], C=x, ldc=64)
        h, wd = (h1 + 2 - 3) // 2 + 1, (w1 + 2 - 3) // 2 + 1
        xp = self._buf('pool', (B, h, wd, 64))
        _lib.check(L.dm_maxpool3x3s2_nhwc_f16(x.data_ptr(), B, h1, w1, 64, xp.data_ptr(), st()), "dm_maxpool3x3s2_nhwc_f16")
        ops.launches += 2
        x, cin = xp, 64
        feats = []
        bi_global = 0
        for li, nb in enumerate(self.LAYERS, start=1):
            for bi in range(nb):
                blk = w['blocks'][bi_global]
                tag = f"l{li}b{bi % 2}" if bi > 0 else f"l{li}first"
                width, cout, stride = blk['width'], blk['cout'], blk['stride']
                M = B * h * wd
                t1 = self._buf(tag + '_t1', (B, h, wd, width))
                ops.gemm(x, cin, blk['c1'][0], cin, M, width, cin, act=A.ACT_RELU, bias=blk['c1'][1], C=t1, ldc=width)
                if stride == 1:
                    ho, wo = h, wd
                    t2 = self._buf(tag + '_t2', (B, ho, wo, width))
                    ops.conv3x3(t1, B, h, wd, width, blk['c2'][0], width, act=A.ACT_RELU, bias=blk['c2'][1], C=t2)
                else:
                    ho, wo = (h + 2 - 3) // 2 + 1, (wd + 2 - 3) // 2 + 1
                    c2 = self._buf(tag + '_cols', (B * ho * wo, 9 * width))
                    ops.im2col_s2(t1, B, h, wd, width, c2)
                    t2 = self._buf(tag + '_t2', (B, ho, wo, width))
                    ops.gemm(c2, 9 * width, blk['c2'][0], 9 * width, B * ho * wo, width, 9 * width, act=A.ACT_RELU, bias=blk['c2'][1], C=t2, ldc=width)
                Mo = B * ho * wo
                if blk['down'] is not None:
                    xs = x
                    if stride == 2:
                        xs = self._buf(tag + '_xs', (B, ho, wo, cin))
                        _lib.check(L.dm_subsample2_nhwc_f16(x.data_ptr(), B, h, wd, cin, xs.data_ptr(), st()), "dm_subsample2_nhwc_f16")
                        ops.launches += 1
                    idn = self._buf(tag + '_idn', (B, ho, wo, cout))
                    ops.gemm(xs, cin, blk['down'][0], cin, Mo, cout, cin, bias=blk['down'][1], C=idn, ldc=cout)
                else:
                    idn = x
                pre = self._buf(tag + '_pre', (B, ho, wo, cout))
                last = bi == nb - 1
                out = self._buf(f"feat{li}" if last else tag + '_out', (B, ho, wo, cout))
                ops.gemm(t2, width, blk['c3'][0], width, Mo, cout, width, bias=blk['c3'][1], C=pre, ldc=cout, C2=out, R=idn, ldr=cout)
                x, cin, h, wd = out, cout, ho, wo
                bi_global += 1
            feats.append((x, h, wd, cin))

        def conv(name, xin, hh, ww, ci, wb, co, act=A.ACT_NONE, R=None, C2=False):
            outp = self._buf(name, (B, hh, ww, co))
            out2 = self._buf(name + '_r', (B, hh, ww, co)) if C2 else None
            ops.conv3x3(xin, B, hh, ww, ci, wb[0], co, act=act, bias=wb[1], C=outp, C2=out2, R=R)
            return out2 if C2 else outp

        def ftb(name, xin, hh, ww, ci, f, cm):
            x1 = conv(name + '_x1', xin, hh, ww, ci, f['c1'], cm, act=A.ACT_RELU)           # the in-place ReLU also rewrites the skip operand
            b1 = conv(name + '_b1', x1, hh, ww, cm, f['b1'], cm, act=A.ACT_RELU)
            return conv(name + '_o', b1, hh, ww, cm, f['b4'], cm, R=x1, C2=True)             # relu(x1 + branch)

        def up2(name, xin, hh, ww, c):
            outp = self._buf(name, (B, 2 * hh, 2 * ww, c))
            ops.resize_nhwc(xin, B, hh, ww, c, outp, 2 * hh, 2 * ww)
            return outp

        f3, h3, w3, c3 = feats[3]
        x = ftb('dconv', f3, h3, w3, c3, w['conv'], 512)
        x = conv('dconv1', x, h3, w3, 512, w['conv1'], 256)
        x = up2('up32', x, h3, w3, 256)
        hh, ww = 2 * h3, 2 * w3
        for k, fi in (('ffm2', 2), ('ffm1', 1), ('ffm0', 0)):
            low, hl, wl, cl = feats[fi]
            assert (hl, wl) == (hh, ww)
            a1 = ftb(k + 'a', low, hl, wl, cl, w[k][0], 256)
            sm = self._buf(k + '_sum', (B, hl, wl, 256))
            _lib.check(L.dm_add_f16(a1.data_ptr(), x.data_ptr(), sm.data_ptr(), sm.numel(), st()), "dm_add_f16")
            ops.launches += 1
            x = ftb(k + 'b', sm, hl, wl, 256, w[k][1], 256)
            x = up2(k + '_up', x, hl, wl, 256)
            hh, ww = 2 * hl, 2 * wl
        x = conv('ao0', x, hh, ww, 256, w['ao0'], 128, act=A.ACT_RELU)
        d32 = self._buf('ao3', (B * hh * ww, 32), torch.float32)
        ops.conv3x3(x, B, hh, ww, 128, w['ao3'][0], 32, epi=A.EPI_STORE_F32, bias=w['ao3'][1], X=d32, ldx=32)
        dn = self._buf('dnet', (B, 2 * hh, 2 * ww), torch.float32)
        _lib.check(L.dm_resize_f32_ld(d32.data_ptr(), 32, B, hh, ww, dn.data_ptr(), 2 * hh, 2 * ww, 0, st()), "dm_resize_f32_ld")
        ops.launches += 1
        assert (2 * hh, 2 * ww) == (net_h, net_w)
        return dn

    def to(self, device):
        return self


class NativeDepthModel:
    """Thin caller of the model-level C-ABI (include/depthmap_b200.h: dm_model_create / dm_depth_forward / dm_model_destroy,
    csrc/model.cu): the handle owns the packed weights, the activation buffers, the resolution tables and a captured CUDA
    graph per shape; a forward is one C call.  Model types 1, 2 (DPT-BEiT-L 512 / 384) and 12, 13, 14 (Depth-Anything-V2)."""

    _DT = {"torch.float32": 0, "torch.float16": 1, "torch.bfloat16": 2}

    def __init__(self, state_dict, model_type, device):
        import torch
        self.L = _lib.load()
        if not hasattr(self.L, "dm_model_create"):
            raise RuntimeError("depthmap_b200: native library lacks dm_model_create; rebuild csrc (no fallback exists)")
        self.device = torch.device(device)
        self.model_type = model_type
        keep, items = [], []
        for name, t in state_dict.items():
            if not torch.is_tensor(t) or not t.is_floating_point():
                continue
            t = t.detach().to("cpu")
            if str(t.dtype) not in self._DT:
                t = t.float()
            t = t.contiguous()
            keep.append(t)
            w = _lib.Weight()
            w.name = name.encode()
            w.data_host = t.data_ptr()
            w.dtype = self._DT[str(t.dtype)]
            w.ndim = min(t.dim(), 4)
            shape = list(t.shape) if t.dim() <= 4 else [int(t.numel())]
            if t.dim() > 4:
                w.ndim = 1
            for k in range(4):
                w.shape[k] = shape[k] if k < len(shape) else 1
            items.append(w)
        arr = (_lib.Weight * len(items))(*items)
        blob = _lib.WeightBlob(arr, len(items))
        h = ctypes.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _lib.check(self.L.dm_model_create(ctypes.byref(h), int(model_type), ctypes.byref(blob), int(idx), 0), "dm_model_create")
        self.handle = h
        del keep

    def net_size(self, W, H, net_w, net_h):
        nw, nh = ctypes.c_int(), ctypes.c_int()
        _lib.check(self.L.dm_model_net_size(self.handle, W, H, net_w, net_h, ctypes.byref(nw), ctypes.byref(nh)), "dm_model_net_size")
        return nw.value, nh.value

    @property
    def launches(self):
        return int(self.L.dm_model_launches(self.handle))

    def forward_batch(self, rgb, net_w, net_h=None, out_hw=None):
        """rgb: uint8 CUDA [B,H,W,3] -> float32 CUDA [B,H,W] raw prediction."""
        import torch
        if self.handle is None:
            raise RuntimeError("model was destroyed")
        if rgb.dtype != torch.uint8 or rgb.dim() != 4 or rgb.shape[-1] != 3:
            raise ValueError("rgb must be a uint8 tensor [B,H,W,3]")
        rgb = rgb.contiguous()
        B, H, W, _ = rgb.shape
        oh, ow = out_hw if out_hw is not None else (H, W)
        out = torch.empty(B, oh, ow, dtype=torch.float32, device=rgb.device)
        _lib.check(self.L.dm_depth_forward(self.handle, rgb.data_ptr(), B, H, W, int(net_w), int(net_h if net_h is not None else net_w),
                                           out.data_ptr(), oh, ow, _lib.stream_ptr()), "dm_depth_forward")
        return out

    def close(self):
        if getattr(self, "handle", None) is not None:
            self.L.dm_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def to(self, device):
        return self


ZOE_CONFIG = dict(n_bins=64, emb=128, min_temp=0.0212, max_temp=50.0, router_dim=128, router_heads=4, router_layers=4)


class ZoeDepthNKEngine(DptBeitEngine):
    """ZoeDepth-NK (model type 9 = zoedepth_nk) on the sm_100a kernels: DepthModel.infer_pil
    (pad + flip test-time augmentation, dzoedepth/models/depth_model.py:57-152), PrepForMidas (base_models/midas.py:175-186),
    the DPT-BEiT-L-384 core with MidasCore's hooks (midas.py:258-319) and the metric head of ZoeDepthNK.forward
    (zoedepth_nk/zoedepth_nk_v1.py:159-243).  Image b and its horizontal flip run as forwards 2b / 2b+1 of ONE batch; the
    router picks nyu / kitti per forward on the device (argmax of two logits, no host sync, no cross-image vote).
    Checkpoint layout: MiDaS weights under "core.core.", head weights at the top level.  ZoeDepthEngine (types 7 and 8)
    shares everything but the head."""

    def __init__(self, state_dict, device, core_name='beitl16_384'):
        core_sd = {k[len("core.core."):]: v for k, v in state_dict.items() if k.startswith("core.core.")}
        self._head_sd = {k: v for k, v in state_dict.items() if not k.startswith("core.")}
        super().__init__(core_sd, core_name, device)
        self._pack_head(self._head_sd)
        self._zbuf_key, self._zbufs = None, {}

    # ---- weights -------------------------------------------------------------------------------------------------------
    def _hw(self, sd, key, rows=None, cols=None):
        """1x1 conv / linear weight -> fp16 [rows, cols] (zero padded)"""
        import torch
        t = sd[key + '.weight'].detach().to(self.device).float()
        t = t.reshape(t.shape[0], -1)
        r, c = rows or t.shape[0], cols or t.shape[1]
        o = torch.zeros(r, c, dtype=torch.float16, device=self.device)
        o[:t.shape[0], :t.shape[1]] = t.to(torch.float16)
        return o

    def _hb(self, sd, key, n=None):
        """bias -> fp32 [n] (zero padded)"""
        import torch
        t = sd[key + '.bias'].detach().to(self.device).float().reshape(-1)
        o = torch.zeros(n or t.numel(), dtype=torch.float32, device=self.device)
        o[:t.numel()] = t
        return o

    def _pack_out_conv(self, z):
        # out_conv with 64 output channels (32 real + 32 zero) so the stored activation is a valid GEMM-friendly NHWC tensor
        z['oc2_w'] = _conv_w(self._oc2_weight.to(self.device), self.F2p, 32)
        z['oc2_b'] = self._oc2_bias.to(self.device).float().contiguous()

    def _pack_head(self, sd):
        import torch
        dev = self.device
        z = {}
        W = lambda key, rows=None, cols=None: self._hw(sd, key, rows, cols)
        Bv = lambda key, n=None: self._hb(sd, key, n)
        z['conv2'] = (W('conv2'), Bv('conv2'))
        z['emb'] = (W('patch_transformer.embedding_convPxP'), Bv('patch_transformer.embedding_convPxP'))
        layers = []
        for i in range(ZOE_CONFIG['router_layers']):
            q = f'patch_transformer.transformer_encoder.layers.{i}'
            f32 = lambda k: sd[k].detach().to(dev).float().contiguous()
            layers.append(dict(
                in_w=sd[q + '.self_attn.in_proj_weight'].detach().to(dev, torch.float16).contiguous(), in_b=f32(q + '.self_attn.in_proj_bias'),
                out=(W(q + '.self_attn.out_proj'), Bv(q + '.self_attn.out_proj')),
                l1=(W(q + '.linear1'), Bv(q + '.linear1')), l2=(W(q + '.linear2'), Bv(q + '.linear2')),
                n1=(f32(q + '.norm1.weight'), f32(q + '.norm1.bias')), n2=(f32(q + '.norm2.weight'), f32(q + '.norm2.bias'))))
        z['layers'] = layers
        z['cls0'] = (W('mlp_classifier.0'), Bv('mlp_classifier.0'))
        z['cls2'] = (W('mlp_classifier.2', rows=32), Bv('mlp_classifier.2', 32))
        z['ones128'] = torch.ones(128, dtype=torch.float32, device=dev)
        z['zeros128'] = torch.zeros(128, dtype=torch.float32, device=dev)
        names = ('nyu', 'kitti')
        # seed bin regressors of both heads side by side: net.0 stacked, net.2 block-diagonal (nyu -> columns 0..63, kitti 64..127)
        z['seed0'] = (torch.cat([W(f'seed_bin_regressors.{n}._net.0') for n in names]), torch.cat([Bv(f'seed_bin_regressors.{n}._net.0') for n in names]))
        w2 = torch.zeros(128, 128, dtype=torch.float16, device=dev)
        for k, n in enumerate(names):
            w2[64 * k:64 * k + 64, 64 * k:64 * k + 64] = W(f'seed_bin_regressors.{n}._net.2')
        z['seed2'] = (w2, torch.cat([Bv(f'seed_bin_regressors.{n}._net.2') for n in names]))
        z['sproj'] = ((W('seed_projector._net.0'), Bv('seed_projector._net.0')), (W('seed_projector._net.2'), Bv('seed_projector._net.2')))
        z['proj'] = [((W(f'projectors.{i}._net.0'), Bv(f'projectors.{i}._net.0')), (W(f'projectors.{i}._net.2'), Bv(f'projectors.{i}._net.2'))) for i in range(4)]
        att = []
        for i in range(4):
            a0 = (torch.cat([W(f'attractors.{n}.{i}._net.0') for n in names]), torch.cat([Bv(f'attractors.{n}.{i}._net.0') for n in names]))
            w2 = torch.zeros(64, 256, dtype=torch.float16, device=dev)
            b2 = torch.zeros(64, dtype=torch.float32, device=dev)
            for k, n in enumerate(names):
                t = W(f'attractors.{n}.{i}._net.2')
                if t.shape[0] != 16:
                    raise NotImplementedError("ZoeDepth-NK attractor layers with other than 16 attractors (the reference always builds 16)")
                w2[32 * k:32 * k + 16, 128 * k:128 * k + 128] = t
                b2[32 * k:32 * k + 16] = Bv(f'attractors.{n}.{i}._net.2')
            att.append((a0, (w2, b2)))
        z['att'] = att
        # conditional log-binomial: mlp.0 split into its out_conv part (32 inputs, evaluated per pixel in clb_final) and its bin
        # embedding part (128 inputs, a GEMM before the up-sampling: a 1x1 conv commutes with bilinear interpolation)
        we = torch.zeros(128, 128, dtype=torch.float16, device=dev)
        wo = torch.zeros(2, 32, 40, dtype=torch.float32, device=dev)
        b0 = torch.zeros(2, 40, dtype=torch.float32, device=dev)
        w2c = torch.zeros(2, 4, 40, dtype=torch.float32, device=dev)
        b2c = torch.zeros(2, 4, dtype=torch.float32, device=dev)
        for k, n in enumerate(names):
            m0 = sd[f'conditional_log_binomial.{n}.mlp.0.weight'].detach().to(dev).float().reshape(40, 160)
            wo[k] = m0[:, :32].t()
            we[64 * k:64 * k + 40] = m0[:, 32:].to(torch.float16)
            b0[k] = sd[f'conditional_log_binomial.{n}.mlp.0.bias'].detach().to(dev).float()
            w2c[k] = sd[f'conditional_log_binomial.{n}.mlp.2.weight'].detach().to(dev).float().reshape(4, 40)
            b2c[k] = sd[f'conditional_log_binomial.{n}.mlp.2.bias'].detach().to(dev).float()
        z['clb'] = (we, wo.contiguous(), b0.contiguous(), w2c.contiguous(), b2c.contiguous())
        self._pack_out_conv(z)
        self.z = z
        self._pe_cache = {}

    def _pack(self, sd):
        self._oc2_weight = sd['scratch.output_conv.2.weight'].detach()
        self._oc2_bias = sd['scratch.output_conv.2.bias'].detach()
        super()._pack(sd)

    def _router_pe(self, S):
        """PositionalEncodingPermute1D replacement of patch_transformer.py:45-62: sin | cos of position * 10000^(-2i/E)."""
        import torch
        if S not in self._pe_cache:
            E = ZOE_CONFIG['router_dim']
            pos = torch.arange(0, S, dtype=torch.float32, device=self.device).unsqueeze(1)
            idx = torch.arange(0, E, 2, dtype=torch.float32, device=self.device).unsqueeze(0)
            div = torch.exp(idx * (-torch.log(torch.tensor(10000.0, device=self.device)) / E))
            pe = pos * div
            self._pe_cache = {S: torch.cat([torch.sin(pe), torch.cos(pe)], dim=1).contiguous()}
        return self._pe_cache[S]

    def _zbuffers(self, F, nh, nw, b):
        """Head buffers; the widths follow the packed weights (NK: two heads side by side; N / K: one head)."""
        import torch
        key = (F, nh, nw)
        if self._zbuf_key == key:
            return self._zbufs
        dev, z = self.device, self.z
        h16 = lambda *s: torch.empty(*s, dtype=torch.float16, device=dev)
        f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        s3 = b['sizes'][3]
        n0 = s3[0] * s3[1]
        S = n0 + 1
        levels = list(b['up_sizes'])                       # (h, w) of refinenet4..1 outputs
        ph = z['sproj'][0][0].shape[0]                      # projector hidden width
        aw, an = z['att'][0][0][0].shape[0], z['att'][0][1][0].shape[0]     # attractor hidden width, attractor GEMM output width
        zb = dict(x16=h16(F * n0, self.Fp), s0=h16(F * n0, z['seed0'][0].shape[0]), seed=f32(F * n0, z['seed2'][0].shape[0]),
                  bprev=f32(F * n0, 64), p0=h16(F * n0, ph), pemb=h16(F * n0, 128), S=S, n0=n0, levels=levels)
        if 'layers' in z:                                  # the router of ZoeDepth-NK
            zb.update(emb=h16(F * n0, 128), X=f32(F * S, 128), h=h16(F * S, 128), qkv=h16(F * S, 384), att=h16(F * S, 128),
                      ff=h16(F * S, 1024), c1=h16(F, 128), logits=f32(F, 32))
        zb['t'] = [h16(F * h * w, ph) for h, w in levels]
        zb['bemb'] = [h16(F * h * w, 128) for h, w in levels]
        zb['xin'] = [h16(F * h * w, 128) for h, w in levels]
        zb['a0'] = [h16(F * h * w, aw) for h, w in levels]
        zb['A'] = [f32(F * h * w, an) for h, w in levels]
        zb['bnew'] = [f32(F * h * w, 64) for h, w in levels]
        zb['ze'] = f32(F * levels[3][0] * levels[3][1], 128)
        zb['o32'] = h16(F, nh, nw, 32)
        zb['d'] = f32(F, nh, nw)
        self._extra_zbuffers(zb, F, levels)
        self._zbufs, self._zbuf_key = zb, key
        return zb

    def _extra_zbuffers(self, zb, F, levels):
        pass

    # ---- forward -------------------------------------------------------------------------------------------------------
    def _lin(self, a, lda, wb, M, N, K, out=None, ldc=None, act=_lib.ACT_NONE, f32out=None, resid=None):
        wt, bias = wb
        if resid is not None:
            self.ops.gemm(a, lda, wt, K, M, N, K, epi=_lib.EPI_RESID_F32, bias=bias, X=resid, ldx=N, gamma=self.z['ones128'])
        elif f32out is not None:
            self.ops.gemm(a, lda, wt, K, M, N, K, epi=_lib.EPI_STORE_F32, act=act, bias=bias, X=f32out, ldx=N)
        else:
            self.ops.gemm(a, lda, wt, K, M, N, K, act=act, bias=bias, C=out, ldc=ldc or N)

    def forward_batch(self, rgb, net_w, net_h=None, out_hw=None):
        """rgb: uint8 CUDA [B,H,W,3] -> float32 CUDA [B,H,W] metric depth (what estimatezoedepth returns; invert = True)."""
        import torch
        L = self.ops.L
        ops = self.ops
        st = _lib.stream_ptr
        B, H, W, _ = rgb.shape
        net_h = net_h if net_h is not None else net_w
        pad_h, pad_w = int(np.sqrt(H / 2) * 3.0), int(np.sqrt(W / 2) * 3.0)       # depth_model.py:80-82 (fh = fw = 3)
        Hp, Wp = H + 2 * pad_h, W + 2 * pad_w
        nw, nh = midas_net_size(Wp, Hp, net_w, net_h)                               # PrepForMidas: keep aspect, x32, "minimal"
        F = 2 * B
        b = self._buffers(F, nh, nw)
        _lib.check(L.dm_zoe_preprocess_patchify(rgb.data_ptr(), B, H, W, pad_h, pad_w, nh, nw, self.PATCH, b['patches'].data_ptr(), self.kpad, st()),
                   "dm_zoe_preprocess_patchify")
        ops.launches += 1
        self.run_network(b, F, nh, nw)
        zb = self._zbuffers(F, nh, nw, b)
        Fp = self.Fp
        # out_conv activation (MidasCore hooks output_conv[3], the 32-channel ReLU)
        t = b['up_sizes'][3]
        ops.conv3x3(b['path'][3], F, t[0], t[1], Fp, self.w['oc1_w'], self.F2p, bias=self.w['oc1_b'], C=b['oc1'])
        ops.resize_nhwc(b['oc1'], F, t[0], t[1], self.F2p, b['oc1u'], nh, nw)
        ops.conv3x3(b['oc1u'], F, nh, nw, self.F2p, self.z['oc2_w'], 32, act=_lib.ACT_RELU, bias=self.z['oc2_b'], C=zb['o32'])
        # x = conv2(bottleneck) (zoedepth_nk_v1.py:176-178, zoedepth_v1.py:145-146)
        self._lin(b['l'][3], Fp, self.z['conv2'], F * zb['n0'], Fp, Fp, out=zb['x16'])
        self._metric_head(b, zb, F, nh, nw)                 # -> zb['d'], metric depth per forward at the net size
        # un-pad / un-flip / average (depth_model.py:88-129)
        out = torch.empty(B, H, W, dtype=torch.float32, device=self.device)
        _lib.check(L.dm_zoe_tta_combine(zb['d'].data_ptr(), B, nh, nw, pad_h, pad_w, H, W, out.data_ptr(), st()), "dm_zoe_tta_combine")
        ops.launches += 1
        return out

    def _seed_embedding(self, zb, F):
        """seed projector (zoedepth_nk_v1.py:206, zoedepth_v1.py:153)"""
        n0, z, ph = zb['n0'], self.z, zb['p0'].shape[1]
        self._lin(zb['x16'], self.Fp, z['sproj'][0], F * n0, ph, self.Fp, out=zb['p0'], act=_lib.ACT_RELU)
        self._lin(zb['p0'], ph, z['sproj'][1], F * n0, 128, ph, out=zb['pemb'])

    def _attractor_levels(self, b, zb, F, attract):
        """the four projector + attractor levels (zoedepth_nk_v1.py:207-214, zoedepth_v1.py:156-161).  attract(i, A, b_prev, hp,
        wp, h, w) runs level i's attractor kernel from the GEMM output A, writing zb['bnew'][i].  Returns the last level's size."""
        z, Fp = self.z, self.Fp
        L = self.ops.L
        bprev, pemb, (hp, wp) = zb['bprev'], zb['pemb'], b['sizes'][3]
        ph = zb['t'][0].shape[1]
        for i, (h, w) in enumerate(zb['levels']):
            M = F * h * w
            aw, an = z['att'][i][0][0].shape[0], z['att'][i][1][0].shape[0]
            self._lin(b['path'][i], Fp, z['proj'][i][0], M, ph, Fp, out=zb['t'][i], act=_lib.ACT_RELU)
            self._lin(zb['t'][i], ph, z['proj'][i][1], M, 128, ph, out=zb['bemb'][i])
            _lib.check(L.dm_resize_add_nhwc_f16(zb['bemb'][i].data_ptr(), pemb.data_ptr(), F, hp, wp, 128, zb['xin'][i].data_ptr(), h, w,
                                                _lib.stream_ptr()), "dm_resize_add_nhwc_f16")
            self._lin(zb['xin'][i], 128, z['att'][i][0], M, aw, 128, out=zb['a0'][i], act=_lib.ACT_RELU)
            self._lin(zb['a0'][i], aw, z['att'][i][1], M, an, aw, f32out=zb['A'][i])
            attract(i, zb['A'][i], bprev, hp, wp, h, w)
            self.ops.launches += 2
            bprev, pemb, (hp, wp) = zb['bnew'][i], zb['bemb'][i], (h, w)
        return hp, wp

    def _metric_head(self, b, zb, F, nh, nw):
        L = self.ops.L
        ops, z = self.ops, self.z
        st = _lib.stream_ptr
        E_, A_ = _lib, _lib
        n0, S = zb['n0'], zb['S']
        lin = self._lin
        # ---- router: PatchTransformerEncoder (patch size 1) + MLP classifier (:186-195) ----
        lin(zb['x16'], self.Fp, z['emb'], F * n0, 128, self.Fp, out=zb['emb'])
        ops.tokens(zb['emb'], z['zeros128'], self._router_pe(S), zb['X'], F, n0, 128)
        _lib.check(L.dm_cast_f32_f16(zb['X'].data_ptr(), F * S * 128, zb['h'].data_ptr(), st()), "dm_cast_f32_f16")
        ops.launches += 1
        for lay in z['layers']:
            lin(zb['h'], 128, (lay['in_w'], lay['in_b']), F * S, 384, 128, out=zb['qkv'])
            _lib.check(L.dm_attention_small_f16(zb['qkv'].data_ptr(), F, S, ZOE_CONFIG['router_heads'], 1.0 / math.sqrt(32.0), zb['att'].data_ptr(), st()),
                       "dm_attention_small_f16")
            lin(zb['att'], 128, lay['out'], F * S, 128, 128, resid=zb['X'])
            _lib.check(L.dm_layernorm_post_f16(zb['X'].data_ptr(), F * S, 128, lay['n1'][0].data_ptr(), lay['n1'][1].data_ptr(), 1e-5, zb['h'].data_ptr(), st()),
                       "dm_layernorm_post_f16")
            lin(zb['h'], 128, lay['l1'], F * S, 1024, 128, out=zb['ff'], act=A_.ACT_RELU)
            lin(zb['ff'], 1024, lay['l2'], F * S, 128, 1024, resid=zb['X'])
            _lib.check(L.dm_layernorm_post_f16(zb['X'].data_ptr(), F * S, 128, lay['n2'][0].data_ptr(), lay['n2'][1].data_ptr(), 1e-5, zb['h'].data_ptr(), st()),
                       "dm_layernorm_post_f16")
            ops.launches += 3
        lin(zb['h'], S * 128, z['cls0'], F, 128, 128, out=zb['c1'], act=A_.ACT_RELU)       # token 0 of every forward (row pitch S*128)
        lin(zb['c1'], 128, z['cls2'], F, 32, 128, f32out=zb['logits'])
        lg = zb['logits']
        # ---- seed bins + seed embedding (:197-206) ----
        lin(zb['x16'], self.Fp, z['seed0'], F * n0, 128, self.Fp, out=zb['s0'], act=A_.ACT_RELU)
        lin(zb['s0'], 128, z['seed2'], F * n0, 128, 128, f32out=zb['seed'])
        _lib.check(L.dm_zoe_select_softplus(zb['seed'].data_ptr(), 128, lg.data_ptr(), 32, F, n0, zb['bprev'].data_ptr(), st()), "dm_zoe_select_softplus")
        self._seed_embedding(zb, F)
        ops.launches += 1
        # ---- attractor levels (:207-214) ----
        def attract(i, A, bprev, hp, wp, h, w):
            _lib.check(L.dm_zoe_attractor(A.data_ptr(), 64, lg.data_ptr(), 32, bprev.data_ptr(), F, hp, wp, h, w, zb['bnew'][i].data_ptr(), st()),
                       "dm_zoe_attractor")
        hp, wp = self._attractor_levels(b, zb, F, attract)
        bprev = zb['bnew'][3]
        # ---- conditional log-binomial + expectation (:216-236) ----
        we, wo, b0, w2c, b2c = z['clb']
        ops.gemm(zb['bemb'][3], 128, we, 128, F * hp * wp, 128, 128, epi=E_.EPI_STORE_F32, X=zb['ze'], ldx=128)
        _lib.check(L.dm_zoe_clb_final(zb['o32'].data_ptr(), 32, zb['ze'].data_ptr(), 128, bprev.data_ptr(), lg.data_ptr(), 32, wo.data_ptr(), b0.data_ptr(),
                                      w2c.data_ptr(), b2c.data_ptr(), F, nh, nw, hp, wp, ZOE_CONFIG['min_temp'], ZOE_CONFIG['max_temp'],
                                      zb['d'].data_ptr(), st()), "dm_zoe_clb_final")
        ops.launches += 1


# ZoeDepth-N / -K as the reference builds them: get_config("zoedepth", "infer"[, config_version="kitti"]) -> ZoeDepth(core, **config)
# (src/depthmap_generation.py:196-205, dzoedepth/models/zoedepth/config_zoedepth*.json).  min / max depth are the constructor's
# defaults for BOTH (infer mode merges no dataset config, so K does not get KITTI's 80); the attractor counts are passed by keyword,
# so the levels really have 16, 8, 4, 1 attractors.
ZOE_SINGLE = {7: dict(name='zoedepth_n', normed=False, n_attractors=(16, 8, 4, 1), min_depth=1e-3, max_depth=10.0),
              8: dict(name='zoedepth_k', normed=True, n_attractors=(16, 8, 4, 1), min_depth=1e-3, max_depth=10.0)}


class ZoeDepthEngine(ZoeDepthNKEngine):
    """ZoeDepth-N (model type 7) and ZoeDepth-K (type 8): the single metric head of ZoeDepth.forward
    (zoedepth/zoedepth_v1.py:120-186) on the core, pre-processing and pad + flip TTA of ZoeDepthNKEngine.  No router.
      N: softplus bin centres (SeedBinRegressorUnnormed + AttractorLayerUnnormed).
      K: normed bin centres (SeedBinRegressor + AttractorLayer): widths normalised over the 64 bins and accumulated into
         centres in [min, max]; each attractor level sorts and clips the scaled centres, the next level gets the unsorted
         normed ones.
    The log-binomial MLP also sees the core's own relative depth, relu(output_conv.4(out_conv)), as a 33rd input channel.
    A missing or mis-shaped head weight raises ValueError naming the key."""

    def __init__(self, state_dict, model_type, device, core_name='beitl16_384'):
        if model_type not in ZOE_SINGLE:
            raise ValueError(f"ZoeDepthEngine builds model types 7 (ZoeDepth-N) and 8 (ZoeDepth-K), not {model_type}")
        self.model_type = model_type
        self.zconf = ZOE_SINGLE[model_type]
        super().__init__(state_dict, device, core_name)

    def _pack(self, sd):
        for k, shape in (('scratch.output_conv.4.weight', (1, 32, 1, 1)), ('scratch.output_conv.4.bias', (1,))):
            if k not in sd:
                raise ValueError(f"ZoeDepth checkpoint: core.core.{k} is missing")
            if tuple(sd[k].shape) != shape:
                raise ValueError(f"ZoeDepth checkpoint: core.core.{k} has shape {tuple(sd[k].shape)}, expected {shape}")
        self._rel_w = sd['scratch.output_conv.4.weight'].detach().float().reshape(32)
        self._rel_b = float(sd['scratch.output_conv.4.bias'].detach().float().reshape(-1)[0])
        super()._pack(sd)

    def head_shapes(self):
        """{key: (out, in)} of every 1x1 conv of the single head (weights [out, in, 1, 1], biases [out])."""
        feat, emb, nb = self.cfg['features'], 128, 64
        per = 2 if self.zconf['normed'] else 1
        s = {'conv2': (feat, feat), 'seed_bin_regressor._net.0': (256, feat), 'seed_bin_regressor._net.2': (nb, 256),
             'seed_projector._net.0': (128, feat), 'seed_projector._net.2': (emb, 128),
             'conditional_log_binomial.mlp.0': ((33 + emb) // 2, 33 + emb), 'conditional_log_binomial.mlp.2': (4, (33 + emb) // 2)}
        for i, n in enumerate(self.zconf['n_attractors']):
            s[f'projectors.{i}._net.0'] = (128, feat)
            s[f'projectors.{i}._net.2'] = (emb, 128)
            s[f'attractors.{i}._net.0'] = (128, emb)
            s[f'attractors.{i}._net.2'] = (per * n, 128)
        return s

    def _pack_head(self, sd):
        import torch
        dev = self.device
        for key, (o, i) in self.head_shapes().items():
            for suffix, shape in (('.weight', (o, i, 1, 1)), ('.bias', (o,))):
                if key + suffix not in sd:
                    raise ValueError(f"ZoeDepth checkpoint: {key + suffix} is missing")
                if tuple(sd[key + suffix].shape) != shape:
                    raise ValueError(f"ZoeDepth checkpoint: {key + suffix} has shape {tuple(sd[key + suffix].shape)}, expected {shape}")
        z = {}
        W = lambda key, rows=None, cols=None: self._hw(sd, key, rows, cols)
        Bv = lambda key, n=None: self._hb(sd, key, n)
        z['ones128'] = torch.ones(128, dtype=torch.float32, device=dev)
        z['conv2'] = (W('conv2'), Bv('conv2'))
        z['seed0'] = (W('seed_bin_regressor._net.0'), Bv('seed_bin_regressor._net.0'))
        z['seed2'] = (W('seed_bin_regressor._net.2'), Bv('seed_bin_regressor._net.2'))
        z['sproj'] = ((W('seed_projector._net.0'), Bv('seed_projector._net.0')), (W('seed_projector._net.2'), Bv('seed_projector._net.2')))
        z['proj'] = [((W(f'projectors.{i}._net.0'), Bv(f'projectors.{i}._net.0')), (W(f'projectors.{i}._net.2'), Bv(f'projectors.{i}._net.2'))) for i in range(4)]
        # attractor GEMM output padded to 32 columns (N: n softplus inputs, K: 2n ReLU inputs of which the even ones are used)
        z['att'] = [((W(f'attractors.{i}._net.0'), Bv(f'attractors.{i}._net.0')), (W(f'attractors.{i}._net.2', rows=32), Bv(f'attractors.{i}._net.2', 32)))
                    for i in range(4)]
        # conditional log-binomial: mlp.0 [80, 161] split into out_conv (32), relative depth (1) and bin embedding (128) columns;
        # the last part is a GEMM before the up-sampling, as for NK
        m0 = sd['conditional_log_binomial.mlp.0.weight'].detach().to(dev).float().reshape(80, 161)
        we = torch.zeros(128, 128, dtype=torch.float16, device=dev)
        we[:80] = m0[:, 33:].to(torch.float16)
        f32 = lambda t: t.detach().to(dev).float().contiguous()
        z['clb'] = (we, f32(m0[:, :32].t()), f32(m0[:, 32]), f32(sd['conditional_log_binomial.mlp.0.bias']),
                    f32(sd['conditional_log_binomial.mlp.2.weight'].reshape(4, 80)), f32(sd['conditional_log_binomial.mlp.2.bias']))
        z['rel'] = (self._rel_w.to(dev).contiguous(), self._rel_b)
        self._pack_out_conv(z)
        self.z = z

    def _extra_zbuffers(self, zb, F, levels):
        import torch
        if self.zconf['normed']:
            h, w = levels[3]
            zb['Bc'] = torch.empty(F * h * w, 64, dtype=torch.float32, device=self.device)    # sorted, clipped centres of the last level
        else:
            zb['head0'] = torch.zeros(F, 2, dtype=torch.float32, device=self.device)          # select_softplus with head 0 for every forward

    def _metric_head(self, b, zb, F, nh, nw):
        L = self.ops.L
        ops, z, c = self.ops, self.z, self.zconf
        st = _lib.stream_ptr
        n0, Fp = zb['n0'], self.Fp
        mn, mx = c['min_depth'], c['max_depth']
        # ---- seed bins (zoedepth_v1.py:147-151) + seed embedding ----
        s0w, nb = z['seed0'][0].shape[0], z['seed2'][0].shape[0]
        self._lin(zb['x16'], Fp, z['seed0'], F * n0, s0w, Fp, out=zb['s0'], act=_lib.ACT_RELU)
        self._lin(zb['s0'], s0w, z['seed2'], F * n0, nb, s0w, f32out=zb['seed'])
        if c['normed']:
            _lib.check(L.dm_zoe_seed_normed(zb['seed'].data_ptr(), nb, F * n0, mn, mx, zb['bprev'].data_ptr(), st()), "dm_zoe_seed_normed")
        else:
            _lib.check(L.dm_zoe_select_softplus(zb['seed'].data_ptr(), nb, zb['head0'].data_ptr(), 2, F, n0, zb['bprev'].data_ptr(), st()),
                       "dm_zoe_select_softplus")
        ops.launches += 1
        self._seed_embedding(zb, F)

        # ---- attractor levels (:156-161) ----
        def attract(i, A, bprev, hp, wp, h, w):
            Bs = zb['Bc'].data_ptr() if (c['normed'] and i == 3) else None
            _lib.check(L.dm_zoe_attractor_single(A.data_ptr(), A.shape[1], c['n_attractors'][i], int(c['normed']), bprev.data_ptr(), F, hp, wp, h, w,
                                                 mn, mx, zb['bnew'][i].data_ptr(), Bs, st()), "dm_zoe_attractor_single")
        hp, wp = self._attractor_levels(b, zb, F, attract)
        centres = zb['Bc'] if c['normed'] else zb['bnew'][3]
        # ---- conditional log-binomial on cat(out_conv, rel_depth, b_emb) + expectation (:163-186) ----
        we, wo, wr, b0, w2c, b2c = z['clb']
        ops.gemm(zb['bemb'][3], 128, we, 128, F * hp * wp, 128, 128, epi=_lib.EPI_STORE_F32, X=zb['ze'], ldx=128)
        _lib.check(L.dm_zoe_clb_final_single(zb['o32'].data_ptr(), 32, zb['ze'].data_ptr(), 128, centres.data_ptr(), wo.data_ptr(), wr.data_ptr(),
                                             b0.data_ptr(), w2c.data_ptr(), b2c.data_ptr(), z['rel'][0].data_ptr(), z['rel'][1], F, nh, nw, hp, wp,
                                             ZOE_CONFIG['min_temp'], ZOE_CONFIG['max_temp'], zb['d'].data_ptr(), st()), "dm_zoe_clb_final_single")
        ops.launches += 1


class ModelHolder:
    """Same public surface as the reference's ModelHolder (src/depthmap_generation.py:40-403)."""

    def __init__(self):
        self.depth_model = None
        self.pix2pix_model = None
        self.depth_model_type = None
        self.device = None
        self.offloaded = False
        self.resize_mode = None
        self.normalization = None
        self.tiling_mode = False
        # settings injected by update_settings(**ops) in the reference (src/backbone.py:36-49,132-137)
        self.no_half = False
        self.precision = "autocast"
        self.boost_rmax = 1600
        self.weights_provider = None  # callable(model_type) -> state_dict; default: torch.load of ./models/... like the reference

    def update_settings(self, **kvargs):
        for k, v in kvargs.items():
            setattr(self, k, v)

    def ensure_models(self, model_type, device, boost: bool, tiling_mode: bool = False):
        if model_type == -1 or model_type is None:
            self.unload_models()
            return
        if (model_type != self.depth_model_type or boost != (self.pix2pix_model is not None) or device != self.device or
                tiling_mode != self.tiling_mode):
            self.unload_models()
            self.load_models(model_type, device, boost, tiling_mode)
        self.reload()

    def load_models(self, model_type, device, boost: bool, tiling_mode: bool = False):
        """Ensure that the depth model is loaded (reference: src/depthmap_generation.py:76-301)."""
        import torch
        _lib.require_cuda()
        if boost and model_type != 0:
            raise NotImplementedError("BOOST is built for the reference's default base network only, LeReS res101 (model type 0); "
                                      "the other base networks (estimatemidasBoost etc.) are not implemented in depthmap_b200")
        if tiling_mode:
            raise NotImplementedError("tiling_mode (circular conv padding) is not implemented in depthmap_b200 yet")
        if getattr(self, "no_half", False):
            # reference: `no_half` keeps the network in fp32 (src/depthmap_generation.py:268-275).  The B200 path feeds the tensor
            # cores fp16 operands (fp32 accumulation, fp32 residual stream) and has no fp32-operand variant: say so instead of
            # silently ignoring the setting
            raise NotImplementedError("no_half (fp32 network) is not implemented in depthmap_b200: the tensor-core path uses fp16 operands "
                                      "with fp32 accumulation; unset the setting")
        if model_type in (12, 13, 14):
            letter = {12: 's', 13: 'b', 14: 'l'}[model_type]
            if self.weights_provider is not None:
                sd = self.weights_provider(model_type)
            else:
                model_path = f"./models/depth_anything_v2/depth_anything_v2_vit{letter}.pth"
                if not os.path.exists(model_path):
                    raise FileNotFoundError(f"{model_path} not found (depthmap_b200 does not download checkpoints)")
                sd = torch.load(model_path, map_location='cpu')
            model = NativeDepthModel(sd, model_type, torch.device(device))
        elif model_type in (1, 2):  # dpt_beit_large_512 / dpt_beit_large_384 (MiDaS 3.1)
            name = {1: 'beitl16_512', 2: 'beitl16_384'}[model_type]
            if self.weights_provider is not None:
                sd = self.weights_provider(model_type)
            else:
                model_path = "./models/midas/" + {1: 'dpt_beit_large_512.pt', 2: 'dpt_beit_large_384.pt'}[model_type]
                if not os.path.exists(model_path):
                    raise FileNotFoundError(f"{model_path} not found (depthmap_b200 does not download checkpoints)")
                sd = torch.load(model_path, map_location='cpu')
                if "optimizer" in sd:       # dmidas/base_model.py:13: training checkpoints wrap the weights
                    sd = sd["model"]
            model = NativeDepthModel(sd, model_type, torch.device(device))
        elif model_type == 0:  # res101 (LeReS)
            if self.weights_provider is not None:
                sd = self.weights_provider(model_type)
            else:
                model_path = "./models/leres/res101.pth"
                if not os.path.exists(model_path):
                    raise FileNotFoundError(f"{model_path} not found (depthmap_b200 does not download checkpoints)")
                sd = torch.load(model_path, map_location='cpu')
                if "depth_model" in sd:      # src/depthmap_generation.py:113-116: strip_prefix_if_present(checkpoint['depth_model'], "module.")
                    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in sd["depth_model"].items()}
            model = LeresEngine(sd, torch.device(device))
            if boost:      # reference :284-299: the pix2pix merge network ('latest_net_G.pth', netG = unet_1024, norm none)
                from .boost import BoostPipeline, UnetMergeEngine
                if self.weights_provider is not None:
                    psd = self.weights_provider("pix2pix")
                else:
                    p2p_path = "./models/pix2pix/latest_net_G.pth"
                    if not os.path.exists(p2p_path):
                        raise FileNotFoundError(f"{p2p_path} not found (depthmap_b200 does not download checkpoints)")
                    psd = torch.load(p2p_path, map_location='cpu')
                self.pix2pix_model = BoostPipeline(model, UnetMergeEngine(psd, torch.device(device)), torch.device(device), model_type)
        elif model_type == 3:  # dpt_large_384 (MiDaS 3.0)
            if self.weights_provider is not None:
                sd = self.weights_provider(model_type)
            else:
                model_path = "./models/midas/dpt_large-midas-2f21e586.pt"
                if not os.path.exists(model_path):
                    raise FileNotFoundError(f"{model_path} not found (depthmap_b200 does not download checkpoints)")
                sd = torch.load(model_path, map_location='cpu')
                if "optimizer" in sd:
                    sd = sd["model"]
            model = NativeDepthModel(sd, model_type, torch.device(device))
        elif model_type in (7, 8, 9):  # zoedepth_n / _k / _nk (src/depthmap_generation.py:196-226: ZoeD_M12_N.pt / _K.pt / _NK.pt)
            if self.weights_provider is not None:
                sd = self.weights_provider(model_type)
            else:
                model_path = "./models/zoedepth/" + {7: "ZoeD_M12_N.pt", 8: "ZoeD_M12_K.pt", 9: "ZoeD_M12_NK.pt"}[model_type]
                if not os.path.exists(model_path):
                    raise FileNotFoundError(f"{model_path} not found (depthmap_b200 does not download checkpoints)")
                sd = torch.load(model_path, map_location='cpu')
                if "model" in sd:           # dzoedepth/models/model_io.py:52-53
                    sd = sd["model"]
            if model_type == 9:
                model = ZoeDepthNKEngine(sd, torch.device(device))
            else:
                model = ZoeDepthEngine(sd, model_type, torch.device(device))
        else:
            raise NotImplementedError(f"model_type {model_type} is not implemented in depthmap_b200 yet "
                                      f"(implemented: 0 = LeReS res101; 1, 2 = DPT-BEiT-L 512/384; 3 = DPT-Large 384; 7, 8, 9 = ZoeDepth-N/K/NK; "
                                      f"12, 13, 14 = Depth-Anything-V2 S/B/L)")
        self.depth_model = model
        self.depth_model_type = model_type
        self.resize_mode = "minimal"
        self.normalization = None
        self.tiling_mode = tiling_mode
        self.device = device

    @staticmethod
    def get_default_net_size(model_type):
        sizes = {0: [448, 448], 1: [512, 512], 2: [384, 384], 3: [384, 384], 4: [384, 384], 5: [384, 384], 6: [256, 256],
                 7: [384, 512], 8: [384, 768], 9: [384, 512], 10: [768, 768], 11: [518, 518], 12: [518, 518], 13: [518, 518],
                 14: [518, 518]}
        if model_type in sizes:
            return sizes[model_type]
        return [512, 512]

    def offload(self):
        """The reference swaps the model to host RAM between calls to free VRAM for Stable Diffusion (:344-348).
        Packed weights stay resident on a 180 GB part; the flag is kept so callers observe the same state machine."""
        if self.device is not None and not self.offloaded:
            self.offloaded = True

    def reload(self):
        if self.offloaded:
            self.offloaded = False

    def move_models_to(self, device):
        pass

    def unload_models(self):
        if self.depth_model is not None or self.pix2pix_model is not None:
            if hasattr(self.depth_model, "close"):
                self.depth_model.close()
            self.depth_model = None
            self.pix2pix_model = None
            gc.collect()
            try:
                import torch
                torch.cuda.empty_cache()
            except Exception:
                pass
        self.depth_model_type = None
        self.device = None

    # ---- prediction ------------------------------------------------------------------------------------------------
    def get_raw_prediction_batch(self, rgb, net_width, net_height):
        """uint8 CUDA [B,H,W,3] -> (float32 CUDA [B,H,W], invert flag).  Batched form of get_raw_prediction."""
        if self.depth_model is None:
            raise RuntimeError("no depth model loaded; call ensure_models first")
        if self.pix2pix_model is not None:
            # boost: estimateboost works on one image at a time (its resolutions and patches depend on the image); the net size is ignored
            import torch
            preds = [self.pix2pix_model.run(rgb[i].cpu().numpy(), self.boost_rmax, to_host=False) for i in range(rgb.shape[0])]
            return torch.stack(preds), self.depth_model_type in [0, 7, 8, 9, 10]
        if self.depth_model_type in (0, 1, 2, 3, 7, 8, 9, 12, 13, 14):
            pred = self.depth_model.forward_batch(rgb, net_width, net_height)
        else:
            raise NotImplementedError(f"model_type {self.depth_model_type}")
        return pred, self.depth_model_type in [0, 7, 8, 9, 10]

    def get_raw_prediction(self, input, net_width, net_height):
        """Get prediction from the model currently loaded by the ModelHolder object (reference :375-403)."""
        import torch
        dev = _lib.require_cuda()
        img = np.asarray(input)
        if img.ndim != 3 or img.shape[2] != 3 or img.dtype != np.uint8:
            img = np.asarray(input.convert('RGB')) if hasattr(input, 'convert') else img
        if self.pix2pix_model is not None:       # boost: net_width / net_height are ignored (reference :376-377, :399-401)
            return self.pix2pix_model.run(img, self.boost_rmax), self.depth_model_type in [0, 7, 8, 9, 10]
        t = torch.from_numpy(np.ascontiguousarray(img)).to(dev).unsqueeze(0)
        pred, invert = self.get_raw_prediction_batch(t, net_width, net_height)
        return pred[0].cpu().numpy(), invert
