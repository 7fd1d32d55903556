"""B200-native ``Unet`` with the reference's constructor / forward API.

``Unet`` is only a parameter container with the reference's ``state_dict`` layout
(imagen_pytorch.py:1112-1442).  The arithmetic lives in ``UnetPlan``: a *compiled launch
plan* -- weights packed once into the layouts the sm_100a kernels want, a static
activation arena, and a flat list of C-ABI kernel launches that the samplers capture into
a CUDA graph and replay per denoising step.  Everything that does not depend on the
denoising step (text projection, PerceiverResampler, per-layer context K/V, null
conditioning) is hoisted into ``UnetPlan.prepare`` and runs once per ``sample()`` call.

There is no torch / CPU fallback for the forward pass: without libb200imagen.so and an
sm_100 device, ``forward`` raises.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from functools import partial

import torch
import torch.nn.functional as F
from torch import nn

from . import _lib, ops
from ._lib import Src, TimeRowJob
from .params import UnetArch, param_table, build_param_tree, pad_attention_heads

LOG2E = 1.4426950408889634
BF16 = torch.bfloat16


def _ceil(a, b):
    return (a + b - 1) // b * b


class Rows:
    """NHWC pixel rows: [rows, C] bf16 with row stride ld; (H, W) is the pixel grid per sample."""
    __slots__ = ('t', 'C', 'ld', 'H', 'W', 'call')

    def __init__(self, t, C, H=1, W=1):
        self.t, self.C, self.ld, self.H, self.W = t, C, t.shape[-1], H, W
        self.call = None      # the GemmCall that produces these rows (a later consumer may attach its pre-norm to that epilogue)

    @property
    def ptr(self):
        return self.t.data_ptr()

    @property
    def rows(self):
        return self.t.shape[0]


class _Arena:
    """Bump allocator over a few large device chunks.  zero=True: chunks come from torch.zeros (activations; padded channels and
    prefix rows rely on it).  staged=True: every chunk has a host twin that `put` fills; `flush` uploads it with one memcpy, so
    packing ~300 weight operands costs no kernel launches (the driver's launch trace then shows the product kernels)."""
    ALIGN = 1024

    def __init__(self, device, *, zero, chunk, staged=False):
        self.device, self.zero, self.chunk, self.staged = device, zero, chunk, staged
        self.chunks, self.hosts, self.off = [], [], 0

    def _grow(self, nbytes):
        size = max(min(self.chunk, (32 << 20) << (2 * len(self.chunks))), nbytes)    # 32 MB, 128 MB, 512 MB, ... up to `chunk`
        self.chunks.append((torch.zeros if self.zero else torch.empty)(size, dtype=torch.uint8, device=self.device))
        if self.staged:
            self.hosts.append(torch.empty(size, dtype=torch.uint8))
        self.off = 0

    def _take(self, nbytes):
        nbytes = max(int(nbytes), 1)
        if not self.chunks or self.off + nbytes > self.chunks[-1].numel():
            self._grow(nbytes)
        o = self.off
        self.off = (o + nbytes + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        return len(self.chunks) - 1, o

    def alloc(self, shape, dtype):
        shape = tuple(int(v) for v in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        n = 1
        for v in shape:
            n *= v
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        c, o = self._take(nbytes)
        return self.chunks[c][o:o + nbytes].view(dtype).view(shape)

    def put(self, host: torch.Tensor):
        assert self.staged and host.device.type == 'cpu'
        host = host.contiguous()
        nbytes = host.numel() * host.element_size()
        c, o = self._take(nbytes)
        if nbytes:
            self.hosts[c][o:o + nbytes].copy_(host.view(-1).view(torch.uint8))
        return self.chunks[c][o:o + max(nbytes, 0)].view(host.dtype).view(host.shape)

    def flush(self):
        for i, (d, h) in enumerate(zip(self.chunks, self.hosts)):
            used = self.off if i == len(self.chunks) - 1 else d.numel()
            d[:used].copy_(h[:used])
        self.hosts = []

    def nbytes(self):
        return sum(c.numel() for c in self.chunks)


class UnetPlan:
    """Launch plan of one U-Net for a fixed (rows R, images B, H, W, schedule slots S)."""

    def __init__(self, unet: 'Unet', R, B, H, W, n_slots, device, gemm_impl=_lib.IMPL_TCGEN05):
        self.lib = _lib.load()
        self.arch = a = unet.arch
        self.R, self.B, self.H, self.W, self.S = R, B, H, W, n_slots
        self.device = device
        self.impl = gemm_impl
        assert R in (B, 2 * B)
        nlev = a.num_levels
        div = 2 ** (nlev if a.memory_efficient else nlev - 1)
        if H % div or W % div:
            raise ValueError(f'image size {H}x{W} must be divisible by {div} for this U-Net')
        # device-side fp32 views of the parameters (no copy when the module already lives on `device`): read by prepare()
        self.sd = {k: v.detach().to(device=device, dtype=torch.float32).contiguous() for k, v in unet.state_dict().items()}
        # host copies for weight packing: the packed bf16 / fp32 operands are assembled on the host into a few staging chunks and
        # reach the device with one memcpy per chunk, so building a plan launches (almost) no kernels of its own
        self.sdc = {k: v.detach().to(device='cpu', dtype=torch.float32) for k, v in unet.state_dict().items()}
        self.fingerprint = unet._fingerprint()
        self._keep, self._post = [], []
        self._act = _Arena(device, zero=True, chunk=1 << 30)      # activations / state: zero-filled chunks (one fill kernel per GiB)
        self._wts = _Arena(device, zero=False, chunk=1 << 28, staged=True)
        # heads narrower than 64 channels run zero-padded to 64 on the same kernels (params.pad_attention_heads); from here on both
        # parameter views describe 64-wide heads
        for k, v in pad_attention_heads(self.sdc, a.dim_head).items():
            self.sdc[k] = v
            self.sd[k] = self._wts.put(v)
        self.inner = a.heads * 64
        self._ops = []
        self._jobs = []
        self.cross_layers, self.self_layers = [], []
        # context geometry (Unet.forward :1656): [own time tokens | lowres time tokens, text tokens | null]
        self.ntt = a.num_time_tokens
        self.n_text = ((a.pool_latents + a.pool_mean_latents) if a.attn_pool else a.max_text_len) if a.cond_on_text else 0
        self.n_static = (self.ntt if a.lowres_cond else 0) + self.n_text
        self.n_ctx = self.ntt + self.n_static
        # per-step state
        self.x_in = self._zeros((B, a.channels, H, W), torch.float32)
        # self-conditioning input (imagen_pytorch.py:1541-1543): the samplers' step kernels write x_start here, zeros before the first step
        self.sc_in = self._zeros((B, a.channels, H, W), torch.float32) if a.self_cond else None
        self.lowres_img = self._zeros((B, a.channels, H, W), torch.float32) if a.lowres_cond else None
        # conditioning image (Unet(cond_images_channels > 0), :1553-1560): static over the t-loop, resized once in prepare()
        self.cond_img = self._zeros((B, a.cond_images_channels, H, W), torch.float32) if a.cond_images_channels else None
        self.pred = self._zeros((R, a.channels_out, H, W), torch.float32)
        self.slots = self._zeros((R,), torch.int32)
        self.time_cond_table = self._zeros((n_slots, a.time_cond_dim), torch.float32)
        self.text_hiddens = self._zeros((R, a.time_cond_dim), torch.float32)
        self._scratch = None
        self.sampler_state = {}      # persistent sampler buffers + captured step graphs (imagen.py / elucidated.py)
        self.fuse_norm = os.environ.get('B200_IMAGEN_FUSE_NORM', '1') != '0'
        self.n_fused = 0             # norms that run inside a GEMM epilogue instead of their own kernel
        self._build()

    # ------------------------------------------------------------------ small helpers
    def _zeros(self, shape, dtype=BF16):
        return self._act.alloc(shape, dtype)

    def _new(self, rows, C, H=1, W=1):
        return Rows(self._zeros((rows, C)), C, H, W)

    def _f32(self, t):
        """host fp32 tensor -> device copy (through the staged weight arena)."""
        return self._wts.put(t.to(dtype=torch.float32).contiguous())

    def _add(self, name, *args):
        self._ops.append((getattr(self.lib, name), args, name))

    def _scratch_ptr(self, nfloats):
        if nfloats <= 0:
            return None
        if self._scratch is None or self._scratch.numel() < nfloats:
            self._scratch = torch.empty(int(nfloats), dtype=torch.float32, device=self.device)
            self._keep.append(self._scratch)
        return self._scratch.data_ptr()

    def _row_fill(self, dst, row):
        """dst[r, :] = row (host fp32 -> bf16) for every r, applied after the staged weights have reached the device."""
        self._post.append((dst, self._wts.put(row.to(BF16).contiguous())))

    def _pack(self, mats, N):
        return self._wts.put(ops.pack_weight(mats, N, 'cpu'))

    def _gemm(self, srcs, segs, grid, wpacked, N, out, *, bias=None, residual=None, out2=None, l2_scale=None, ldc=None, **epi):
        gB, gH, gW = grid
        M, npad = gB * gH * gW, _lib.npad(N)
        if self.impl == _lib.IMPL_SIMT_CHECKER:
            nscratch, ksplit = M * npad, 1
        else:   # split-K workspace when the library would split this shape (few row tiles, long K: the 8x8 levels)
            ktot = sum(-(-srcs[g[0]].C // 64) * 64 for g in segs)
            ksplit = self.lib.b200_conv_gemm_splitk(gB, gH, gW, N, ktot)
            nscratch = ksplit * M * npad if ksplit > 1 else 0
        call = ops.GemmCall(
            [(s.ptr, s.C, s.ld) for s in srcs], segs, grid, wpacked, N, out if (out is None or isinstance(out, int)) else out.data_ptr(),
            bias=self._wts.put(ops.padded_bias(bias, N, 'cpu')) if bias is not None else None,
            residual=residual.ptr if residual is not None else None, ldr=residual.ld if residual is not None else 0,
            out2_ptr=(out2 if isinstance(out2, int) else out2.data_ptr()) if out2 is not None else None,
            l2_scale=l2_scale, ldc=ldc if ldc is not None else 0, impl=self.impl,
            scratch_ptr=self._scratch_ptr(nscratch), **epi)
        call.desc['ksplit'] = ksplit
        self._keep.append(call)
        self._ops.append((call.lib.b200_conv_gemm, call.args, 'b200_conv_gemm'))
        return call

    def _linear(self, x: Rows, W, N, out: Rows = None, out_raw=True, **epi):
        """pixel-row linear layer y = x @ W^T (W: [N, C]).  out_raw=False: only the fused norm output (epi: norm2...) is stored."""
        M = x.rows
        if out is None:
            out = self._new(M, N, x.H, x.W)
        wp = self._pack([W], N)
        out.call = self._gemm([x], [(0, 0, 0)], (1, 1, M), wp, N, out.t if out_raw else None, ldc=out.ld, **epi)
        return out

    def _conv_taps(self, k):
        return ops.conv_taps(k)

    def _conv(self, srcs, Wt, N, out, *, split=None, **epi):
        """k x k conv (pad k//2) over the channel concat of srcs; Wt: [N, sum C, k, k]; split = channel counts in Wt."""
        segs, mats = ops.conv_segments(Wt, split or [s.C for s in srcs])
        s0 = srcs[0]
        return self._gemm(srcs, segs, (self.R, s0.H, s0.W), self._pack(mats, N), N, out, **epi)

    # ---- norm fusion (north star: "GroupNorm+SiLU and time-embed FiLM scale/shift fused into the preceding conv epilogue").
    # Where one GEMM tile spans all channels (64 <= C <= 256) the per-pixel norm runs in the producing GEMM's epilogue
    # (b200_epilogue.norm1 / norm2) instead of a separate HBM round trip.  B200_IMAGEN_FUSE_NORM=0 plans the stand-alone kernels.
    def _fusable(self, C):
        return self.fuse_norm and self.impl == _lib.IMPL_TCGEN05 and 64 <= C <= 256 and C % 32 == 0

    def _attach_norm(self, x: Rows, kind, gt, **film):
        """Try to let x's producer GEMM also emit norm(x): returns the normalised Rows or None."""
        c = x.call
        if c is None or not self.fuse_norm or not c.norm_capable() or c.e.norm2 != 0:
            return None
        if isinstance(c, ops.GemmCall) and not self._fusable(x.C):             # a GEMM tile must span all channels; row kernels take any width
            return None
        out = self._new(x.rows, x.C, x.H, x.W)
        c.set_norm2(kind, gt, out.ptr, out.ld, **film)
        self.n_fused += 1
        return out

    def _prenorm_ln(self, x: Rows, g):
        """LayerNorm(x) * g feeding a linear layer: fused into x's producer when possible, else the row kernel."""
        out = self._attach_norm(x, _lib.NORM_LN, self._f32(g.flatten()))
        return out if out is not None else self._layernorm(x, g)

    def _rms_film_silu(self, srcs, gamma, din, skip, n, film_off=None):
        """ChanRMSNorm -> [FiLM] -> SiLU over the channel concat of srcs (Block, imagen_pytorch.py:683-691)."""
        gt = self._f32(gamma.flatten() * math.sqrt(din))
        film = {}
        if film_off is not None:
            film = dict(film_ptr=self.film.data_ptr() + 4 * film_off, film_ld=self.film.shape[1], rows_per_sample=n)
        if len(srcs) == 1:
            out = self._attach_norm(srcs[0], _lib.NORM_RMS_FILM_SILU, gt, **film)
            if out is not None:
                return out
        M = srcs[0].rows
        out = self._new(M, din, srcs[0].H, srcs[0].W)
        sa = (Src * len(srcs))(*[Src(s.ptr, s.C, s.ld) for s in srcs])
        self._keep.append(sa)
        self._add('b200_rmsnorm_film_silu', sa, len(srcs), skip, gt.data_ptr(), film.get('film_ptr'), film.get('film_ld', 0), n, out.ptr, out.ld, M)
        return out

    def _layernorm(self, x: Rows, g, residual: Rows = None):
        """LayerNorm(x) * g [+ residual] as a chained row kernel; a later consumer's norm may be attached to the same pass."""
        out = self._new(x.rows, x.C, x.H, x.W)
        gt = self._f32(g.flatten())
        if not self.fuse_norm:
            self._add('b200_layernorm', x.ptr, x.ld, gt.data_ptr(), None, 1e-5, residual.ptr if residual else None,
                      residual.ld if residual else 0, out.ptr, out.ld, x.rows, x.C)
            return out
        rc = ops.RowChainCall(x.ptr, x.ld, x.rows, x.C, norm1_g=gt, residual_ptr=residual.ptr if residual else None,
                              ldr=residual.ld if residual else 0, out_ptr=out.ptr, ldo=out.ld)
        self._keep.append(rc)
        self._ops.append((rc.lib.b200_row_chain, rc.args, 'b200_row_chain'))
        if residual is not None:          # (a bare pre-norm output feeds a GEMM: nothing to attach to)
            out.call = rc
        return out

    # ------------------------------------------------------------------ blocks
    def _resnet(self, p, srcs, dout, *, cross_heads=None, linear_cross=False, gca=False):
        """ResnetBlock.forward (imagen_pytorch.py:735-757); linear_cross: LinearCrossAttention instead of CrossAttention (:719)."""
        a, sd, R = self.arch, self.sdc, self.R
        Hc, Wc = srcs[0].H, srcs[0].W
        n = Hc * Wc
        M = R * n
        din = sum(s.C for s in srcs)
        skip = a.skip_scale if len(srcs) == 2 else 1.0
        # block1: ChanRMSNorm -> SiLU -> conv3x3 (:683-691); block2: ChanRMSNorm -> FiLM(scale+1, shift) -> SiLU -> conv3x3.
        # Both norms are emitted by the epilogue of the GEMM that produces their input when a tile spans all channels.
        a1 = self._rms_film_silu(srcs, sd[p + '.block1.norm.gamma'], din, skip, n)
        W1, b1 = sd[p + '.block1.project.weight'], sd[p + '.block1.project.bias']
        g2, film_off = sd[p + '.block2.norm.gamma'], self.film_offsets[p]
        if cross_heads is None and self._fusable(dout):
            # conv1's epilogue writes a2 = SiLU(FiLM(RMSNorm(h))) directly; h itself is never stored
            a2 = self._new(M, dout, Hc, Wc)
            self._conv([a1], W1, dout, None, bias=b1, norm2=_lib.NORM_RMS_FILM_SILU, norm2_g=self._f32(g2.flatten() * math.sqrt(dout)),
                       film_ptr=self.film.data_ptr() + 4 * film_off, film_ld=self.film.shape[1], rows_per_sample=n, out_norm_ptr=a2.ptr, ld_norm=a2.ld)
            self.n_fused += 1
        else:
            h = self._new(M, dout, Hc, Wc)
            h.call = self._conv([a1], W1, dout, h.t, ldc=h.ld, bias=b1)
            if cross_heads is not None:
                attn = self._linear_cross_attention if linear_cross else self._cross_attention
                a2 = attn(p + '.cross_attn', h, cross_heads, g2, film_off)
            else:
                a2 = self._rms_film_silu([h], g2, dout, 1.0, n, film_off)
        W2, b2 = sd[p + '.block2.project.weight'], sd[p + '.block2.project.bias']
        has_res = (p + '.res_conv.weight') in sd
        if has_res:
            Wr = sd[p + '.res_conv.weight'][:, :, 0, 0].clone()
            if len(srcs) == 2:
                Wr[:, srcs[0].C:] *= skip            # cat((x, skip * 2^-0.5)) (:1694) folded into the 1x1 weights
            br = sd[p + '.res_conv.bias']
        else:
            assert len(srcs) == 1 and din == dout
        out = self._new(M, dout, Hc, Wc)
        if gca:
            h3 = self._new(M, dout, Hc, Wc)
            self._conv([a2], W2, dout, h3.t, ldc=h3.ld, bias=b2)
            gate = self._gca(p + '.gca', h3)
            if has_res:
                r = self._new(M, dout, Hc, Wc)
                o, mats, segs = 0, [], []
                for i, s in enumerate(srcs):
                    segs.append((i, 0, 0))
                    mats.append(Wr[:, o:o + s.C])
                    o += s.C
                self._gemm(srcs, segs, (R, Hc, Wc), self._pack(mats, dout), dout, r.t, ldc=r.ld, bias=br)
            else:
                r = srcs[0]
            if self.fuse_norm:
                rc = ops.RowChainCall(h3.ptr, h3.ld, M, dout, gate=gate, rows_per_sample=n, residual_ptr=r.ptr, ldr=r.ld, out_ptr=out.ptr, ldo=out.ld)
                self._keep.append(rc)
                self._ops.append((rc.lib.b200_row_chain, rc.args, 'b200_row_chain'))
                out.call = rc
            else:
                self._add('b200_gate_residual', h3.ptr, h3.ld, gate.data_ptr(), r.ptr, r.ld, out.ptr, out.ld, M, dout, n)
        elif has_res:
            # conv3x3(a2) + res_conv(x) accumulated in ONE implicit GEMM: 9 tap segments on a2 + 1x1 segments on the raw inputs
            segs = [(0, dh, dw) for (dh, dw) in self._conv_taps(3)]
            mats = [W2[:, :, dh + 1, dw + 1] for (dh, dw) in self._conv_taps(3)]
            o = 0
            for i, s in enumerate(srcs):
                segs.append((i + 1, 0, 0))
                mats.append(Wr[:, o:o + s.C])
                o += s.C
            out.call = self._gemm([a2, *srcs], segs, (R, Hc, Wc), self._pack(mats, dout), dout, out.t, ldc=out.ld, bias=b2 + br)
        else:
            out.call = self._conv([a2], W2, dout, out.t, ldc=out.ld, bias=b2, residual=srcs[0])
        return out

    def _gca(self, p, h: Rows):
        """GlobalContext (imagen_pytorch.py:945-970) -> gate [R, C] fp32."""
        sd, R = self.sdc, self.R
        n, Cc = h.H * h.W, h.C
        hid = sd[p + '.net.0.weight'].shape[0]
        nchunk = self.lib.b200_gca_chunks(n, Cc)
        scratch = self._zeros((R * nchunk * (Cc + 2) + R * Cc + R * hid + R * n,), torch.float32)
        gate = self._zeros((R, Cc), torch.float32)
        wk = self._f32(sd[p + '.to_k.weight'].flatten())
        w1 = self._f32(sd[p + '.net.0.weight'].reshape(hid, Cc))
        b1 = self._f32(sd[p + '.net.0.bias'])
        w2 = self._f32(sd[p + '.net.2.weight'].reshape(Cc, hid))
        b2 = self._f32(sd[p + '.net.2.bias'])
        self._add('b200_gca_gate', h.ptr, h.ld, R, n, Cc, wk.data_ptr(), float(sd[p + '.to_k.bias'].item()), w1.data_ptr(), b1.data_ptr(),
                  hid, w2.data_ptr(), b2.data_ptr(), scratch.data_ptr(), nchunk, gate.data_ptr())
        return gate

    def _logit_bound(self, p):
        """|q.k| <= 8 * max_d |q_scale_d * k_scale_d| for unit q, k (Cauchy-Schwarz), in log2 units, +2% for bf16 rounding.
        The attention ABI takes the tcgen05 fixed-bound path when this is <= 40, else the online-softmax kernel."""
        if os.environ.get('B200_IMAGEN_ATTN', 'tc') == 'mma':
            return 0.0
        return float((self.sdc[p + '.q_scale'].abs() * self.sdc[p + '.k_scale'].abs()).max().item()) * 8.0 * LOG2E * 1.02

    def _cross_attention(self, p, h: Rows, heads, g2, film_off):
        """CrossAttention.forward + residual (imagen_pytorch.py:793-834, :749), followed by block2's ChanRMSNorm -> FiLM -> SiLU
        (:683-691): returns a2, the input of block2's conv.  When a GEMM tile spans all channels the pre-norm LayerNorm runs in the
        epilogue of the conv that produced h, and to_out's epilogue does LayerNorm -> + h -> RMSNorm/FiLM/SiLU: 2 launches
        (to_q, attention) + to_out instead of 5 + the block norm."""
        sd, R = self.sdc, self.R
        n, M = h.H * h.W, h.rows
        inner = heads * 64
        hn = self._prenorm_ln(h, sd[p + '.norm.g'])
        qs =self._f32(sd[p + '.q_scale'] * (8.0 * LOG2E))
        q = self._linear(hn, sd[p + '.to_q.weight'], inner, l2_cols=inner, l2_scale=qs)
        Kc, Vc, nk = self._context_kv(p, heads, linear=False)
        o = self._new(M, inner, h.H, h.W)
        self._add('b200_attention', q.ptr, o.ptr, n * inner, 64, inner, n, Kc.data_ptr(), Vc.data_ptr(), nk * inner, 64, inner, nk, R, heads,
                  self._logit_bound(p))
        return self._attn_out(p, o, h, g2, film_off)

    def _context_kv(self, p, heads, *, linear):
        """Per-layer context K/V buffers [R, n_ctx + 1, heads*64]: prepare() writes the static rows, b200_update_time_rows the
        time-token rows of each sample's schedule slot every step; the null key/value is the last row, the same for every head
        (:805-808).  CrossAttention stores K l2-normalised * k_scale; LinearCrossAttention (linear=True) uses K raw (:851-866)."""
        sd, R = self.sdc, self.R
        inner, nk = heads * 64, self.n_ctx + 1
        Kc, Vc = self._zeros((R, nk, inner)), self._zeros((R, nk, inner))
        Kt, Vt = self._zeros((self.S, self.ntt, inner)), self._zeros((self.S, self.ntt, inner))
        self.cross_layers.append(dict(p=p, K=Kc, V=Vc, Kt=Kt, Vt=Vt, heads=heads, nk=nk, linear=linear))
        for tb, dst in ((Kt, Kc), (Vt, Vc)):
            self._jobs.append(TimeRowJob(tb.data_ptr(), dst.data_ptr(), nk * inner, self.ntt, inner))
        nkv = sd[p + '.null_kv']
        self._row_fill(Kc[:, nk - 1, :], (nkv[0] if linear else F.normalize(nkv[0], dim=-1) * sd[p + '.k_scale']).repeat(heads))
        self._row_fill(Vc[:, nk - 1, :], nkv[1].repeat(heads))
        return Kc, Vc, nk

    def _linear_cross_attention(self, p, h: Rows, heads, g2, film_off):
        """LinearCrossAttention.forward + residual (imagen_pytorch.py:836-874, :749), followed by block2's norm like _cross_attention:
        to_q (plain: the softmax over the head width replaces l2norm / q_scale), the per-step context matrix C = 8 softmax_j(k)^T v of
        every (row, head), O = softmax_d(q) C, and the same to_out epilogue."""
        sd, R, a = self.sdc, self.R, self.arch
        n, M = h.H * h.W, h.rows
        inner = heads * 64
        hn = self._prenorm_ln(h, sd[p + '.norm.g'])
        q = self._linear(hn, sd[p + '.to_q.weight'], inner)
        Kc, Vc, nk = self._context_kv(p, heads, linear=True)
        ctx = self._zeros((R, heads, 64, 64))
        self._add('b200_linear_xattn_context', Kc.data_ptr(), Vc.data_ptr(), nk * inner, inner, nk, R, heads, a.dim_head, ctx.data_ptr())
        o = self._new(M, inner, h.H, h.W)
        self._add('b200_linear_cross_attention', q.ptr, o.ptr, n * inner, inner, n, ctx.data_ptr(), R, heads, a.dim_head)
        return self._attn_out(p, o, h, g2, film_off)

    def _attn_out(self, p, o: Rows, h: Rows, g2, film_off):
        """to_out Linear -> LayerNorm -> + h -> block2's ChanRMSNorm / FiLM / SiLU of a cross-attention layer: returns a2."""
        sd = self.sdc
        n, M, Cc = h.H * h.W, h.rows, h.C
        if self._fusable(Cc):
            a2 = self._new(M, Cc, h.H, h.W)
            self._linear(o, sd[p + '.to_out.0.weight'], Cc, out=a2, out_raw=False, norm1=_lib.NORM_LN, norm1_g=self._f32(sd[p + '.to_out.1.g'].flatten()),
                         residual=h, norm2=_lib.NORM_RMS_FILM_SILU, norm2_g=self._f32(g2.flatten() * math.sqrt(Cc)),
                         film_ptr=self.film.data_ptr() + 4 * film_off, film_ld=self.film.shape[1], rows_per_sample=n, out_norm_ptr=a2.ptr, ld_norm=a2.ld)
            self.n_fused += 2
            return a2
        y = self._linear(o, sd[p + '.to_out.0.weight'], Cc)
        h2 = self._layernorm(y, sd[p + '.to_out.1.g'], residual=h)
        return self._rms_film_silu([h2], g2, Cc, 1.0, n, film_off)

    def _transformer(self, p, x: Rows, depth, has_ctx):
        """TransformerBlock.forward (imagen_pytorch.py:1012-1022): multi-query self-attention + feed-forward."""
        a, sd, R = self.arch, self.sdc, self.R
        n, M, Cc = x.H * x.W, x.rows, x.C
        heads, inner = a.heads, self.inner
        for l in range(depth):
            q_, ff = f'{p}.layers.{l}.0', f'{p}.layers.{l}.1'
            xn = self._prenorm_ln(x, sd[q_ + '.norm.g'])
            qs = self._f32(sd[q_ + '.q_scale'] * (8.0 * LOG2E))
            q = self._linear(xn, sd[q_ + '.to_q.weight'], inner, l2_cols=inner, l2_scale=qs)
            npre = (self.n_ctx if has_ctx else 0) + 1
            Mtot = npre + n
            Kb, Vb = self._zeros((R, Mtot, 64)), self._zeros((R, Mtot, 64))
            ks = self._f32(sd[q_ + '.k_scale'])
            # to_kv epilogue: k l2-normalised * k_scale, scattered straight behind the [context | null] prefix rows
            self._gemm([xn], [(0, 0, 0)], (1, 1, M), self._pack([sd[q_ + '.to_kv.weight']], 128), 128, Kb, ldc=64, out2=Vb, ldc2=64,
                       split_col=64, rows_per_group=n, group_stride=Mtot, row_offset=npre, l2_cols=64, l2_scale=ks)
            nkv = sd[q_ + '.null_kv']
            self._row_fill(Kb[:, npre - 1, :], F.normalize(nkv[0], dim=-1) * sd[q_ + '.k_scale'])
            self._row_fill(Vb[:, npre - 1, :], nkv[1])
            layer = dict(p=q_, K=Kb, V=Vb, has_ctx=has_ctx, Mtot=Mtot)
            if has_ctx:
                Kt, Vt = self._zeros((self.S, self.ntt, 64)), self._zeros((self.S, self.ntt, 64))
                layer.update(Kt=Kt, Vt=Vt)
                for tb, dst in ((Kt, Kb), (Vt, Vb)):
                    self._jobs.append(TimeRowJob(tb.data_ptr(), dst.data_ptr(), Mtot * 64, self.ntt, 64))
            self.self_layers.append(layer)
            o = self._new(M, inner, x.H, x.W)
            # all heads of a sample share K/V: heads*n query rows of width 64 form ONE attention problem
            self._add('b200_attention', q.ptr, o.ptr, n * inner, 0, 64, heads * n, Kb.data_ptr(), Vb.data_ptr(), Mtot * 64, 0, 64, Mtot, R, 1,
                      self._logit_bound(q_))
            hid = sd[ff + '.1.weight'].shape[0]
            if self._fusable(Cc):
                # to_out epilogue: LayerNorm -> + x (= x1) -> LayerNorm of the feed-forward (:1018-1020, :975): two outputs, no row kernels
                x1, f = self._new(M, Cc, x.H, x.W), self._new(M, Cc, x.H, x.W)
                self._linear(o, sd[q_ + '.to_out.0.weight'], Cc, out=x1, norm1=_lib.NORM_LN, norm1_g=self._f32(sd[q_ + '.to_out.1.g'].flatten()),
                             residual=x, norm2=_lib.NORM_LN, norm2_g=self._f32(sd[ff + '.0.g'].flatten()), out_norm_ptr=f.ptr, ld_norm=f.ld)
                self.n_fused += 2
            else:
                y = self._linear(o, sd[q_ + '.to_out.0.weight'], Cc)
                x1 = self._layernorm(y, sd[q_ + '.to_out.1.g'], residual=x)
                f = self._layernorm(x1, sd[ff + '.0.g'])
            if self._fusable(hid):
                # FF1 epilogue: GELU -> LayerNorm over the hidden width (:976-978); only the normalised tensor is stored
                hn = self._new(M, hid, x.H, x.W)
                self._linear(f, sd[ff + '.1.weight'], hid, out=hn, out_raw=False, act=_lib.ACT_GELU, norm2=_lib.NORM_LN,
                             norm2_g=self._f32(sd[ff + '.3.g'].flatten()), out_norm_ptr=hn.ptr, ld_norm=hn.ld)
                self.n_fused += 1
            else:
                hdn = self._linear(f, sd[ff + '.1.weight'], hid, act=_lib.ACT_GELU)
                hn = self._layernorm(hdn, sd[ff + '.3.g'])
            x = self._linear(hn, sd[ff + '.4.weight'], Cc, residual=x1)     # x.call: the next layer's pre-norm attaches here
        return x

    def _downsample(self, p, x: Rows, dout):
        """Downsample = pixel-unshuffle + 1x1 conv (imagen_pytorch.py:633-640)."""
        sd, R = self.sdc, self.R
        H2, W2 = x.H // 2, x.W // 2
        xs = self._new(R * H2 * W2, 4 * x.C, H2, W2)
        self._add('b200_pixel_unshuffle', x.ptr, x.ld, R, x.H, x.W, x.C, xs.ptr)
        Wd = sd[p + '.weight'][:, :, 0, 0]                                     # [dout, c*4 + s]
        Wd = Wd.view(dout, x.C, 4).permute(0, 2, 1).reshape(dout, 4 * x.C)     # -> [dout, s*C + c]
        return self._linear(xs, Wd, dout, bias=sd[p + '.bias'])

    def _upsample(self, p, x: Rows, dout):
        """PixelShuffleUpsample: 1x1 conv -> SiLU -> PixelShuffle(2) fused in one GEMM epilogue (:603-631)."""
        sd, R = self.sdc, self.R
        Wu = sd[p + '.net.0.weight'][:, :, 0, 0]                               # [c'*4 + r, C]
        Wu = Wu.view(dout, 4, x.C).permute(1, 0, 2).reshape(4 * dout, x.C)     # -> [r*C' + c', C]
        bu = sd[p + '.net.0.bias'].view(dout, 4).permute(1, 0).reshape(-1)
        out = self._new(R * 4 * x.H * x.W, dout, 2 * x.H, 2 * x.W)
        wp = self._pack([Wu], 4 * dout)
        self._gemm([x], [(0, 0, 0)], (R, x.H, x.W), wp, 4 * dout, out.t, ldc=out.ld, bias=bu, act=_lib.ACT_SILU,
                   out_mode=_lib.OUT_PIXEL_SHUFFLE, ps_C=dout)
        return out

    # ------------------------------------------------------------------ plan
    def _build(self):
        a, sd, R, B, H, W = self.arch, self.sdc, self.R, self.B, self.H, self.W
        # FiLM table: every ResnetBlock's time_mlp Linear batched into one GEMM per step (:711-714, :739-741)
        names = [k[:-len('.time_mlp.1.weight')] for k in param_table(a) if k.endswith('.time_mlp.1.weight')]
        self.film_offsets, off = {}, 0
        for nme in names:
            self.film_offsets[nme] = off
            off += sd[nme + '.time_mlp.1.weight'].shape[0]
        self.film = self._zeros((R, off), torch.float32)
        film_W = torch.cat([sd[nme + '.time_mlp.1.weight'] for nme in names], 0)
        film_b = torch.cat([sd[nme + '.time_mlp.1.bias'] for nme in names], 0)

        # ---- stem: cross-embed init conv as ONE GEMM over gathered patches (:1051-1076, :1564)
        ks, Cin = max(a.init_kernels), a.init_channels
        Kinit = _ceil(ks * ks * Cin, 64)
        M0 = B * H * W
        patches = self._new(M0, Kinit)
        stem = []
        self._ops = stem
        # cat order: (cond_images, x, self_cond, lowres_cond_img) (:1543, :1551, :1560)
        imgs = ([self.cond_img] if a.cond_images_channels else []) + [self.x_in] + ([self.sc_in] if a.self_cond else []) + \
               ([self.lowres_img] if a.lowres_cond else [])
        imgs += [None] * (4 - len(imgs))
        self._add('b200_im2col_init4', *[v for im in imgs for v in ((im.data_ptr(), im.shape[1]) if im is not None else (None, 0))],
                  B, H, W, ks, patches.ptr, Kinit)
        Wi = torch.zeros(a.init_dim, ks, ks, Cin)
        bi = torch.zeros(a.init_dim)
        row = 0
        for i, (k, ds) in enumerate(zip(a.init_kernels, a.init_dim_scales)):
            pre = f'init_conv.convs.{i}' if a.init_cross_embed else 'init_conv'
            o = (ks - k) // 2
            Wi[row:row + ds, o:o + k, o:o + k, :] = sd[pre + '.weight'].permute(0, 2, 3, 1)
            bi[row:row + ds] = sd[pre + '.bias']
            row += ds
        x = self._new(R * H * W, a.init_dim, H, W)
        self._gemm([patches], [(0, 0, 0)], (1, 1, M0), self._pack([Wi.reshape(a.init_dim, -1)], a.init_dim), a.init_dim, x.t, ldc=x.ld,
                   bias=bi, dup_rows=M0 if R == 2 * B else 0)
        # ---- per-step time conditioning
        self.t_silu = self._new(R, a.time_cond_dim)
        self._add('b200_make_time_cond', self.time_cond_table.data_ptr(), self.text_hiddens.data_ptr(), self.slots.data_ptr(), R,
                  a.time_cond_dim, self.t_silu.ptr)
        self._gemm([self.t_silu], [(0, 0, 0)], (1, 1, R), self._pack([film_W], film_W.shape[0]), film_W.shape[0], self.film,
                   ldc=self.film.shape[1], bias=film_b, out_mode=_lib.OUT_F32)

        body = []
        self._ops = body
        if a.memory_efficient:
            x = self._resnet('init_resnet_block', [x], a.init_dim, gca=a.use_gca)
        hiddens = []
        for i in range(a.num_levels):                                          # Unet.forward :1671-1685
            L = a.down_level(i)
            p = f'downs.{i}'
            if a.memory_efficient:
                x = self._downsample(p + '.0.1', x, L['dim_out'])
            x = self._resnet(p + '.1', [x], L['cur'], cross_heads=a.heads if L['cross'] else None, linear_cross=L['linear_cross'])
            for j in range(L['nres']):
                x = self._resnet(f'{p}.2.{j}', [x], L['cur'], gca=a.use_gca)
                hiddens.append(x)
            if L['attn']:
                x = self._transformer(p + '.3', x, L['depth'], True)
            hiddens.append(x)
            if not a.memory_efficient:
                if not L['is_last']:
                    x = self._downsample(p + '.4.1', x, L['dim_out'])
                else:                                                          # Parallel(conv3x3, conv1x1) summed (:1366): 1x1 folded into the centre tap
                    W3 = sd[p + '.4.fns.0.weight'].clone()
                    W3[:, :, 1, 1] += sd[p + '.4.fns.1.weight'][:, :, 0, 0]
                    y = self._new(x.rows, L['dim_out'], x.H, x.W)
                    self._conv([x], W3, L['dim_out'], y.t, ldc=y.ld, bias=sd[p + '.4.fns.0.bias'] + sd[p + '.4.fns.1.bias'])
                    x = y
        mid = a.dims[-1]
        x = self._resnet('mid_block1', [x], mid, cross_heads=8)
        if a.attend_at_middle:
            x = self._transformer('mid_attn', x, a.mid_depth, False)
        x = self._resnet('mid_block2', [x], mid, cross_heads=8)
        for i in range(a.num_levels):                                          # :1698-1708
            U = a.up_level(i)
            p = f'ups.{i}'
            x = self._resnet(p + '.0', [x, hiddens.pop()], U['dim_out'], cross_heads=a.heads if U['cross'] else None,
                             linear_cross=U['linear_cross'])
            for j in range(U['nres']):
                x = self._resnet(f'{p}.1.{j}', [x, hiddens.pop()], U['dim_out'], gca=a.use_gca)
            if U['attn']:
                x = self._transformer(p + '.2', x, U['depth'], True)
            if (not U['is_last']) or a.memory_efficient:
                x = self._upsample(p + '.3', x, U['dim_in'])
        assert not hiddens
        x = self._resnet('final_res_block', [x], a.dim, gca=True)
        Wf, bf = sd['final_conv.weight'], sd['final_conv.bias']
        if a.lowres_cond:                                                      # cat((x, lowres_cond_img)) before final_conv (:1722-1723)
            self.lowres_rows = self._new(R * H * W, 8, H, W)
            Wpad = torch.zeros(Wf.shape[0], a.dim + 8, *Wf.shape[2:])
            Wpad[:, :a.dim + a.channels] = Wf
            self._conv([x, self.lowres_rows], Wpad, a.channels_out, self.pred, split=[a.dim, 8], bias=bf, out_mode=_lib.OUT_F32_NCHW)
        else:
            self._conv([x], Wf, a.channels_out, self.pred, bias=bf, out_mode=_lib.OUT_F32_NCHW)

        # ---- assemble: stem, time rows of every context K/V buffer, body
        ops = list(stem)
        if self._jobs:
            jobs = (TimeRowJob * len(self._jobs))(*self._jobs)
            jb = self._wts.put(torch.frombuffer(bytearray(bytes(jobs)), dtype=torch.uint8))
            max_elems = max(j.rows * j.width for j in self._jobs)
            ops.append((self.lib.b200_update_time_rows, (jb.data_ptr(), len(self._jobs), self.slots.data_ptr(), R, max_elems), 'b200_update_time_rows'))
        self._ops = ops + body
        # staged host chunks -> device (one memcpy per chunk), then the few constant rows that live inside activation buffers
        self._wts.flush()
        for dst, src in self._post:
            dst.copy_(src.expand_as(dst))
        self._post = None
        del self.sdc
        # our kernel launches per U-Net evaluation (b200_gca_gate = fused logits/pooling kernel + cluster MLP kernel)
        self.n_launches = len(self._ops) + sum(1 for o in self._ops if o[2] == 'b200_gca_gate') * 1 + \
            sum(1 for c in self._keep if getattr(c, 'desc', {}).get('ksplit', 1) > 1)      # + split-K finishing kernels (GemmCall.desc)

    # ------------------------------------------------------------------ execution
    def describe_gemms(self):
        """[{B,H,W,N,K,...}] of every b200_conv_gemm launch of one evaluation, in launch order (profiling aid)."""
        return [c.desc for c in self._keep if isinstance(c, ops.GemmCall)]

    def launch_timed(self):
        """Profiling aid: one evaluation with a CUDA-event pair around every C-ABI call -> [(name, microseconds)].
        The host runs ahead of the GPU (one call = one to five kernels), so each delta is that call's execution time with the
        caches in the state the previous call left them -- what the captured graph sees, unlike ncu's flushed-cache numbers."""
        st = torch.cuda.current_stream(self.device)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self._ops) + 1)]
        evs[0].record(st)
        for i, (fn, args, name) in enumerate(self._ops):
            rc = fn(*args, st.cuda_stream)
            if rc != 0:
                raise _lib.B200Error(f'{name} failed ({rc}): {self.lib.b200_last_error().decode()}')
            evs[i + 1].record(st)
        torch.cuda.synchronize(self.device)
        return [(self._ops[i][2], evs[i].elapsed_time(evs[i + 1]) * 1e3) for i in range(len(self._ops))]

    def launch(self, stream=None):
        """Enqueue one U-Net evaluation (x_in -> pred) on the current stream. CUDA-graph capturable."""
        st = stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream
        err = self.lib.b200_last_error
        for fn, args, name in self._ops:
            rc = fn(*args, st)
            if rc != 0:
                raise _lib.B200Error(f'{name} failed ({rc}): {err().decode()}')

    # ------------------------------------------------------------------ conditioning head (once per sample() call)
    def _call(self, name, *args):
        rc = getattr(self.lib, name)(*args, torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise _lib.B200Error(f'{name} failed ({rc}): {self.lib.b200_last_error().decode()}')

    def _lin(self, x, W, b=None, in_act=0, out_act=0, res=None):
        x2 = x.reshape(-1, x.shape[-1])
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        N, K = W.shape
        y = torch.empty(x2.shape[0], N, dtype=torch.float32, device=self.device)
        r2 = res.reshape(-1, N).contiguous() if res is not None else None
        self._call('b200_linear_f32', x2.data_ptr(), K, W.data_ptr(), b.data_ptr() if b is not None else None, in_act, out_act,
                   r2.data_ptr() if r2 is not None else None, N, y.data_ptr(), N, x2.shape[0], N, K)
        return y.view(*x.shape[:-1], N)

    def _ln(self, x, g, beta=None, eps=1e-5):
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        y = torch.empty_like(x2)
        Cc = x2.shape[1]
        self._call('b200_layernorm_f32', x2.data_ptr(), Cc, g.data_ptr() if g is not None else None,
                   beta.data_ptr() if beta is not None else None, eps, y.data_ptr(), Cc, x2.shape[0], Cc)
        return y.view(x.shape)

    def _store_heads(self, x, col0, ngroups, normalize, scale, dst, dst_off_elems, rpg, s_grp, s_row, s_head):
        x2 = x.reshape(-1, x.shape[-1])
        assert x2.is_contiguous()
        self._call('b200_headnorm_store', x2.data_ptr(), x2.shape[1], col0, ngroups, int(normalize),
                   scale.data_ptr() if scale is not None else None, dst.data_ptr() + 2 * dst_off_elems, rpg, s_grp, s_row, s_head, x2.shape[0])

    def _perceiver(self, tokens):
        """PerceiverResampler.forward (imagen_pytorch.py:481-498) in fp32."""
        a, sd = self.arch, self.sd
        T, L, cd = tokens.shape
        p = 'attn_pool'
        x_pos = tokens + sd[p + '.pos_emb.weight'][:L]
        latents = sd[p + '.latents'].unsqueeze(0).expand(T, -1, -1)
        pooled = tokens.sum(dim=1) / float(L)                                   # masked_mean with an all-ones mask (:490)
        ml = self._lin(self._ln(pooled, sd[p + '.to_latents_from_mean_pooled_seq.0.g']),
                       sd[p + '.to_latents_from_mean_pooled_seq.1.weight'], sd[p + '.to_latents_from_mean_pooled_seq.1.bias'])
        latents = torch.cat((ml.view(T, a.pool_mean_latents, cd), latents), dim=1).contiguous()
        nl, inner, H = latents.shape[1], self.inner, a.heads
        for l in range(a.pool_depth):
            q_, ff = f'{p}.layers.{l}.0', f'{p}.layers.{l}.1'
            xn = self._ln(x_pos, sd[q_ + '.norm.weight'], sd[q_ + '.norm.bias'])
            ln_lat = self._ln(latents, sd[q_ + '.norm_latents.weight'], sd[q_ + '.norm_latents.bias'])
            q = self._lin(ln_lat, sd[q_ + '.to_q.weight'])
            kv = self._lin(torch.cat((xn, ln_lat), dim=1), sd[q_ + '.to_kv.weight'])         # [T, L+nl, 2*inner]
            o = torch.empty(T, nl, inner, dtype=torch.float32, device=self.device)
            self._call('b200_attn_f32', q.data_ptr(), inner, kv.data_ptr(), kv.data_ptr() + 4 * inner, 2 * inner,
                       sd[q_ + '.q_scale'].data_ptr(), sd[q_ + '.k_scale'].data_ptr(), o.data_ptr(), inner, T, H, nl, L + nl)
            out = self._ln(self._lin(o, sd[q_ + '.to_out.0.weight']), sd[q_ + '.to_out.1.weight'], sd[q_ + '.to_out.1.bias'])
            latents = out + latents
            h = self._lin(self._ln(latents, sd[ff + '.0.g']), sd[ff + '.1.weight'], out_act=_lib.ACT_GELU)
            latents = self._lin(self._ln(h, sd[ff + '.3.g']), sd[ff + '.4.weight'], res=latents)
        return latents

    @torch.no_grad()
    def prepare(self, times, *, text_embeds=None, text_mask=None, keep=None, lowres_cond_img=None, lowres_noise_times=None,
                slot_of_row=None, cond_images=None):
        """Everything of Unet.forward that does not depend on x (imagen_pytorch.py:1573-1660), for all schedule slots.

        times: fp32 [S'] U-Net time input per schedule slot (S' <= n_slots).
        keep : bool [R]; False rows get the null text conditioning (cond_drop_prob == 1 branch, :1599-1650).
        Row r is conditioned on text_embeds[r % B] / lowres_cond_img[r % B]."""
        a, sd, R, B, dev = self.arch, self.sd, self.R, self.B, self.device
        times = times.to(device=dev, dtype=torch.float32).flatten().contiguous()
        S = times.numel()
        assert S <= self.S, f'{S} schedule slots > plan capacity {self.S}'
        cd, tcd, ntt = a.cond_dim, a.time_cond_dim, self.ntt
        keep = torch.ones(R, dtype=torch.bool, device=dev) if keep is None else keep.to(dev)
        img_of_row = torch.arange(R, device=dev) % B
        assert not ((a.cond_images_channels > 0) ^ (cond_images is not None)), \
            'you either requested to condition on an image on the unet, but the conditioning image is not supplied, or vice versa'
        if cond_images is not None:                                             # :1557-1560 (the concat itself happens in the stem gather)
            assert cond_images.shape[1] == a.cond_images_channels, \
                'the number of channels on the conditioning image you are passing in does not match what you specified on initialiation of the unet'
            ci = cond_images.to(device=dev, dtype=torch.float32)
            if ci.shape[-1] != self.W:
                ci = F.interpolate(ci, self.W, mode=a.cfg['resize_mode'])
            self.cond_img.copy_(ci)

        def time_path(prefix, tvals):                                          # :1573-1578 / :1584-1586
            n = tvals.numel()
            half = a.sinu_dim // 2
            emb = torch.empty(n, 2 * half + 1, dtype=torch.float32, device=dev)
            self._call('b200_sinu_pos_emb', tvals.data_ptr(), sd[f'{prefix}_hiddens.0.weights'].data_ptr(), n, half, emb.data_ptr())
            hid = self._lin(emb, sd[f'{prefix}_hiddens.1.weight'], sd[f'{prefix}_hiddens.1.bias'], out_act=_lib.ACT_SILU)
            tok = self._lin(hid, sd[f'{prefix}_tokens.0.weight'], sd[f'{prefix}_tokens.0.bias']).view(n, ntt, cd)
            tcond = self._lin(hid, sd[f'{prefix}_cond.0.weight'], sd[f'{prefix}_cond.0.bias'])
            return tok, tcond

        tok, tcond = time_path('to_time', times)
        self.time_cond_table[:S].copy_(tcond)
        c_time = self._ln(tok, sd['norm_cond.weight'], sd['norm_cond.bias'])    # norm_cond is per token (:1660)
        hidden_rows = torch.zeros(R, tcd, dtype=torch.float32, device=dev)
        static = []
        if a.lowres_cond:
            assert lowres_cond_img is not None and lowres_noise_times is not None, 'low resolution conditioning image / noise time must be present'
            lt = lowres_noise_times.to(device=dev, dtype=torch.float32).flatten()
            if lt.numel() == 1:
                lt = lt.expand(B)
            ltok, lcond = time_path('to_lowres_time', lt.contiguous())
            hidden_rows += lcond[img_of_row]                                    # t = t + lowres_t (:1588)
            static.append(self._ln(ltok, sd['norm_cond.weight'], sd['norm_cond.bias'])[img_of_row])
            self.lowres_img.copy_(lowres_cond_img.to(device=dev, dtype=torch.float32))
            low8 = torch.empty(B * self.H * self.W, 8, dtype=BF16, device=dev)
            self._call('b200_nchw_to_rows', self.lowres_img.data_ptr(), B, a.channels, self.H, self.W, low8.data_ptr(), 8)
            self.lowres_rows.t.view(R // B, -1, 8).copy_(low8.view(1, -1, 8).expand(R // B, -1, -1))
        if a.cond_on_text and text_embeds is not None:
            te = text_embeds.to(device=dev, dtype=torch.float32)
            Bt, L = te.shape[0], a.max_text_len
            assert Bt == B, f'text_embeds batch {Bt} != image batch {B}'
            tokens = self._lin(te, sd['text_to_cond.weight'], sd['text_to_cond.bias'])[:, :L]   # :1606-1608
            mask = text_mask.to(dev)[:, :L] if text_mask is not None else None
            rem = L - tokens.shape[1]
            if rem > 0:
                tokens = F.pad(tokens, (0, 0, 0, rem))
                if mask is not None:
                    mask = F.pad(mask, (0, rem), value=False)
            null_embed = sd['null_text_embed']
            if mask is not None:
                tokens = torch.where(mask[:, :, None], tokens, null_embed)      # :1619-1632 (keep-mask part: whole rows, below)
            all_tokens = torch.cat((tokens, null_embed), dim=0).contiguous()    # last entry = null conditioning
            lat = self._perceiver(all_tokens) if a.attn_pool else all_tokens
            mean = lat.mean(dim=-2)                                             # :1640
            th = self._ln(mean, sd['to_text_non_attn_cond.0.weight'], sd['to_text_non_attn_cond.0.bias'])
            th = self._lin(self._lin(th, sd['to_text_non_attn_cond.1.weight'], sd['to_text_non_attn_cond.1.bias'], out_act=_lib.ACT_SILU),
                           sd['to_text_non_attn_cond.3.weight'], sd['to_text_non_attn_cond.3.bias'])
            th = th.clone()
            th[Bt] = sd['null_text_hidden'][0]                                  # where(keep, text_hiddens, null_text_hidden) (:1646-1650)
            ctx_of_row = torch.where(keep, img_of_row, torch.full_like(img_of_row, Bt))
            hidden_rows += th[ctx_of_row]
            static.append(self._ln(lat, sd['norm_cond.weight'], sd['norm_cond.bias'])[ctx_of_row])
        elif a.cond_on_text:
            raise ValueError('text_embeds must be passed to a text-conditioned U-Net')
        self.text_hiddens.copy_(hidden_rows)
        ctx_static = torch.cat(static, dim=1).contiguous() if static else None  # [R, n_static, cd]
        ns = self.n_static
        assert (ctx_static.shape[1] if ctx_static is not None else 0) == ns

        for Lr in self.cross_layers:                                            # CrossAttention to_kv of the context (:799-814)
            p, heads, nk = Lr['p'], Lr['heads'], Lr['nk']
            inner = heads * 64
            Wkv = sd[p + '.to_kv.weight']
            knorm, ksc = (False, None) if Lr['linear'] else (True, sd[p + '.k_scale'])   # LinearCrossAttention: raw k (softmax over tokens)
            kvt = self._lin(c_time, Wkv)                                        # [S, ntt, 2*inner]
            self._store_heads(kvt, 0, heads, knorm, ksc, Lr['Kt'], 0, ntt, ntt * inner, inner, 64)
            self._store_heads(kvt, inner, heads, False, None, Lr['Vt'], 0, ntt, ntt * inner, inner, 64)
            if ns:
                kvs = self._lin(ctx_static, Wkv)                                # [R, ns, 2*inner]
                self._store_heads(kvs, 0, heads, knorm, ksc, Lr['K'], ntt * inner, ns, nk * inner, inner, 64)
                self._store_heads(kvs, inner, heads, False, None, Lr['V'], ntt * inner, ns, nk * inner, inner, 64)
        for Ls in self.self_layers:                                             # Attention.to_context (:551-555, :559-561)
            if not Ls['has_ctx']:
                continue
            p, Mtot = Ls['p'], Ls['Mtot']
            lw, lb = sd[p + '.to_context.0.weight'], sd[p + '.to_context.0.bias']
            Wc, bc, ksc = sd[p + '.to_context.1.weight'], sd[p + '.to_context.1.bias'], sd[p + '.k_scale']
            kvt = self._lin(self._ln(c_time, lw, lb), Wc, bc)                   # [S, ntt, 128]
            self._store_heads(kvt, 0, 1, True, ksc, Ls['Kt'], 0, ntt, ntt * 64, 64, 0)
            self._store_heads(kvt, 64, 1, False, None, Ls['Vt'], 0, ntt, ntt * 64, 64, 0)
            if ns:
                kvs = self._lin(self._ln(ctx_static, lw, lb), Wc, bc)
                self._store_heads(kvs, 0, 1, True, ksc, Ls['K'], ntt * 64, ns, Mtot * 64, 64, 0)
                self._store_heads(kvs, 64, 1, False, None, Ls['V'], ntt * 64, ns, Mtot * 64, 64, 0)
        if slot_of_row is None:
            self.slots.zero_()
        else:
            self.slots.copy_(slot_of_row.to(device=dev, dtype=torch.int32))


class Unet(nn.Module):
    """Drop-in for imagen_pytorch.Unet (imagen_pytorch.py:1112-1725) on B200.

    Same keyword constructor, ``forward`` / ``forward_with_cond_scale`` signatures, attributes read by
    ``Imagen`` (``lowres_cond``, ``cond_on_text``, ``channels``, ``channels_out``, ``_locals``,
    ``cast_model_parameters``) and ``state_dict`` layout.  Inference only (``torch.no_grad``)."""

    def __init__(self, **kwargs):
        super().__init__()
        self.arch = UnetArch(**kwargs)
        self._locals = dict(self.arch.cfg)                                     # :1173-1175
        a = self.arch
        self.channels, self.channels_out = a.channels, a.channels_out
        self.lowres_cond, self.cond_on_text = a.lowres_cond, a.cond_on_text
        self.self_cond = a.self_cond
        self.has_cond_image = a.cond_images_channels > 0
        self.cond_images_channels = a.cond_images_channels
        self.max_text_len = a.max_text_len
        build_param_tree(self, param_table(a))
        self._plans = {}
        self._gemm_impl = _lib.IMPL_TCGEN05

    # --- reference API ------------------------------------------------------------------------
    def cast_model_parameters(self, *, lowres_cond, text_embed_dim, channels, channels_out, cond_on_text):   # :1446-1470
        if lowres_cond == self.lowres_cond and channels == self.channels and cond_on_text == self.cond_on_text and \
                text_embed_dim == self._locals['text_embed_dim'] and channels_out == self.channels_out:
            return self
        updated = dict(lowres_cond=lowres_cond, text_embed_dim=text_embed_dim, channels=channels, channels_out=channels_out,
                       cond_on_text=cond_on_text)
        return self.__class__(**{**self._locals, **updated})

    def to_config_and_state_dict(self):
        return self._locals, self.state_dict()

    @classmethod
    def from_config_and_state_dict(klass, config, state_dict):
        unet = klass(**config)
        unet.load_state_dict(state_dict)
        return unet

    def _fingerprint(self):
        """Identity of the parameter storage a plan was packed from: (data_ptr, in-place version counter) of every parameter.
        load_state_dict (also through a parent module's), .to(device), p.data.copy_() / EMA swaps all change it."""
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    # --- plans ---------------------------------------------------------------------------------
    def plan(self, R, B, H, W, n_slots, device=None):
        device = device if device is not None else next(self.parameters()).device
        device = torch.device(device)
        if device.type != 'cuda':
            raise _lib.B200Error('imagen_pytorch_b200.Unet runs on an sm_100 CUDA device only (no CPU / torch fallback); '
                                 'move the module to cuda first')
        _lib.require_device(device.index if device.index is not None else torch.cuda.current_device())
        key = (R, B, H, W, n_slots, str(device), self._gemm_impl)
        fp = self._fingerprint()
        if any(pl.fingerprint != fp for pl in self._plans.values()):            # parameters moved or were updated in place: packed weights are stale
            self._plans.clear()
        if key not in self._plans:
            with torch.no_grad(), torch.cuda.device(device):
                self._plans[key] = UnetPlan(self, R, B, H, W, n_slots, device, self._gemm_impl)
        return self._plans[key]

    @torch.no_grad()
    def _run(self, x, time, keep_rows, R, *, lowres_cond_img, lowres_noise_times, text_embeds, text_mask, self_cond=None, cond_images=None):
        B, _, H, W = x.shape
        plan = self.plan(R, B, H, W, B, x.device)
        with torch.cuda.device(x.device):
            plan.prepare(time, text_embeds=text_embeds, text_mask=text_mask, keep=keep_rows, lowres_cond_img=lowres_cond_img,
                         lowres_noise_times=lowres_noise_times, slot_of_row=torch.arange(R, device=x.device) % B, cond_images=cond_images)
            plan.x_in.copy_(x.to(torch.float32))
            if self.self_cond:                                                  # default: zeros_like(x) (:1542)
                plan.sc_in.zero_() if self_cond is None else plan.sc_in.copy_(self_cond.to(torch.float32))
            plan.launch()
        return plan.pred

    @torch.no_grad()
    def forward(self, x, time, *, lowres_cond_img=None, lowres_noise_times=None, text_embeds=None, text_mask=None,
                cond_images=None, self_cond=None, cond_drop_prob=0.):
        assert not (self.lowres_cond and lowres_cond_img is None), 'low resolution conditioning image must be present'
        assert not (self.lowres_cond and lowres_noise_times is None), 'low resolution conditioning noise time must be present'
        B = x.shape[0]
        if cond_drop_prob == 1:
            keep = torch.zeros(B, dtype=torch.bool, device=x.device)
        elif cond_drop_prob == 0:
            keep = torch.ones(B, dtype=torch.bool, device=x.device)
        else:                                                                   # prob_mask_like (:201-207)
            keep = torch.zeros(B, device=x.device).float().uniform_(0, 1) < (1 - cond_drop_prob)
        out = self._run(x, time, keep, B, lowres_cond_img=lowres_cond_img, lowres_noise_times=lowres_noise_times,
                        text_embeds=text_embeds, text_mask=text_mask, self_cond=self_cond, cond_images=cond_images)
        return out.clone()

    @torch.no_grad()
    def forward_with_cond_scale(self, x, time, *, cond_scale=1., **kwargs):    # :1510-1522
        if cond_scale == 1:
            return self.forward(x, time, **kwargs)
        B = x.shape[0]
        keep = torch.cat((torch.ones(B, dtype=torch.bool, device=x.device), torch.zeros(B, dtype=torch.bool, device=x.device)))
        out = self._run(x, time, keep, 2 * B, lowres_cond_img=kwargs.get('lowres_cond_img'), lowres_noise_times=kwargs.get('lowres_noise_times'),
                        text_embeds=kwargs.get('text_embeds'), text_mask=kwargs.get('text_mask'), self_cond=kwargs.get('self_cond'),
                        cond_images=kwargs.get('cond_images'))
        logits, null_logits = out[:B], out[B:]
        return null_logits + (logits - null_logits) * cond_scale


class NullUnet(nn.Module):
    """Placeholder U-Net (imagen_pytorch.py:1729-1739)."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        self.lowres_cond = False
        self.dummy_parameter = nn.Parameter(torch.tensor([0.]))

    def cast_model_parameters(self, *args, **kwargs):
        return self

    def forward(self, x, *args, **kwargs):
        return x


def _preset(defaults):
    class _P(Unet):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **{**defaults, **kwargs})
    return _P


# presets with the hyper-parameters of the paper's appendix (imagen_pytorch.py:1743-1783)
BaseUnet64 = _preset(dict(dim=512, dim_mults=(1, 2, 3, 4), num_resnet_blocks=3, layer_attns=(False, True, True, True),
                          layer_cross_attns=(False, True, True, True), attn_heads=8, ff_mult=2., memory_efficient=False))
SRUnet256 = _preset(dict(dim=128, dim_mults=(1, 2, 4, 8), num_resnet_blocks=(2, 4, 8, 8), layer_attns=(False, False, False, True),
                         layer_cross_attns=(False, False, False, True), attn_heads=8, ff_mult=2., memory_efficient=True))
SRUnet1024 = _preset(dict(dim=128, dim_mults=(1, 2, 4, 8), num_resnet_blocks=(2, 4, 8, 8), layer_attns=False,
                          layer_cross_attns=(False, False, False, True), attn_heads=8, ff_mult=2., memory_efficient=True))
BaseUnet64.__name__, SRUnet256.__name__, SRUnet1024.__name__ = 'BaseUnet64', 'SRUnet256', 'SRUnet1024'
