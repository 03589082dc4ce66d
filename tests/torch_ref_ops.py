"""TEST INFRASTRUCTURE — a plain-torch op set with the same interface as panacea_b200.ops.NativeOps.

It exists so that the host-side orchestration (panacea_b200/engine.py: packing, layouts, epilogue fusion
bookkeeping, view/neighbour tables, caching) can be checked on CPU, without a GPU, against the oracle and the
reference's golden outputs. It is never imported by the package: the product path has no fallback.
Semantics follow include/panacea_b200.h literally (channels-last, fused epilogues).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

F32 = torch.float32


class TorchRefOps:
    """fp32 everywhere: operands are plain fp32 tensors, weights stay fp32."""
    operand_mult = 1
    qkv_dtype = F32
    act_dtype = F32
    fused_operand_emit = False
    token_dtype = F32
    fold_layernorm = False

    def __init__(self):
        self.launches = 0

    def pack_matrix(self, w, taps=1):
        return w.detach().to(F32).contiguous()

    def pack_small(self, w):
        return w.detach().to(F32).contiguous()

    def gemm(self, a, w, *, bias=None, rowvec=None, rows_per_group=0, n_groups=0, residual=None, residual2=None,
             geglu=False, out_dtype=F32, taps=(1, 1), out=None, ln=None, ln_stats_out=False):
        th, tw = taps
        C = a.shape[-1]
        N = w.shape[0]
        wf = w.float()
        if (th, tw) == (1, 1):
            lead = a.shape[:-1]
            y = a.float().reshape(-1, C) @ wf.t()
            if ln is not None:      # pn_gemm_args.ln_*: finish the folded LayerNorm from the producer's partial row sums
                st, colsum, eps = ln
                sm, sq = st[..., 0].sum(1), st[..., 1].sum(1)
                mu = sm / C
                rstd = torch.rsqrt((sq / C - mu * mu).clamp_min(0) + eps)
                y = rstd[:, None] * (y - mu[:, None] * colsum[None, :])
        else:
            NB, H, W, _ = a.shape
            lead = (NB, H, W)
            ap = F.pad(a.float(), (0, 0, tw // 2, tw // 2, th // 2, th // 2))
            y = torch.zeros(NB * H * W, N)
            for i in range(th):
                for j in range(tw):
                    tap = i * tw + j
                    y += ap[:, i:i + H, j:j + W, :].reshape(-1, C) @ wf[:, tap * C:(tap + 1) * C].t()
        rows = y.shape[0]
        if bias is not None:
            y = y + bias
        if rowvec is not None:
            grp = (torch.arange(rows) // rows_per_group) % n_groups
            y = y + rowvec[grp]
        if geglu:
            y3 = y.reshape(rows, -1, 2, 16)          # packed layout: 16 value columns, then their 16 gate columns
            y = (y3[:, :, 0] * F.gelu(y3[:, :, 1])).reshape(rows, -1)
        if residual is not None:
            y = y + residual.reshape(rows, -1)
        if residual2 is not None:
            y = y + residual2.reshape(rows, -1)
        y = y.to(out_dtype)
        stats = None
        if ln_stats_out:            # two partial (sum, sumsq) pairs per 160-wide column tile, like the streaming epilogue
            yy = y.float()
            n = yy.shape[1]
            bn = 160 if n % 160 == 0 else 128
            parts = []
            for c0 in range(0, n, bn):
                for chunks in ((0, 2, 4), (1, 3)) if bn == 160 else ((0, 2), (1, 3)):
                    cols = torch.cat([yy[:, c0 + 32 * c:c0 + 32 * c + 32] for c in chunks], 1)
                    parts.append(torch.stack([cols.sum(1), (cols * cols).sum(1)], -1))
            stats = torch.stack(parts, 1).contiguous()
        if out is not None:
            out.reshape(rows, -1).copy_(y)
            res = out.reshape(*lead, y.shape[1])
        else:
            res = y.reshape(*lead, y.shape[1])
        return (res, stats) if ln_stats_out else res

    def groupnorm(self, x, gamma, beta, eps, silu, want_raw=False, out_f32=False):
        Fr, C = x.shape[0], x.shape[-1]
        z = x.reshape(Fr, -1, C).permute(0, 2, 1)
        y = F.group_norm(z, 32, gamma, beta, eps)
        if silu:
            y = F.silu(y)
        y = y.permute(0, 2, 1).reshape(x.shape).contiguous()
        return (y, x.clone()) if want_raw else y

    def groupnorm_pixel(self, x, gamma, beta, eps, silu):
        b, T, P, C = x.shape
        z = x.permute(0, 2, 3, 1).reshape(b * P, C, T)
        y = F.group_norm(z, 32, gamma, beta, eps)
        if silu:
            y = F.silu(y)
        return y.reshape(b, P, C, T).permute(0, 3, 1, 2).contiguous()

    def layernorm(self, x, gamma, beta, eps=1e-5):
        return F.layer_norm(x, (x.shape[-1],), gamma, beta, eps)

    @staticmethod
    def _mha(q, k, v, heads):
        B, Nq, C = q.shape
        d = C // heads
        qh = q.reshape(B, Nq, heads, d).transpose(1, 2)
        kh = k.reshape(B, -1, heads, d).transpose(1, 2)
        vh = v.reshape(B, -1, heads, d).transpose(1, 2)
        s = (qh @ kh.transpose(-1, -2)) * (d ** -0.5)
        return (s.softmax(-1) @ vh).transpose(1, 2).reshape(B, Nq, C)

    def attention_view(self, qkv, heads, cross, neighbours):
        Fr, H, V, w, C3 = qkv.shape
        C = C3 // 3
        q, k, v = qkv.float().split(C, dim=-1)
        out = torch.empty(Fr, H, V, w, C)
        for i in range(V):
            nb = neighbours[i] if cross else (i,)
            ki = torch.cat([k[:, :, j] for j in nb], dim=2).reshape(Fr, -1, C)
            vi = torch.cat([v[:, :, j] for j in nb], dim=2).reshape(Fr, -1, C)
            out[:, :, i] = self._mha(q[:, :, i].reshape(Fr, H * w, C), ki, vi, heads).reshape(Fr, H, w, C)
        return out.to(qkv.dtype)

    def attention_text(self, q, kv, heads):
        C = q.shape[-1]
        return self._mha(q.float(), kv.float()[..., :C], kv.float()[..., C:], heads).to(q.dtype)

    def attention_temporal(self, qkv, heads):
        b, T, P, C3 = qkv.shape
        C = C3 // 3
        q, k, v = qkv.float().split(C, dim=-1)
        seq = lambda z: z.permute(0, 2, 1, 3).reshape(b * P, T, C)
        o = self._mha(seq(q), seq(k), seq(v), heads)
        return o.reshape(b, P, T, C).permute(0, 2, 1, 3).contiguous().to(qkv.dtype)

    def conv3x3_direct(self, x, w_packed, bias, cout, *, stride=1, silu=False, addend=None, out_dtype=F32):
        cin = x.shape[-1]
        w = w_packed[:, :cin, :cout].reshape(3, 3, cin, cout).permute(3, 2, 0, 1)
        y = F.conv2d(x.float().permute(0, 3, 1, 2), w, bias, stride=stride, padding=1)
        if silu:
            y = F.silu(y)
        y = y.permute(0, 2, 3, 1)
        if addend is not None:
            y = y + addend
        return y.contiguous().to(out_dtype)

    def im2col_s2(self, x, pad=1):
        Fr, H, W, C = x.shape
        if pad == 1:
            Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
            xp = F.pad(x, (0, 0, 1, 1, 1, 1))
        else:
            Ho, Wo = (H - 2) // 2 + 1, (W - 2) // 2 + 1
            xp = F.pad(x, (0, 0, 0, 2, 0, 2))
        cols = torch.stack([xp[:, i:i + 2 * Ho:2, j:j + 2 * Wo:2, :] for i in range(3) for j in range(3)], dim=3)
        return cols.reshape(Fr * Ho * Wo, 9 * C), (Fr, Ho, Wo)

    def upsample2x(self, x):
        return x.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2)

    def concat_add(self, h, skip, ctrl):
        return torch.cat([h, skip if ctrl is None else skip + ctrl], dim=-1)

    def add_(self, x, y):
        return x.add_(y)

    def cast_operand(self, x):
        return x

    def softmax_rows(self, s, scale):
        return torch.softmax(s.float() * scale, dim=-1)

    def nchw_to_nhwc(self, x, out=None, ch_off=0):
        y = x.permute(0, 2, 3, 1)
        if out is None:
            return y.contiguous()
        out[..., ch_off:ch_off + x.shape[1]] = y
        return out

    def nhwc_to_nchw(self, x, channels=None):
        return (x if channels is None else x[..., :channels]).permute(0, 3, 1, 2).contiguous()

    def timestep_embedding(self, t, dim):
        half = dim // 2
        freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=F32) / half)
        args = t[:, None].float() * freqs[None]
        return torch.cat([torch.cos(args), torch.sin(args)], dim=-1)

    def linear_small(self, x, w, bias, silu_in=False, silu_out=False):
        y = F.linear(F.silu(x) if silu_in else x, w.float(), bias)
        return F.silu(y) if silu_out else y

    def sampler_step(self, mode, x, net2=None, x_in_next=None, *, x_eval=None, d=None, old_denoised=None, noise=None,
                     seed=None, draw=0, sigma=1.0, sigma_q=None, dt=0.0, scale=1.0, c_in_next=0.0, m=(0.0, 0.0, 0.0, 0.0),
                     noise_mul=1.0, noise_amp=0.0, lms_coeff=(), lms_ring=0, lms_slot=0, use_old=False,
                     net_is_denoised=False):
        """pn_sampler_step restated with fp32 torch tensor ops in the reference's operation order
        (include/panacea_b200.h). Noise comes from the caller's buffer only: the in-kernel Philox is not restated here."""
        self.launches += 1
        n = x.shape[0]
        m1, m2, m3, m4 = m
        new_x, next_in = x, None
        if mode != "input":
            xe = x_eval if mode in ("heun_b", "dpmpp2s_b") else x
            du, dc = net2[:n], net2[n:]
            if not net_is_denoised:
                sq = sigma if sigma_q is None else sigma_q
                du, dc = du * -sq + xe, dc * -sq + xe
            den = du + scale * (dc - du)
        if mode == "euler":
            new_x = x + dt * ((x - den) / sigma)
        elif mode == "heun_a":
            dd = (x - den) / sigma
            d.copy_(dd)
            next_in = x + dt * dd
            x_eval.copy_(next_in)
        elif mode == "heun_b":
            new_x = x + ((d + (x_eval - den) / sigma) / 2.0) * dt
        elif mode == "dpmpp2s_a":
            next_in = m1 * x - m2 * den
            x_eval.copy_(next_in)
        elif mode == "dpmpp2s_b":
            new_x = m3 * x - m4 * den
        elif mode == "dpmpp2m":
            new_x = m1 * x - m2 * ((m3 * den - m4 * old_denoised) if use_old else den)
            old_denoised.copy_(den)
        elif mode == "lms":
            ring = d.view(lms_ring, *x.shape)
            ring[lms_slot] = (x - den) / sigma
            acc = 0
            for j, c in enumerate(lms_coeff):
                acc = acc + c * ring[(lms_slot - j) % lms_ring]
            new_x = x + acc
        if next_in is None:
            if seed is not None:
                raise NotImplementedError("in-kernel Philox noise is not restated on the CPU")
            if noise is not None:
                new_x = new_x + noise * noise_mul * noise_amp
            x.copy_(new_x)
            next_in = x
        if x_in_next is not None:
            x_in_next.copy_(torch.cat([next_in, next_in]) * c_in_next)
        return x

    def scale_dup(self, x, s, copies):
        return torch.cat([x * s] * copies)


class TorchFoldOps(TorchRefOps):
    """TorchRefOps with the LayerNorm fold switched on (the NativeOps fast-path orchestration: row statistics from the
    producers of the token stream, W diag(gamma) / column sums / W beta in the consumers), fp32 stream on CPU."""
    fold_layernorm = True
    LN_FOLD_MAX_C = 640


def _enc(x):
    """operand.cuh PN_OP_SPLIT3: fp32 [..., C] -> bf16 [..., 3C] = [hi | lo | hi]."""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo, hi], dim=-1)


class TorchSplitOps(TorchRefOps):
    """CPU emulation of panacea_b200.ops.ParityOps: producers store split-bf16 operands [hi | lo | hi], weights are
    packed [W_hi | W_hi | W_lo] by the product's own split3(), and the GEMM multiplies the bf16 VALUES exactly as the
    tensor core does (bf16 x bf16 products are exact in fp32). Checks the engine's parity-mode packing/orchestration and
    the precision claim of the encoding without a GPU."""
    operand_mult = 3

    def pack_matrix(self, w, taps=1):
        from panacea_b200.ops import split3
        return split3(w, taps)

    def gemm(self, a, w, *, geglu=False, out_dtype=F32, **kw):
        y = super().gemm(a, w, geglu=geglu, out_dtype=F32, **kw)
        return _enc(y) if geglu else y

    def groupnorm(self, x, gamma, beta, eps, silu, want_raw=False, out_f32=False):
        r = super().groupnorm(x, gamma, beta, eps, silu, want_raw)
        if out_f32:
            return r
        return (_enc(r[0]), _enc(r[1])) if want_raw else _enc(r)

    def groupnorm_pixel(self, *a, **k):
        return _enc(super().groupnorm_pixel(*a, **k))

    def layernorm(self, *a, **k):
        return _enc(super().layernorm(*a, **k))

    def attention_view(self, *a, **k):
        return _enc(super().attention_view(*a, **k))

    def attention_text(self, *a, **k):
        return _enc(super().attention_text(*a, **k))

    def attention_temporal(self, *a, **k):
        return _enc(super().attention_temporal(*a, **k))

    def im2col_s2(self, x, pad=1):
        cols, geo = super().im2col_s2(x, pad)
        C = x.shape[-1]
        return _enc(cols.reshape(cols.shape[0], 9, C)).reshape(cols.shape[0], 27 * C), geo

    def upsample2x(self, x):
        return _enc(super().upsample2x(x))

    def cast_operand(self, x):
        return _enc(x)
