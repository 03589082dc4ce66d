"""Op layer: torch CUDA tensors in, hand-written sm_100a kernels (via the C ABI) out.

Every method validates shapes/dtypes, builds the plain-C argument struct and launches on torch's current
stream. No method computes anything in torch: torch is only the allocator and stream owner here.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

BF16 = torch.bfloat16
F32 = torch.float32
OP_BF16, OP_SPLIT3, OP_F32 = 0, 1, 2      # include/panacea_b200.h pn_operand_mode
SAMPLER_MODES = {"input": 0, "euler": 1, "heun_a": 2, "heun_b": 3, "dpmpp2s_a": 4, "dpmpp2s_b": 5, "dpmpp2m": 6,
                 "lms": 7}                 # include/panacea_b200.h pn_sampler_mode
NOISE_NONE, NOISE_PHILOX, NOISE_BUFFER = 0, 1, 2   # pn_noise_source


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(cond, msg):
    if not cond:
        raise ValueError(msg)


def geglu_pack(t: torch.Tensor) -> torch.Tensor:
    """Row layout the GEGLU epilogue of pn_gemm expects, from the reference's [value rows | gate rows] layout
    (GEGLU.proj, attention.py:94-99): blocks of 32 rows = 16 value rows then the 16 gate rows of the same outputs,
    so one 32-column accumulator chunk holds both halves of 16 outputs (and packs into f32x2 register pairs)."""
    half = t.shape[0] // 2
    _req(t.shape[0] % 32 == 0, "geglu_pack: 2*inner must be a multiple of 32")
    v = t[:half].reshape(half // 16, 16, *t.shape[1:])
    g = t[half:].reshape(half // 16, 16, *t.shape[1:])
    return torch.stack([v, g], 1).reshape(t.shape).contiguous()


def split3(t: torch.Tensor, taps: int = 1) -> torch.Tensor:
    """Parity-mode packing of a WEIGHT matrix [N, taps*C] (fp32) -> bf16 [N, taps*3C]: per tap [W_hi | W_hi | W_lo] with
    W_hi = bf16(W), W_lo = bf16(W - W_hi). Against an activation operand stored [a_hi | a_lo | a_hi] (operand.cuh)
    the bf16 GEMM then computes a_hi W_hi + a_lo W_hi + a_hi W_lo = a W up to 2^-18 relative."""
    n, k = t.shape
    w = t.detach().to(F32).reshape(n, taps, k // taps)
    hi = w.to(BF16)
    lo = (w - hi.to(F32)).to(BF16)
    return torch.cat([hi, hi, lo], dim=2).reshape(n, 3 * k).contiguous()


class NativeOps:
    """The production op set (bf16 operands). `launches` counts kernel launches issued through the C ABI.
    `operand_mode` / `operand_mult` describe how producers store GEMM operands (ParityOps overrides them)."""

    operand_mode = OP_BF16
    operand_mult = 1          # operand row width = operand_mult * C
    qkv_dtype = BF16          # dtype of attention inputs
    act_dtype = BF16          # dtype of intermediates consumed by CUDA-core kernels (hint stem, GEGLU output, head input)
    fused_operand_emit = True # a GEMM epilogue may store the next GEMM's operand directly (out_dtype=bf16)
    token_dtype = BF16        # token stream inside a transformer block (proj_in .. proj_out): 3 residual adds per block
    fold_layernorm = True     # LayerNorm folded into the GEMMs around the bf16 token stream (C <= LN_FOLD_MAX_C)
    LN_FOLD_MAX_C = 640       # the producers' streaming bf16 epilogue (which emits the row sums) covers K <= 640

    def __init__(self):
        import os
        self.lib = _lib.load()
        self.launches = 0
        self._freqs = {}
        if os.environ.get("PN_TOKEN_F32") == "1" and self.operand_mode == OP_BF16:      # A/B measurement of the bf16 token stream
            self.token_dtype = F32
        if os.environ.get("PN_LN_FOLD") == "0" or self.token_dtype != BF16:              # A/B measurement of the LayerNorm fold
            self.fold_layernorm = False

    def pack_matrix(self, w: torch.Tensor, taps: int = 1) -> torch.Tensor:
        """fp32 weight [N, taps*C] -> the B operand pn_gemm reads in this op set's precision mode."""
        return w.detach().to(BF16).contiguous()

    def pack_small(self, w: torch.Tensor) -> torch.Tensor:
        """weight of the M<=32 time-embedding linears (pn_linear_small)."""
        return w.detach().to(BF16).contiguous()

    def _operand_empty(self, shape, device, mode=None):
        mode = self.operand_mode if mode is None else mode
        if mode == OP_F32:
            return torch.empty(shape, device=device, dtype=F32)
        if mode == OP_SPLIT3:
            return torch.empty((*shape[:-1], 3 * shape[-1]), device=device, dtype=BF16)
        return torch.empty(shape, device=device, dtype=BF16)

    # ------------------------------------------------------------------ GEMM / implicit conv
    def gemm(self, a, w, *, bias=None, rowvec=None, rows_per_group=0, n_groups=0, residual=None, residual2=None,
             geglu=False, out_dtype=F32, taps=(1, 1), out=None, ln=None, ln_stats_out=False):
        """out[row, :] = epi(sum_taps A[shifted pixel] @ w^T). See include/panacea_b200.h::pn_gemm.

        a: bf16 [..., C] (taps == (1,1): any leading dims, rows may be strided views with C contiguous)
           or bf16 [NB, H, W, C] for taps (3,3) / (3,1).
        w: bf16 [N, taps_h*taps_w*C].
        ln = (stats fp32 [rows, parts, 2], colsum fp32 [N], eps): LayerNorm of the rows of `a` (the un-normalised bf16
             token stream) folded into this GEMM, w = W diag(gamma), bias = W beta (+ bias); see pn_gemm_args.
        ln_stats_out: also return the per-row partial (sum, sumsq) of the bf16 output rows: (out, stats).
        """
        _req(a.is_cuda and a.dtype == BF16 and w.dtype == BF16, "gemm: a and w must be CUDA bf16")
        _req(a.stride(-1) == 1 and w.is_contiguous(), "gemm: innermost dim must be contiguous")
        th, tw = taps
        Cc = a.shape[-1]
        N = w.shape[0]
        _req(w.shape[1] == th * tw * Cc, f"gemm: weight K {w.shape[1]} != taps*C {th * tw * Cc}")
        if (th, tw) == (1, 1):
            lead = a.shape[:-1]
            a2 = a.reshape(-1, Cc) if a.is_contiguous() else a
            if a2.dim() != 2:
                # strided view: collapse leading dims only if they are uniformly strided
                rows = 1
                for s in lead:
                    rows *= s
                st = a.stride(-2)
                ok = all(a.stride(i) == a.stride(i + 1) * a.shape[i + 1] for i in range(a.dim() - 2))
                _req(ok, "gemm: cannot flatten strided A view")
                a2 = a.as_strided((rows, Cc), (st, 1))
            NB, H, W = 1, 1, a2.shape[0]
            sw = a2.stride(0)
            sh = sw * W
            sn = sh
            a_use = a2
        else:
            _req(a.dim() == 4, "gemm: conv mode expects [NB,H,W,C]")
            NB, H, W = a.shape[0], a.shape[1], a.shape[2]
            sn, sh, sw = a.stride(0), a.stride(1), a.stride(2)
            lead = a.shape[:-1]
            a_use = a
        rows = NB * H * W
        n_out = N // 2 if geglu else N
        if out is None:
            out = torch.empty((rows, n_out), device=a.device, dtype=out_dtype)
        else:
            _req(out.dtype == out_dtype and out.stride(-1) == 1, "gemm: bad out tensor")
        out2 = out.reshape(rows, -1) if out.is_contiguous() else out
        args = _lib.GemmArgs()
        args.A = a_use.data_ptr(); args.B = w.data_ptr(); args.out = out2.data_ptr()
        args.bias = None if bias is None else bias.data_ptr()
        args.rowvec = None if rowvec is None else rowvec.data_ptr()
        args.residual = None if residual is None else residual.data_ptr()
        if bias is not None:
            _req(bias.dtype == F32 and bias.numel() == N, "gemm: bias must be fp32 [N]")
        if rowvec is not None:
            _req(rowvec.dtype == F32 and rowvec.dim() == 2 and rowvec.stride(1) == 1 and rowvec.shape[1] == N,
                 "gemm: rowvec fp32 [G,N] (rows may be strided)")
            _req(rows_per_group > 0 and n_groups > 0 and rowvec.shape[0] == n_groups, "gemm: rowvec groups")
            args.rowvec_ld = rowvec.stride(0)
        if residual is not None:
            _req(residual.stride(-1) == 1 and (residual.dtype == F32 or (residual.dtype == BF16 and out_dtype == BF16)),
                 "gemm: residual must be fp32 (or bf16 with a bf16 output)")
            r2 = residual.reshape(rows, -1) if residual.is_contiguous() else residual
            args.ldr = r2.stride(0)
            args.residual_bf16 = int(residual.dtype == BF16)
        if residual2 is not None:
            _req(residual2.dtype == F32 and residual2.is_contiguous() and out_dtype == F32, "gemm: residual2 must be fp32")
            args.residual2 = residual2.data_ptr()
            args.ldr2 = residual2.numel() // rows
        args.NB, args.H, args.W, args.C = NB, H, W, Cc
        args.a_stride_w, args.a_stride_h, args.a_stride_n = sw, sh, sn
        args.ldo = out2.stride(0)
        args.N = N; args.taps_h = th; args.taps_w = tw
        args.rows_per_group = rows_per_group; args.n_groups = n_groups
        args.out_bf16 = 1 if out_dtype == BF16 else 0
        args.geglu = 1 if geglu else 0
        stats = None
        if ln is not None:
            st_in, colsum, eps = ln
            _req(st_in.dtype == F32 and st_in.is_contiguous() and st_in.dim() == 3 and st_in.shape[0] == rows and st_in.shape[2] == 2,
                 "gemm: ln stats must be fp32 [rows, parts, 2]")
            _req(colsum.dtype == F32 and colsum.numel() == N, "gemm: ln colsum must be fp32 [N]")
            args.ln_stats_in, args.ln_colsum, args.ln_parts_in, args.ln_eps = st_in.data_ptr(), colsum.data_ptr(), st_in.shape[1], float(eps)
        if ln_stats_out:
            parts = self.lib.pn_gemm_ln_parts(N)
            _req(parts > 0, "gemm: ln_stats_out needs N % 160 == 0 or N % 128 == 0")
            stats = torch.empty((rows, parts, 2), device=a.device, dtype=F32)
            args.ln_stats_out = stats.data_ptr()
        _lib.check(self.lib.pn_gemm(C.byref(args), _stream()), "pn_gemm")
        self.launches += 1
        res = out.reshape(*lead, n_out) if out.is_contiguous() else out
        return (res, stats) if ln_stats_out else res

    # ------------------------------------------------------------------ normalisation
    def groupnorm(self, x, gamma, beta, eps, silu, want_raw=False, out_f32=False):
        """x fp32 [F, P, C] (or [F,H,W,C]) -> operand of the same shape (bf16; [.., 3C] in parity mode; fp32 when
        out_f32, for a CUDA-core consumer); statistics over (C/32, all pixels of a frame)."""
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous(), "groupnorm: x must be contiguous CUDA fp32")
        Fr, Cc = x.shape[0], x.shape[-1]
        P = x.numel() // (Fr * Cc)
        mode = OP_F32 if out_f32 else self.operand_mode
        y = self._operand_empty(x.shape, x.device, mode)
        raw = self._operand_empty(x.shape, x.device, mode) if want_raw else None
        nws = self.lib.pn_groupnorm_workspace_floats(Fr, P, Cc)
        ws = torch.empty(nws, device=x.device, dtype=F32)
        _lib.check(self.lib.pn_groupnorm_silu(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(raw), _ptr(ws), Fr, P, Cc,
                                             float(eps), int(bool(silu)), mode, _stream()), "pn_groupnorm_silu")
        self.launches += 2        # counter memset + kernel
        return (y, raw) if want_raw else y

    def groupnorm_pixel(self, x, gamma, beta, eps, silu):
        """x fp32 [b, T, P, C] -> bf16; statistics over (C/32, T) per pixel (temporal branch of ResBlock3D)."""
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous() and x.dim() == 4, "groupnorm_pixel: x fp32 [b,T,P,C]")
        b, T, P, Cc = x.shape
        y = self._operand_empty(x.shape, x.device)
        _lib.check(self.lib.pn_groupnorm_pixel_silu(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), b, T, P, Cc, float(eps),
                                                   int(bool(silu)), self.operand_mode, _stream()), "pn_groupnorm_pixel_silu")
        self.launches += 1
        return y

    def layernorm(self, x, gamma, beta, eps=1e-5):
        _req(x.is_cuda and x.dtype in (F32, BF16) and x.is_contiguous(), "layernorm: x must be contiguous CUDA fp32 / bf16")
        Cc = x.shape[-1]
        rows = x.numel() // Cc
        y = self._operand_empty(x.shape, x.device)
        _lib.check(self.lib.pn_layernorm(_ptr(x), int(x.dtype == BF16), _ptr(gamma), _ptr(beta), _ptr(y), rows, Cc, float(eps),
                                         self.operand_mode, _stream()), "pn_layernorm")
        self.launches += 1
        return y

    # ------------------------------------------------------------------ attention
    def _attention(self, q, k, v, out, *, q_ld, kv_ld, out_ld, F, H, V, W, Hk, Vk, Wk, kv_frame_div, heads, views, head_dim=64):
        a = _lib.AttnArgs()
        a.q, a.k, a.v, a.out = q, k, v, out
        a.q_ld, a.kv_ld, a.out_ld = q_ld, kv_ld, out_ld
        a.F, a.H, a.V, a.W = F, H, V, W
        a.Hk, a.Vk, a.Wk = Hk, Vk, Wk
        a.kv_frame_div = kv_frame_div
        a.heads, a.head_dim = heads, head_dim
        for vi, lst in enumerate(views):
            a.kv_view_count[vi] = len(lst)
            for j, kvv in enumerate(lst):
                a.kv_views[vi][j] = kvv
        a.scale = head_dim ** -0.5
        _lib.check(self.lib.pn_attention(C.byref(a), _stream()), "pn_attention")
        self.launches += 1

    def attention_view(self, qkv, heads, cross, neighbours):
        """qkv bf16 [F, H, V, w, 3C] (fused q|k|v channels) -> bf16 [F, H, V, w, C].
        cross=False: each view attends itself; cross=True: view v attends neighbours[v]."""
        _req(qkv.is_cuda and qkv.dtype == BF16 and qkv.is_contiguous() and qkv.dim() == 5, "attention_view: qkv bf16 [F,H,V,w,3C]")
        Fr, H, V, w, C3 = qkv.shape
        Cc = C3 // 3
        d = Cc // heads
        _req(Cc == heads * d and d in (64, 80), "attention_view: head_dim must be 64 or 80")
        out = torch.empty((Fr, H, V, w, Cc), device=qkv.device, dtype=BF16)
        views = [list(neighbours[v]) for v in range(V)] if cross else [[v] for v in range(V)]
        base = qkv.data_ptr()
        self._attention(base, base + 2 * Cc, base + 4 * Cc, out.data_ptr(), q_ld=C3, kv_ld=C3, out_ld=Cc, F=Fr, H=H, V=V, W=w,
                        Hk=H, Vk=V, Wk=w, kv_frame_div=1, heads=heads, views=views, head_dim=d)
        return out

    def attention_text(self, q, kv, heads):
        """q bf16 [b, Nq, C]; kv bf16 [b, Nk, 2C] (k | v channels), Nk <= 128 -> bf16 [b, Nq, C]."""
        _req(q.is_cuda and q.dtype == BF16 and q.is_contiguous() and kv.dtype == BF16 and kv.is_contiguous(), "attention_text: bf16 contiguous")
        b, Nq, Cc = q.shape
        Nk = kv.shape[1]
        d = Cc // heads
        _req(kv.shape[0] == b and kv.shape[2] == 2 * Cc and Cc == heads * d and d in (64, 80) and Nk <= (128 if d == 64 else 112),
             "attention_text: bad shapes")
        out = torch.empty_like(q)
        base = kv.data_ptr()
        self._attention(q.data_ptr(), base, base + 2 * Cc, out.data_ptr(), q_ld=Cc, kv_ld=2 * Cc, out_ld=Cc, F=b, H=1, V=1,
                        W=Nq, Hk=1, Vk=1, Wk=Nk, kv_frame_div=1, heads=heads, views=[[0]], head_dim=d)
        return out

    def attention_temporal(self, qkv, heads):
        """qkv bf16 [b, T, P, 3C] -> bf16 [b, T, P, C]; softmax over the T frames of each pixel."""
        _req(qkv.is_cuda and qkv.dtype == BF16 and qkv.is_contiguous() and qkv.dim() == 4, "attention_temporal: qkv bf16 [b,T,P,3C]")
        b, T, P, C3 = qkv.shape
        Cc = C3 // 3
        d = Cc // heads
        _req(Cc == heads * d and d in (64, 80), "attention_temporal: head_dim must be 64 or 80")
        out = torch.empty((b, T, P, Cc), device=qkv.device, dtype=BF16)
        base = qkv.data_ptr()
        _lib.check(self.lib.pn_attention_temporal(base, base + 2 * Cc, base + 4 * Cc, out.data_ptr(), b, T, P, heads, d, C3, Cc,
                                                 d ** -0.5, _stream()), "pn_attention_temporal")
        self.launches += 1
        return out

    # ------------------------------------------------------------------ small convs / layout / sampler helpers
    def conv3x3_direct(self, x, w_packed, bias, cout, *, stride=1, silu=False, addend=None, out_dtype=F32):
        """x fp32|bf16 [F,H,W,Cin] channels-last; w_packed fp32 [9, Cin, Cout_pad]; -> [F,Ho,Wo,cout]."""
        _req(x.is_cuda and x.is_contiguous() and x.dim() == 4 and x.dtype in (F32, BF16), "conv3x3_direct: x [F,H,W,Cin]")
        Fr, H, W, Cin = x.shape
        _req(w_packed.dtype == F32 and w_packed.is_contiguous() and w_packed.shape[0] == 9 and w_packed.shape[1] == Cin,
             "conv3x3_direct: w_packed fp32 [9,Cin,Cout_pad]")
        cpad = w_packed.shape[2]
        Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
        y = torch.empty((Fr, Ho, Wo, cout), device=x.device, dtype=out_dtype)
        yf = _ptr(y) if out_dtype == F32 else None
        yb = _ptr(y) if out_dtype == BF16 else None
        _lib.check(self.lib.pn_conv3x3_direct(_ptr(x), int(x.dtype == BF16), _ptr(w_packed), _ptr(bias), _ptr(addend), yf, yb,
                                             Fr, H, W, Cin, cout, cpad, stride, int(bool(silu)), _stream()), "pn_conv3x3_direct")
        self.launches += 1
        return y

    def im2col_s2(self, x, pad=1):
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous() and x.dim() == 4, "im2col_s2: x fp32 [F,H,W,C]")
        Fr, H, W, Cc = x.shape
        Ho, Wo = ((H - 1) // 2 + 1, (W - 1) // 2 + 1) if pad == 1 else ((H - 2) // 2 + 1, (W - 2) // 2 + 1)
        out = torch.empty((Fr * Ho * Wo, 9 * self.operand_mult * Cc), device=x.device, dtype=BF16)
        _lib.check(self.lib.pn_im2col3x3_s2(_ptr(x), _ptr(out), Fr, H, W, Cc, pad, self.operand_mode, _stream()), "pn_im2col3x3_s2")
        self.launches += 1
        return out, (Fr, Ho, Wo)

    def upsample2x(self, x):
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous() and x.dim() == 4, "upsample2x: x fp32 [F,H,W,C]")
        Fr, H, W, Cc = x.shape
        y = self._operand_empty((Fr, 2 * H, 2 * W, Cc), x.device)
        _lib.check(self.lib.pn_upsample2x(_ptr(x), _ptr(y), Fr, H, W, Cc, self.operand_mode, _stream()), "pn_upsample2x")
        self.launches += 1
        return y

    def concat_add(self, h, skip, ctrl):
        _req(h.dtype == F32 and skip.dtype == F32 and h.is_contiguous() and skip.is_contiguous(), "concat_add: fp32 contiguous")
        C1, C2 = h.shape[-1], skip.shape[-1]
        rows = h.numel() // C1
        _req(skip.numel() // C2 == rows, "concat_add: row mismatch")
        out = torch.empty((*h.shape[:-1], C1 + C2), device=h.device, dtype=F32)
        _lib.check(self.lib.pn_concat_add(_ptr(h), _ptr(skip), _ptr(ctrl), _ptr(out), rows, C1, C2, _stream()), "pn_concat_add")
        self.launches += 1
        return out

    def add_(self, x, y):
        _req(x.dtype == F32 and y.dtype == F32 and x.is_contiguous() and y.is_contiguous() and x.numel() == y.numel(), "add_: fp32 same size")
        _lib.check(self.lib.pn_add_inplace(_ptr(x), _ptr(y), x.numel(), _stream()), "pn_add_inplace")
        self.launches += 1
        return x

    def cast_operand(self, x):
        """fp32 [..., C] -> GEMM operand (bf16 [..., C]; [..., 3C] in parity mode)."""
        _req(x.dtype == F32 and x.is_contiguous(), "cast_operand: fp32 contiguous")
        Cc = x.shape[-1]
        y = self._operand_empty(x.shape, x.device)
        _lib.check(self.lib.pn_cast_operand(_ptr(x), _ptr(y), x.numel() // Cc, Cc, self.operand_mode, _stream()), "pn_cast_operand")
        self.launches += 1
        return y

    def nchw_to_nhwc(self, x, out=None, ch_off=0):
        """x fp32 [F,C,H,W] -> out[F,H,W,ch_off:ch_off+C] (out may be wider: channel concat)."""
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous() and x.dim() == 4, "nchw_to_nhwc: x fp32 [F,C,H,W]")
        Fr, Cc, H, W = x.shape
        if out is None:
            out = torch.empty((Fr, H, W, Cc), device=x.device, dtype=F32)
        _lib.check(self.lib.pn_transpose_f32(_ptr(x), _ptr(out), Fr, Cc, H * W, H * W, out.shape[-1], ch_off, _stream()), "pn_transpose_f32")
        self.launches += 1
        return out

    def nhwc_to_nchw(self, x, channels=None):
        """x fp32 [F,H,W,C] -> [F, channels or C, H, W] (the first `channels` of C: the out-head GEMM pads its N to 8)."""
        _req(x.is_cuda and x.dtype == F32 and x.is_contiguous() and x.dim() == 4, "nhwc_to_nchw: x fp32 [F,H,W,C]")
        Fr, H, W, ld = x.shape
        Cc = ld if channels is None else channels
        _req(0 < Cc <= ld, "nhwc_to_nchw: channels out of range")
        out = torch.empty((Fr, Cc, H, W), device=x.device, dtype=F32)
        _lib.check(self.lib.pn_transpose_f32(_ptr(x), _ptr(out), Fr, H * W, Cc, ld, H * W, 0, _stream()), "pn_transpose_f32")
        self.launches += 1
        return out

    def timestep_embedding(self, t, dim):
        _req(t.is_cuda and t.dtype == torch.int64 and t.is_contiguous(), "timestep_embedding: t must be CUDA int64")
        out = torch.empty((t.numel(), dim), device=t.device, dtype=F32)
        key = (dim, t.device)
        if key not in self._freqs:
            # the reference's own expression on the host (util.py:236-240), so t * f is bit-identical to the reference's
            import math
            half = dim // 2
            self._freqs[key] = torch.exp(-math.log(10000) * torch.arange(start=0, end=half, dtype=F32) / half).to(t.device)
        _lib.check(self.lib.pn_timestep_embedding(_ptr(t), _ptr(out), t.numel(), dim, _ptr(self._freqs[key]), _stream()),
                   "pn_timestep_embedding")
        self.launches += 1
        return out

    def linear_small(self, x, w, bias, silu_in=False, silu_out=False):
        """x fp32 [M<=32, K]; w bf16 or fp32 [N, K]; -> fp32 [M, N]."""
        _req(x.dtype == F32 and x.is_contiguous() and w.dtype in (BF16, F32) and w.is_contiguous(), "linear_small: dtypes")
        M, K = x.shape
        N = w.shape[0]
        y = torch.empty((M, N), device=x.device, dtype=F32)
        _lib.check(self.lib.pn_linear_small(_ptr(x), _ptr(w), int(w.dtype == F32), _ptr(bias), _ptr(y), M, N, K, N, int(silu_in),
                                           int(silu_out), _stream()), "pn_linear_small")
        self.launches += 1
        return y

    def cfg_euler_step(self, x, net2, x_in_next, sigma, sigma_next, scale, c_in_next, sigma_q=None, net_is_denoised=False):
        """One CFG + Euler step from sigma to sigma_next: the "euler" mode of sampler_step. dt is the float32 difference
        of the float32-rounded sigmas, like the reference's tensors (a float64 difference can differ in the last bit)."""
        from .sgm.modules.diffusionmodules.sampling_utils import sub32      # not at the top: sgm imports this module
        return self.sampler_step("euler", x, net2, x_in_next, sigma=sigma, sigma_q=sigma_q, dt=sub32(sigma_next, sigma),
                                 scale=scale, c_in_next=c_in_next, net_is_denoised=net_is_denoised)

    def sampler_step(self, mode, x, net2=None, x_in_next=None, *, x_eval=None, d=None, old_denoised=None, noise=None,
                     seed=None, draw=0, sigma=1.0, sigma_q=None, dt=0.0, scale=1.0, c_in_next=0.0, m=(0.0, 0.0, 0.0, 0.0),
                     noise_mul=1.0, noise_amp=0.0, lms_coeff=(), lms_ring=0, lms_slot=0, use_old=False,
                     net_is_denoised=False):
        """One pn_sampler_step (include/panacea_b200.h): `mode` is a key of SAMPLER_MODES. Noise: `noise` (fp32, like x)
        adds those draws, otherwise `seed` (not None) adds the Philox draw `draw`, otherwise none is added."""
        n = x.numel()
        _req(x.dtype == F32 and x.is_contiguous(), "sampler_step: x must be fp32 contiguous")
        for name, t, size in (("net2", net2, 2 * n), ("x_in_next", x_in_next, 2 * n), ("x_eval", x_eval, n),
                              ("d", d, lms_ring * n if mode == "lms" else n), ("old_denoised", old_denoised, n), ("noise", noise, n)):
            _req(t is None or (t.dtype == F32 and t.is_contiguous() and t.numel() == size and t.device == x.device),
                 f"sampler_step: {name} must be fp32 contiguous with {size} elements on {x.device}")
        a = _lib.SamplerArgs()
        a.x, a.net2, a.x_in_next, a.x_eval, a.d, a.old_denoised, a.noise = (
            None if t is None else t.data_ptr() for t in (x, net2, x_in_next, x_eval, d, old_denoised, noise))
        a.n = n
        a.noise_source = NOISE_BUFFER if noise is not None else (NOISE_PHILOX if seed is not None else NOISE_NONE)
        a.seed, a.draw = (int(seed) if seed is not None else 0) & (2 ** 64 - 1), int(draw)
        a.sigma, a.sigma_q, a.dt = float(sigma), float(sigma if sigma_q is None else sigma_q), float(dt)
        a.cfg_scale, a.c_in_next = float(scale), float(c_in_next)
        a.m1, a.m2, a.m3, a.m4 = (float(v) for v in m)
        a.noise_mul, a.noise_amp = float(noise_mul), float(noise_amp)
        for j, c in enumerate(lms_coeff):
            a.lms_coeff[j] = float(c)
        a.mode = SAMPLER_MODES[mode]
        a.net_is_denoised, a.use_old = int(bool(net_is_denoised)), int(bool(use_old))
        a.lms_order, a.lms_ring, a.lms_slot = len(lms_coeff), int(lms_ring), int(lms_slot)
        _lib.check(self.lib.pn_sampler_step(C.byref(a), _stream()), "pn_sampler_step")
        self.launches += 1
        return x

    def philox_normal(self, shape, seed, draw=0, device="cuda"):
        """fp32 tensor of N(0,1) draws: element e is draw `draw` of e under `seed`, the values pn_sampler_step adds."""
        out = torch.empty(shape, device=device, dtype=F32)
        _lib.check(self.lib.pn_philox_normal(_ptr(out), out.numel(), int(seed) & (2 ** 64 - 1), int(draw), _stream()),
                   "pn_philox_normal")
        self.launches += 1
        return out

    def softmax_rows(self, s, scale):
        """fp32 [rows, N] -> bf16 [rows, N] = softmax(scale * s) per row (VAE mid-block attention)."""
        _req(s.is_cuda and s.dtype == F32 and s.dim() == 2 and s.is_contiguous() and s.shape[1] % 4 == 0, "softmax_rows: fp32 [rows, N]")
        out = torch.empty(s.shape, device=s.device, dtype=BF16)
        _lib.check(self.lib.pn_softmax_rows(_ptr(s), _ptr(out), s.shape[0], s.shape[1], s.stride(0), out.stride(0), float(scale),
                                           _stream()), "pn_softmax_rows")
        self.launches += 1
        return out

    def fingerprint(self, x):
        """(sum, weighted sum) of the 32-bit words of a contiguous CUDA tensor, as Python ints (synchronises)."""
        _req(x.is_cuda and x.is_contiguous() and (x.numel() * x.element_size()) % 4 == 0, "fingerprint: contiguous CUDA tensor")
        out = torch.empty(2, device=x.device, dtype=torch.int64)
        _lib.check(self.lib.pn_fingerprint(_ptr(x), x.numel() * x.element_size(), _ptr(out), _stream()), "pn_fingerprint")
        self.launches += 1
        a, b = out.tolist()
        return (a, b, tuple(x.shape), x.dtype)

    def scale_dup(self, x, s, copies):
        _req(x.dtype == F32 and x.is_contiguous(), "scale_dup: fp32 contiguous")
        out = torch.empty((copies * x.shape[0], *x.shape[1:]), device=x.device, dtype=F32)
        _lib.check(self.lib.pn_scale_dup(_ptr(x), _ptr(out), x.numel(), float(s), copies, _stream()), "pn_scale_dup")
        self.launches += 1
        return out


class ParityOps(NativeOps):
    """fp32-class precision mode (the literal rtol 1e-3 / atol 1e-4 bar of BASELINE.json against the reference's fp32
    math). Same kernels, different operand encoding: every producer stores the GEMM operand as bf16 [hi | lo | hi]
    (3C wide), weights are packed [W_hi | W_hi | W_lo], so the tcgen05 GEMM/conv kernel computes fp32-class products by
    K-concatenation; attention runs in fp32 on CUDA cores (pn_attention_f32); GEGLU uses the exact erf; the
    time-embedding linears read fp32 weights. About 3-4x the cost of the bf16 path."""

    operand_mode = OP_SPLIT3
    operand_mult = 3
    qkv_dtype = F32
    act_dtype = F32
    fused_operand_emit = False
    token_dtype = F32
    fold_layernorm = False

    def pack_matrix(self, w, taps=1):
        return split3(w, taps)

    def pack_small(self, w):
        return w.detach().to(F32).contiguous()

    def gemm(self, a, w, *, geglu=False, out_dtype=F32, **kw):
        if geglu:
            # fp32 GEMM output in the packed (16 value | 16 gate) column layout, then the exact-erf GEGLU as its own pass
            _req(kw.get("residual") is None and kw.get("out") is None, "parity gemm: GEGLU takes no residual / out")
            h = super().gemm(a, w, out_dtype=F32, **kw)
            inner = h.shape[-1] // 2
            rows = h.numel() // h.shape[-1]
            y = self._operand_empty((*h.shape[:-1], inner), h.device)
            _lib.check(self.lib.pn_geglu_operand(_ptr(h), _ptr(y), rows, inner, self.operand_mode, _stream()), "pn_geglu_operand")
            self.launches += 1
            return y
        _req(out_dtype == F32, "parity gemm: outputs are fp32 (operands are produced by cast_operand)")
        return super().gemm(a, w, out_dtype=F32, **kw)

    # ------------------------------------------------------------------ attention (fp32, CUDA cores)
    def _attention_f32(self, q, k, v, out, *, q_ld, kv_ld, F, H, V, W, Hk, Vk, Wk, heads, head_dim, views):
        a = _lib.AttnArgs()
        a.q, a.k, a.v, a.out = q, k, v, out
        a.q_ld, a.kv_ld, a.out_ld = q_ld, kv_ld, heads * head_dim
        a.F, a.H, a.V, a.W = F, H, V, W
        a.Hk, a.Vk, a.Wk = Hk, Vk, Wk
        a.kv_frame_div = 1
        a.heads, a.head_dim = heads, head_dim
        for vi, lst in enumerate(views):
            a.kv_view_count[vi] = len(lst)
            for j, kvv in enumerate(lst):
                a.kv_views[vi][j] = kvv
        a.scale = head_dim ** -0.5
        _lib.check(self.lib.pn_attention_f32(C.byref(a), self.operand_mode, _stream()), "pn_attention_f32")
        self.launches += 1

    def attention_view(self, qkv, heads, cross, neighbours):
        _req(qkv.is_cuda and qkv.dtype == F32 and qkv.is_contiguous() and qkv.dim() == 5, "attention_view(parity): qkv fp32 [F,H,V,w,3C]")
        Fr, H, V, w, C3 = qkv.shape
        Cc = C3 // 3
        d = Cc // heads
        out = self._operand_empty((Fr, H, V, w, Cc), qkv.device)
        views = [list(neighbours[v]) for v in range(V)] if cross else [[v] for v in range(V)]
        base = qkv.data_ptr()
        self._attention_f32(base, base + 4 * Cc, base + 8 * Cc, out.data_ptr(), q_ld=C3, kv_ld=C3, F=Fr, H=H, V=V, W=w, Hk=H, Vk=V, Wk=w,
                            heads=heads, head_dim=d, views=views)
        return out

    def attention_text(self, q, kv, heads):
        _req(q.is_cuda and q.dtype == F32 and q.is_contiguous() and kv.dtype == F32 and kv.is_contiguous(), "attention_text(parity): fp32")
        b, Nq, Cc = q.shape
        Nk = kv.shape[1]
        _req(kv.shape[0] == b and kv.shape[2] == 2 * Cc, "attention_text: bad shapes")
        out = self._operand_empty((b, Nq, Cc), q.device)
        base = kv.data_ptr()
        self._attention_f32(q.data_ptr(), base, base + 4 * Cc, out.data_ptr(), q_ld=Cc, kv_ld=2 * Cc, F=b, H=1, V=1, W=Nq, Hk=1, Vk=1,
                            Wk=Nk, heads=heads, head_dim=Cc // heads, views=[[0]])
        return out

    def attention_temporal(self, qkv, heads):
        _req(qkv.is_cuda and qkv.dtype == F32 and qkv.is_contiguous() and qkv.dim() == 4, "attention_temporal(parity): qkv fp32 [b,T,P,3C]")
        b, T, P, C3 = qkv.shape
        Cc = C3 // 3
        d = Cc // heads
        out = self._operand_empty((b, T, P, Cc), qkv.device)
        base = qkv.data_ptr()
        _lib.check(self.lib.pn_attention_temporal_f32(base, base + 4 * Cc, base + 8 * Cc, out.data_ptr(), b, T, P, heads, d, C3, d ** -0.5,
                                                     self.operand_mode, _stream()), "pn_attention_temporal_f32")
        self.launches += 1
        return out
