"""TEST INFRASTRUCTURE — CPU oracle: a plain-PyTorch fp32 restatement of the reference's denoising network
(wenyuqing/panacea: ControlNet3D + ControlledUNetModel3D behind OpenAIWrapperControlLDM3D).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
module, and only as the checker / the timed CPU baseline. The product (panacea_b200/) never imports it.

Pinned (not "parity unpinned"): tests/test_oracle_golden.py checks this port against golden tensors produced
by the unmodified reference modules imported in the build container (oracle/make_golden.py, fixtures under
tests/golden/), and tests/test_oracle_vs_reference.py checks its state-dict key set and zero-init tails against
the reference's. The reference itself ships no tests or golden vectors (SURVEY.md section 4).

It is a functional restatement, not a copy: there is no nn.Module tree, weights are looked up in a flat
state dict by the reference's key names, the topology is derived once from the config, and the view height
is passed explicitly (the reference infers it with sqrt(N/12), attention.py:428,537, which only works for
2:1 views). Each function cites the reference lines it follows (paths relative to sgm/modules/).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional

import torch
import torch.nn.functional as F

# reference quirk (attention.py:545-559): view i attends {i-1, i+1}; view 0 attends {5, 1}; the wrap branch
# for the last view is dead code and the out-of-range slice is empty, so view 5 attends {4} only.
CROSS_VIEW_NEIGHBOURS = ((5, 1), (0, 2), (1, 3), (2, 4), (3, 5), (4,))


@dataclass
class NetConfig:
    """configs/inference_nuscenes.yaml:32-50 (UNet) / :53-71 (ControlNet) keyword arguments."""
    in_channels: int = 8
    out_channels: int = 4
    model_channels: int = 320
    attention_resolutions: tuple = (4, 2, 1)
    num_res_blocks: int = 2
    channel_mult: tuple = (1, 2, 4, 4)
    num_head_channels: int = 64
    context_dim: int = 1024
    num_frames: int = 8
    hint_channels: int = 19
    control_scales: float = 1.0
    num_views: int = 6

    @staticmethod
    def from_kwargs(kw: dict, hint_channels: int = 19) -> "NetConfig":
        return NetConfig(
            in_channels=kw["in_channels"], out_channels=kw.get("out_channels", 4),
            model_channels=kw["model_channels"], attention_resolutions=tuple(kw["attention_resolutions"]),
            num_res_blocks=kw["num_res_blocks"], channel_mult=tuple(kw["channel_mult"]),
            num_head_channels=kw["num_head_channels"], context_dim=kw["context_dim"],
            num_frames=kw["num_frames"], hint_channels=hint_channels)


@dataclass
class Layer:
    kind: str          # "conv" | "res" | "stt" | "down" | "up"
    key: str           # state-dict prefix, e.g. "input_blocks.1.0"
    cin: int = 0
    cout: int = 0
    heads: int = 0


@dataclass
class Topology:
    input_blocks: list = field(default_factory=list)   # list[list[Layer]]
    middle: list = field(default_factory=list)
    output_blocks: list = field(default_factory=list)
    input_chans: list = field(default_factory=list)    # channels of every encoder output (skip widths)


def build_topology(cfg: NetConfig, with_decoder: bool = True) -> Topology:
    """openaimodel.py:961-1251 (UNetModel3D.__init__): resblock_updown=False, transformer_depth=1, legacy=False."""
    t = Topology()
    mc = cfg.model_channels
    t.input_blocks.append([Layer("conv", "input_blocks.0.0", cfg.in_channels, mc)])
    chans = [mc]
    ch, ds = mc, 1
    idx = 1
    for level, mult in enumerate(cfg.channel_mult):
        for _ in range(cfg.num_res_blocks):
            layers = [Layer("res", f"input_blocks.{idx}.0", ch, mult * mc)]
            ch = mult * mc
            if ds in cfg.attention_resolutions:
                layers.append(Layer("stt", f"input_blocks.{idx}.1", ch, ch, ch // cfg.num_head_channels))
            t.input_blocks.append(layers)
            chans.append(ch)
            idx += 1
        if level != len(cfg.channel_mult) - 1:
            t.input_blocks.append([Layer("down", f"input_blocks.{idx}.0", ch, ch)])
            chans.append(ch)
            idx += 1
            ds *= 2
    t.input_chans = list(chans)
    t.middle = [Layer("res", "middle_block.0", ch, ch),
                Layer("stt", "middle_block.1", ch, ch, ch // cfg.num_head_channels),
                Layer("res", "middle_block.2", ch, ch)]
    if with_decoder:
        idx = 0
        for level, mult in list(enumerate(cfg.channel_mult))[::-1]:
            for i in range(cfg.num_res_blocks + 1):
                ich = chans.pop()
                layers = [Layer("res", f"output_blocks.{idx}.0", ch + ich, mc * mult)]
                ch = mc * mult
                if ds in cfg.attention_resolutions:
                    layers.append(Layer("stt", f"output_blocks.{idx}.1", ch, ch, ch // cfg.num_head_channels))
                if level and i == cfg.num_res_blocks:
                    layers.append(Layer("up", f"output_blocks.{idx}.{len(layers)}", ch, ch))
                    ds //= 2
                t.output_blocks.append(layers)
                idx += 1
    return t


# ------------------------------------------------------------------------------------------------
# leaf ops
# ------------------------------------------------------------------------------------------------
def timestep_embedding(timesteps: torch.Tensor, dim: int, max_period: float = 10000.0) -> torch.Tensor:
    """diffusionmodules/util.py:224-248: [cos(t f), sin(t f)], f_k = exp(-ln(1e4) k / half)."""
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32) / half)
    args = timesteps[:, None].float() * freqs[None]
    emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
    if dim % 2:
        emb = torch.cat([emb, torch.zeros_like(emb[:, :1])], dim=-1)
    return emb


def temporal_pos_embedding(T: int, dim: int) -> torch.Tensor:
    """attention.py:1140-1159. The frequency vector is cast to int64 (:1148), so only frequency 0 survives:
    pe[t] = [sin t, cos t, 0, 1, 0, 1, ...]."""
    i = torch.arange(dim // 2, dtype=torch.float32) / (dim / 2)
    inv = (1.0 / torch.pow(torch.tensor(10000.0), i)).to(torch.long)
    out = torch.arange(T, dtype=torch.long)[:, None] * inv[None, :]
    pe = torch.zeros(T, dim)
    pe[:, 0::2] = torch.sin(out)
    pe[:, 1::2] = torch.cos(out)
    return pe


def _lin(sd, key, x):
    return F.linear(x, sd[key + ".weight"], sd.get(key + ".bias"))


def _mha(q, k, v, heads):
    """softmax(q k^T / sqrt(d)) v with heads split from the channel dim; q [B,Nq,C], k/v [B,Nk,C]."""
    B, Nq, Cc = q.shape
    d = Cc // heads
    qh = q.reshape(B, Nq, heads, d).transpose(1, 2)
    kh = k.reshape(B, k.shape[1], heads, d).transpose(1, 2)
    vh = v.reshape(B, v.shape[1], heads, d).transpose(1, 2)
    o = F.scaled_dot_product_attention(qh, kh, vh)
    return o.transpose(1, 2).reshape(B, Nq, Cc)


def view_attention(sd, key, x, heads, H, V, cross: bool):
    """attention.py:407-489 (intra-view) / :518-610 (cross-view). x: [B, H*V*w, C] tokens in (y, view, x) order."""
    B, N, Cc = x.shape
    assert V == 6, "the reference hard-codes six views (attention.py:436,545)"
    w = N // (H * V)
    q = _lin(sd, key + ".to_q", x).reshape(B, H, V, w, Cc)
    k = _lin(sd, key + ".to_k", x).reshape(B, H, V, w, Cc)
    v = _lin(sd, key + ".to_v", x).reshape(B, H, V, w, Cc)
    out = torch.empty_like(q)
    for i in range(V):
        qi = q[:, :, i].reshape(B, H * w, Cc)
        if cross:
            nb = CROSS_VIEW_NEIGHBOURS[i]
            # the reference concatenates neighbour views along width, then flattens (h, w_cat)
            ki = torch.cat([k[:, :, j] for j in nb], dim=2).reshape(B, H * w * len(nb), Cc)
            vi = torch.cat([v[:, :, j] for j in nb], dim=2).reshape(B, H * w * len(nb), Cc)
        else:
            ki = k[:, :, i].reshape(B, H * w, Cc)
            vi = v[:, :, i].reshape(B, H * w, Cc)
        out[:, :, i] = _mha(qi, ki, vi, heads).reshape(B, H, w, Cc)
    return _lin(sd, key + ".to_out.0", out.reshape(B, N, Cc))


def cross_attention(sd, key, x, context, heads):
    """attention.py:229-291 CrossAttention: self-attention when context is None."""
    ctx = x if context is None else context
    q = _lin(sd, key + ".to_q", x)
    k = _lin(sd, key + ".to_k", ctx)
    v = _lin(sd, key + ".to_v", ctx)
    return _lin(sd, key + ".to_out.0", _mha(q, k, v, heads))


def feed_forward(sd, key, x):
    """attention.py:91-117: Linear(C, 8C) -> value * gelu_erf(gate) -> Linear(4C, C)."""
    h = _lin(sd, key + ".net.0.proj", x)
    a, g = h.chunk(2, dim=-1)
    return _lin(sd, key + ".net.2", a * F.gelu(g))


def _ln(sd, key, x):
    return F.layer_norm(x, (x.shape[-1],), sd[key + ".weight"], sd[key + ".bias"], 1e-5)


def basic_transformer_block(sd, key, x, context, heads, mode, H=0, V=0):
    """attention.py:726-747. mode: "intra" | "cross" | "temporal"."""
    h = _ln(sd, key + ".norm1", x)
    if mode == "temporal":
        x = cross_attention(sd, key + ".attn1", h, None, heads) + x
    else:
        x = view_attention(sd, key + ".attn1", h, heads, H, V, cross=(mode == "cross")) + x
    x = cross_attention(sd, key + ".attn2", _ln(sd, key + ".norm2", x), context, heads) + x
    x = feed_forward(sd, key + ".ff", _ln(sd, key + ".norm3", x)) + x
    return x


def _gn(sd, key, x, eps):
    return F.group_norm(x, 32, sd[key + ".weight"], sd[key + ".bias"], eps)


def spatial_temporal_transformer(sd, key, x, context, heads, T, V):
    """attention.py:1064-1134 with use_linear=True, insert_crossview=True.
    x: [(b t), C, H, W]; context: [(b t), 77, Cctx]."""
    BT, Cc, H, W = x.shape
    b = BT // T

    def tokens(z):
        return z.permute(0, 2, 3, 1).reshape(BT, H * W, Cc)

    def image(z):
        return z.reshape(BT, H, W, Cc).permute(0, 3, 1, 2)

    # (1) intra-view  :1068-1085
    h = _lin(sd, key + ".proj_in", tokens(_gn(sd, key + ".norm", x, 1e-6)))
    h = basic_transformer_block(sd, key + ".transformer_blocks.0", h, context, heads, "intra", H, V)
    x = image(_lin(sd, key + ".proj_out", h)) + x
    # (2) cross-view  :1087-1104
    h = _lin(sd, key + ".proj_in_crossview", tokens(_gn(sd, key + ".norm_crossview", x, 1e-6)))
    h = basic_transformer_block(sd, key + ".transformer_blocks_crossview.0", h, context, heads, "cross", H, V)
    x = image(_lin(sd, key + ".proj_out_crossview", h)) + x
    # (3) temporal  :1107-1134; tokens regrouped to ((b h w), t, c); text context of frame 0 of each b
    h = _lin(sd, key + ".proj_in_temporal", tokens(_gn(sd, key + ".norm_temporal", x, 1e-6)))
    h = h.reshape(b, T, H * W, Cc).permute(0, 2, 1, 3).reshape(b * H * W, T, Cc)
    h = h + temporal_pos_embedding(T, Cc).to(h)
    ctx = context.reshape(b, T, *context.shape[1:])[:, 0]                       # [b, 77, Cctx]
    ctx = ctx[:, None].expand(b, H * W, *ctx.shape[1:]).reshape(b * H * W, *ctx.shape[1:])
    h = basic_transformer_block(sd, key + ".transformer_blocks_temporal.0", h, ctx, heads, "temporal")
    h = h.reshape(b, H * W, T, Cc).permute(0, 2, 1, 3).reshape(BT, H * W, Cc)
    return x + image(_lin(sd, key + ".proj_out_temporal", h))


def _temporal_branch(sd, key, h, T):
    """openaimodel.py:509-515 / :534-539: GroupNorm over (C/32, T) per pixel, SiLU, Conv1d(k=3,pad=1) over frames."""
    BT, Cc, H, W = h.shape
    b = BT // T
    z = h.reshape(b, T, Cc, H, W).permute(0, 3, 4, 2, 1).reshape(b * H * W, Cc, T)
    z = F.silu(_gn(sd, key + ".0", z, 1e-5))
    conv_key = key + (".2" if (key + ".2.weight") in sd else ".3")
    z = F.conv1d(z, sd[conv_key + ".weight"], sd[conv_key + ".bias"], padding=1)
    return z.reshape(b, H, W, Cc, T).permute(0, 4, 3, 1, 2).reshape(BT, Cc, H, W)


def res_block_3d(sd, key, x, emb, T):
    """openaimodel.py:499-542 (no up/down, no scale-shift norm, dropout 0)."""
    h = F.conv2d(F.silu(_gn(sd, key + ".in_layers.0", x, 1e-5)), sd[key + ".in_layers.2.weight"],
                 sd[key + ".in_layers.2.bias"], padding=1)
    h = h + _temporal_branch(sd, key + ".in_layers_temporal", h, T)
    h = h + _lin(sd, key + ".emb_layers.1", F.silu(emb))[:, :, None, None]
    h = F.conv2d(F.silu(_gn(sd, key + ".out_layers.0", h, 1e-5)), sd[key + ".out_layers.3.weight"],
                 sd[key + ".out_layers.3.bias"], padding=1)
    h = h + _temporal_branch(sd, key + ".out_layers_temporal", h, T)
    if (key + ".skip_connection.weight") in sd:
        x = F.conv2d(x, sd[key + ".skip_connection.weight"], sd[key + ".skip_connection.bias"])
    return x + h


def run_layers(sd, prefix, layers, h, emb, context, cfg: NetConfig):
    """openaimodel.py:85-103 TimestepEmbedSequential dispatch."""
    for L in layers:
        key = prefix + L.key
        if L.kind == "conv":
            h = F.conv2d(h, sd[key + ".weight"], sd[key + ".bias"], padding=1)
        elif L.kind == "res":
            h = res_block_3d(sd, key, h, emb, cfg.num_frames)
        elif L.kind == "stt":
            h = spatial_temporal_transformer(sd, key, h, context, L.heads, cfg.num_frames, cfg.num_views)
        elif L.kind == "down":   # openaimodel.py:161-201 Downsample: conv3x3 stride 2 pad 1
            h = F.conv2d(h, sd[key + ".op.weight"], sd[key + ".op.bias"], stride=2, padding=1)
        elif L.kind == "up":     # openaimodel.py:106-142 Upsample: nearest x2 then conv3x3
            h = F.interpolate(h, scale_factor=2, mode="nearest")
            h = F.conv2d(h, sd[key + ".conv.weight"], sd[key + ".conv.bias"], padding=1)
        else:
            raise ValueError(L.kind)
    return h


def time_embed(sd, prefix, timesteps, cfg: NetConfig):
    """openaimodel.py:936-943: Linear(mc, 4mc) -> SiLU -> Linear(4mc, 4mc)."""
    e = timestep_embedding(timesteps, cfg.model_channels)
    e = _lin(sd, prefix + "time_embed.0", e)
    return _lin(sd, prefix + "time_embed.2", F.silu(e))


HINT_STRIDES = (1, 1, 2, 1, 2, 1, 2, 1)   # controlmodel.py:43-59


def hint_stem(sd, prefix, hint):
    """controlmodel.py:43-59,118: 8 convs (indices 0,2,...,14) with SiLU between, no activation after the last."""
    h = hint
    for i, s in enumerate(HINT_STRIDES):
        k = f"{prefix}input_hint_block.{2 * i}"
        h = F.conv2d(h, sd[k + ".weight"], sd[k + ".bias"], stride=s, padding=1)
        if i != len(HINT_STRIDES) - 1:
            h = F.silu(h)
    return h


def controlnet_forward(sd, prefix, cfg: NetConfig, x, hint, timesteps, context):
    """controlmodel.py:86-142. Returns the 13 control residuals (encoder outputs + middle), zero-conv'd."""
    topo = build_topology(cfg, with_decoder=False)
    emb = time_embed(sd, prefix, timesteps, cfg)
    guided = hint_stem(sd, prefix, hint)
    T = cfg.num_frames
    ctx = context[:, None].expand(-1, T, -1, -1).reshape(-1, *context.shape[1:])   # :121-122
    outs = []
    h = x
    for i, layers in enumerate(topo.input_blocks):
        h = run_layers(sd, prefix, layers, h, emb, ctx, cfg)
        if i == 0:
            h = h + guided                                                            # :126-129
        zk = f"{prefix}zero_convs.{i}.0"
        outs.append(F.conv2d(h, sd[zk + ".weight"], sd[zk + ".bias"]) * cfg.control_scales)
    h = run_layers(sd, prefix, topo.middle, h, emb, ctx, cfg)
    mk = f"{prefix}middle_block_out.0"
    outs.append(F.conv2d(h, sd[mk + ".weight"], sd[mk + ".bias"]) * cfg.control_scales)
    return outs


def unet_forward(sd, prefix, cfg: NetConfig, x, timesteps, context, control: Optional[list]):
    """controlmodel.py:160-202."""
    topo = build_topology(cfg, with_decoder=True)
    emb = time_embed(sd, prefix, timesteps, cfg)
    T = cfg.num_frames
    ctx = context[:, None].expand(-1, T, -1, -1).reshape(-1, *context.shape[1:])
    control = None if control is None else list(control)
    hs = []
    h = x
    for layers in topo.input_blocks:
        h = run_layers(sd, prefix, layers, h, emb, ctx, cfg)
        hs.append(h)
    h = run_layers(sd, prefix, topo.middle, h, emb, ctx, cfg)
    if control is not None:
        h = h + control.pop()
    for layers in topo.output_blocks:
        skip = hs.pop()
        if control is not None:
            skip = skip + control.pop()
        h = run_layers(sd, prefix, layers, torch.cat([h, skip], dim=1), emb, ctx, cfg)
    h = F.silu(_gn(sd, prefix + "out.0", h, 1e-5))
    return F.conv2d(h, sd[prefix + "out.2.weight"], sd[prefix + "out.2.bias"], padding=1)


@torch.no_grad()
def wrapper_forward(sd, cfg: NetConfig, x, t, c: dict, prefix: str = "diffusion_model."):
    """wrappers.py:37-70 OpenAIWrapperControlLDM3D.forward: eps = UNet(cat(x, concat), control=ControlNet(...))."""
    if "concat" in c and c["concat"] is not None:
        x = torch.cat([x, c["concat"]], dim=1)
    x = x.float()
    ctx = c["crossattn"].float()
    control = controlnet_forward(sd, prefix + "controlnet.", cfg, x, c["cond_feat"].float(), t, ctx)
    return unet_forward(sd, prefix, cfg, x, t, ctx, control)


# ------------------------------------------------------------------------------------------------
# state-dict specification and seeded weights (shared by the golden generator and the GPU parity tests)
# ------------------------------------------------------------------------------------------------
def _res_spec(spec, key, cin, cout, emb_ch):
    spec[key + ".in_layers.0.weight"] = (cin,); spec[key + ".in_layers.0.bias"] = (cin,)
    spec[key + ".in_layers.2.weight"] = (cout, cin, 3, 3); spec[key + ".in_layers.2.bias"] = (cout,)
    spec[key + ".in_layers_temporal.0.weight"] = (cout,); spec[key + ".in_layers_temporal.0.bias"] = (cout,)
    spec[key + ".in_layers_temporal.2.weight"] = (cout, cout, 3); spec[key + ".in_layers_temporal.2.bias"] = (cout,)
    spec[key + ".emb_layers.1.weight"] = (cout, emb_ch); spec[key + ".emb_layers.1.bias"] = (cout,)
    spec[key + ".out_layers.0.weight"] = (cout,); spec[key + ".out_layers.0.bias"] = (cout,)
    spec[key + ".out_layers.3.weight"] = (cout, cout, 3, 3); spec[key + ".out_layers.3.bias"] = (cout,)
    spec[key + ".out_layers_temporal.0.weight"] = (cout,); spec[key + ".out_layers_temporal.0.bias"] = (cout,)
    spec[key + ".out_layers_temporal.3.weight"] = (cout, cout, 3); spec[key + ".out_layers_temporal.3.bias"] = (cout,)
    if cin != cout:
        spec[key + ".skip_connection.weight"] = (cout, cin, 1, 1); spec[key + ".skip_connection.bias"] = (cout,)


def _btb_spec(spec, key, c, ctx):
    for a, kdim in (("attn1", c), ("attn2", ctx)):
        spec[f"{key}.{a}.to_q.weight"] = (c, c)
        spec[f"{key}.{a}.to_k.weight"] = (c, kdim)
        spec[f"{key}.{a}.to_v.weight"] = (c, kdim)
        spec[f"{key}.{a}.to_out.0.weight"] = (c, c); spec[f"{key}.{a}.to_out.0.bias"] = (c,)
    spec[key + ".ff.net.0.proj.weight"] = (8 * c, c); spec[key + ".ff.net.0.proj.bias"] = (8 * c,)
    spec[key + ".ff.net.2.weight"] = (c, 4 * c); spec[key + ".ff.net.2.bias"] = (c,)
    for n in ("norm1", "norm2", "norm3"):
        spec[f"{key}.{n}.weight"] = (c,); spec[f"{key}.{n}.bias"] = (c,)


def _stt_spec(spec, key, c, ctx):
    for sfx in ("", "_temporal", "_crossview"):
        spec[f"{key}.norm{sfx}.weight"] = (c,); spec[f"{key}.norm{sfx}.bias"] = (c,)
        spec[f"{key}.proj_in{sfx}.weight"] = (c, c); spec[f"{key}.proj_in{sfx}.bias"] = (c,)
        spec[f"{key}.proj_out{sfx}.weight"] = (c, c); spec[f"{key}.proj_out{sfx}.bias"] = (c,)
        _btb_spec(spec, f"{key}.transformer_blocks{sfx}.0", c, ctx)


def _net_spec(spec, prefix, cfg: NetConfig, with_decoder: bool):
    mc = cfg.model_channels
    emb = 4 * mc
    spec[prefix + "time_embed.0.weight"] = (emb, mc); spec[prefix + "time_embed.0.bias"] = (emb,)
    spec[prefix + "time_embed.2.weight"] = (emb, emb); spec[prefix + "time_embed.2.bias"] = (emb,)
    topo = build_topology(cfg, with_decoder)
    for layers in topo.input_blocks + [topo.middle] + topo.output_blocks:
        for L in layers:
            key = prefix + L.key
            if L.kind == "conv":
                spec[key + ".weight"] = (L.cout, L.cin, 3, 3); spec[key + ".bias"] = (L.cout,)
            elif L.kind == "res":
                _res_spec(spec, key, L.cin, L.cout, emb)
            elif L.kind == "stt":
                _stt_spec(spec, key, L.cin, cfg.context_dim)
            elif L.kind == "down":
                spec[key + ".op.weight"] = (L.cout, L.cin, 3, 3); spec[key + ".op.bias"] = (L.cout,)
            elif L.kind == "up":
                spec[key + ".conv.weight"] = (L.cout, L.cin, 3, 3); spec[key + ".conv.bias"] = (L.cout,)
    return topo


def state_spec(cfg: NetConfig, prefix: str = "diffusion_model.") -> dict:
    """key -> shape of every tensor in the reference wrapper's state_dict (2,478 tensors for the YAML config)."""
    spec: dict = {}
    _net_spec(spec, prefix, cfg, True)
    mc = cfg.model_channels
    spec[prefix + "out.0.weight"] = (mc,); spec[prefix + "out.0.bias"] = (mc,)
    spec[prefix + "out.2.weight"] = (cfg.out_channels, mc, 3, 3); spec[prefix + "out.2.bias"] = (cfg.out_channels,)
    cp = prefix + "controlnet."
    topo = _net_spec(spec, cp, cfg, False)
    chs = [cfg.hint_channels, 16, 16, 32, 32, 96, 96, 256, mc]
    for i in range(8):
        spec[f"{cp}input_hint_block.{2 * i}.weight"] = (chs[i + 1], chs[i], 3, 3)
        spec[f"{cp}input_hint_block.{2 * i}.bias"] = (chs[i + 1],)
    for i, ch in enumerate(topo.input_chans):
        spec[f"{cp}zero_convs.{i}.0.weight"] = (ch, ch, 1, 1); spec[f"{cp}zero_convs.{i}.0.bias"] = (ch,)
    ch = topo.input_chans[-1]
    spec[cp + "middle_block_out.0.weight"] = (ch, ch, 1, 1); spec[cp + "middle_block_out.0.bias"] = (ch,)
    return spec


def seeded_state_dict(spec: dict, seed: int = 0, gain: float = 0.7) -> dict:
    """Deterministic non-degenerate weights. The reference zero-initialises every block's last layer
    (openaimodel.py:418,454-476,1251; attention.py:1040-1059; controlmodel.py:58,82-84), which makes a
    freshly built model output exactly 0 — useless for parity — so EVERY tensor is re-drawn here:
    matrices/kernels ~ N(0, gain^2 / fan_in), norm scales ~ 1 + 0.1 N(0,1), biases ~ 0.05 N(0,1).
    Keys are visited in sorted order with one CPU generator, so any holder of the same spec gets the
    same weights on any machine."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd = {}
    for key in sorted(spec):
        shape = tuple(spec[key])
        if key.endswith(".bias"):
            sd[key] = 0.05 * torch.randn(shape, generator=g)
        elif len(shape) == 1:
            sd[key] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            fan_in = 1
            for s in shape[1:]:
                fan_in *= s
            sd[key] = torch.randn(shape, generator=g) * (gain / math.sqrt(fan_in))
    return sd
