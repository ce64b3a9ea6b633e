"""Windowed relative-position self-attention encoder -- PyTorch mirror of the reference's
`modules/rel_transformer.py` (RelativeEncoder :257-320, MultiHeadAttention :103-254, FFN :323-345,
LayerNorm :24-42, SinusoidalPositionalEmbedding :45-100).

These modules are the prior network that runs before `z_p` (SURVEY.md 8f rows f1/f2).  On a CUDA device
`RelativeEncoder.forward` is one call into the native library (fp32 kernels, or tcgen05 kernels in bf16 mode, for
utterances of any length), so the prior network runs on the GPU with the hot path.  The PyTorch formulation here is
the readable statement of that arithmetic and the CPU path.  It is written from the reference's behaviour, with the
reference's parameter names and shapes (so checkpoints load), but in its own formulation: the relative-position
logits/values are moved between "relative" and "absolute" indexing with diagonal views instead of the pad-and-reshape
trick.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F


class LayerNorm(nn.Module):
    """Channel layer-norm over dim 1 of [B, C, T], eps 1e-4, parameters `gamma` / `beta` (reference :24-42)."""

    def __init__(self, channels, eps=1e-4):
        super().__init__()
        self.channels, self.eps = channels, eps
        self.gamma = nn.Parameter(torch.ones(channels))
        self.beta = nn.Parameter(torch.zeros(channels))

    def forward(self, x):
        return F.layer_norm(x.transpose(1, -1), (self.channels,), self.gamma, self.beta, self.eps).transpose(1, -1)


class SinusoidalPositionalEmbedding(nn.Module):
    """tensor2tensor-style sinusoidal table indexed by the running count of non-padding entries (reference :45-100).
    Keeps the reference's `_float_tensor` buffer so state-dicts match."""

    def __init__(self, embedding_dim, padding_idx, init_size=1024):
        super().__init__()
        self.embedding_dim, self.padding_idx = embedding_dim, padding_idx
        self.weights = self.get_embedding(init_size, embedding_dim, padding_idx)
        self.register_buffer("_float_tensor", torch.FloatTensor(1))

    @staticmethod
    def get_embedding(num_embeddings, embedding_dim, padding_idx=None):
        half = embedding_dim // 2
        freq = torch.exp(torch.arange(half, dtype=torch.float) * -(math.log(10000) / (half - 1)))
        ang = torch.arange(num_embeddings, dtype=torch.float)[:, None] * freq[None, :]
        table = torch.cat([ang.sin(), ang.cos()], dim=1)
        if embedding_dim % 2 == 1:
            table = torch.cat([table, torch.zeros(num_embeddings, 1)], dim=1)
        if padding_idx is not None:
            table[padding_idx] = 0
        return table

    def table(self, n_rows, device):
        """The sinusoidal table with at least n_rows rows on `device` (row padding_idx is zero): what the native length
        regulator indexes with the frame positions it computes itself."""
        if self.weights is None or n_rows > self.weights.size(0):
            self.weights = self.get_embedding(n_rows, self.embedding_dim, self.padding_idx)
        if self.weights.device != torch.device(device) or self.weights.dtype != torch.float32:
            self.weights = self.weights.to(device=device, dtype=torch.float32)
        return self.weights

    def forward(self, bsz, seq_len, input):
        """`input` [B, T]: entries equal to padding_idx are padding.  Returns [bsz, seq_len, -1] exactly as the reference
        does (a `.view`, which only equals [B, T, dim] when seq_len == T -- reference encoder.py:51 relies on that)."""
        need = self.padding_idx + 1 + seq_len
        if self.weights is None or need > self.weights.size(0) or input.shape[1] + self.padding_idx + 1 > self.weights.size(0):
            self.weights = self.get_embedding(max(need, input.shape[1] + self.padding_idx + 1), self.embedding_dim,
                                              self.padding_idx)
        self.weights = self.weights.to(self._float_tensor)
        keep = input.ne(self.padding_idx).int()
        positions = (torch.cumsum(keep, dim=1).type_as(keep) * keep).long() + self.padding_idx
        return self.weights.index_select(0, positions.reshape(-1)).view(bsz, seq_len, -1).detach()


class MultiHeadAttention(nn.Module):
    """Self-attention with learned relative-position key/value embeddings inside a +-window (reference :103-254).
    Outside the window the relative logit is 0 (not -inf): attention stays global."""

    def __init__(self, channels, out_channels, n_heads, window_size=None, heads_share=True, p_dropout=0.0,
                 block_length=None, proximal_bias=False, proximal_init=False):
        super().__init__()
        assert channels % n_heads == 0
        if block_length is not None or proximal_bias:
            raise NotImplementedError("block_length / proximal_bias are never used by VISinger")
        self.channels, self.out_channels, self.n_heads = channels, out_channels, n_heads
        self.window_size, self.heads_share = window_size, heads_share
        self.k_channels = channels // n_heads
        self.conv_q = nn.Conv1d(channels, channels, 1)
        self.conv_k = nn.Conv1d(channels, channels, 1)
        self.conv_v = nn.Conv1d(channels, channels, 1)
        if window_size is not None:
            n_rel = 1 if heads_share else n_heads
            std = self.k_channels ** -0.5
            self.emb_rel_k = nn.Parameter(torch.randn(n_rel, window_size * 2 + 1, self.k_channels) * std)
            self.emb_rel_v = nn.Parameter(torch.randn(n_rel, window_size * 2 + 1, self.k_channels) * std)
        self.conv_o = nn.Conv1d(channels, out_channels, 1)
        nn.init.xavier_uniform_(self.conv_q.weight)
        nn.init.xavier_uniform_(self.conv_k.weight)
        if proximal_init:
            self.conv_k.weight.data.copy_(self.conv_q.weight.data)
            self.conv_k.bias.data.copy_(self.conv_q.bias.data)
        nn.init.xavier_uniform_(self.conv_v.weight)

    def forward(self, x, c, attn_mask=None):
        B, _, T = x.shape
        h, d = self.n_heads, self.k_channels
        q = self.conv_q(x).view(B, h, d, T).transpose(2, 3)            # [B, h, T, d]
        k = self.conv_k(c).view(B, h, d, -1).transpose(2, 3)
        v = self.conv_v(c).view(B, h, d, -1).transpose(2, 3)
        scale = 1.0 / math.sqrt(d)
        scores = torch.matmul(q, k.transpose(-2, -1)) * scale           # [B, h, T, T]
        w = self.window_size
        if w is not None:
            assert k.shape[2] == T, "Relative attention is only available for self-attention."
            rel = torch.matmul(q, self.emb_rel_k.unsqueeze(0).transpose(-2, -1)) * scale   # [B, h, T, 2w+1]
            for r in range(2 * w + 1):                                   # relative offset o = r - w on diagonal o
                o = r - w
                n = T - abs(o)
                if n <= 0:
                    continue
                i0 = max(0, -o)
                scores.diagonal(offset=o, dim1=-2, dim2=-1).add_(rel[:, :, i0:i0 + n, r])
        if attn_mask is not None:
            scores = scores.masked_fill(attn_mask == 0, -1e4)
        p = F.softmax(scores, dim=-1)
        out = torch.matmul(p, v)                                         # [B, h, T, d]
        if w is not None:
            p_rel = p.new_zeros(B, h, T, 2 * w + 1)
            for r in range(2 * w + 1):
                o = r - w
                n = T - abs(o)
                if n <= 0:
                    continue
                i0 = max(0, -o)
                p_rel[:, :, i0:i0 + n, r] = p.diagonal(offset=o, dim1=-2, dim2=-1)
            out = out + torch.matmul(p_rel, self.emb_rel_v.unsqueeze(0))
        out = out.transpose(2, 3).contiguous().view(B, h * d, T)
        return self.conv_o(out)


class FFN(nn.Module):
    """conv(k) -> ReLU -> conv(1), both on masked input (reference :323-345; `activation` is never passed => ReLU)."""

    def __init__(self, in_channels, out_channels, filter_channels, kernel_size, p_dropout=0.0, activation=None):
        super().__init__()
        self.activation = activation
        self.conv_1 = nn.Conv1d(in_channels, filter_channels, kernel_size, padding=kernel_size // 2)
        self.conv_2 = nn.Conv1d(filter_channels, out_channels, 1)

    def forward(self, x, x_mask):
        x = self.conv_1(x * x_mask)
        x = x * torch.sigmoid(1.702 * x) if self.activation == "gelu" else torch.relu(x)
        return self.conv_2(x * x_mask)


class RelativeEncoder(nn.Module):
    """Post-LN transformer encoder over [B, C, T] with an optional condition `g` (reference :257-320).

    On a CUDA device `forward` is ONE call into the native library (`vsg_relenc_forward`: fused QKV projection, windowed
    relative-position attention kernel, fused residual + channel-LayerNorm + condition + mask, FFN on the convolution
    kernels; SURVEY.md section 8 row f1).  The PyTorch formulation below (`forward_torch`) is kept as the readable
    statement of the same arithmetic and for CPU-side tooling; set `native = False` to force it."""

    native = True
    precision = "fp32"

    def __init__(self, hidden_channels, filter_channels, n_heads, n_layers, kernel_size=1, p_dropout=0.0, window_size=4,
                 block_length=None, pre_ln=False, gin_channels=None, **kwargs):
        super().__init__()
        self.hidden_channels, self.n_layers, self.pre_ln = hidden_channels, n_layers, pre_ln
        self.filter_channels, self.n_heads, self.kernel_size = filter_channels, n_heads, kernel_size
        self.window_size, self.block_length, self.gin_channels = window_size, block_length, gin_channels
        self.attn_layers = nn.ModuleList()
        self.norm_layers_1 = nn.ModuleList()
        self.ffn_layers = nn.ModuleList()
        self.norm_layers_2 = nn.ModuleList()
        for _ in range(n_layers):
            self.attn_layers.append(MultiHeadAttention(hidden_channels, hidden_channels, n_heads, window_size=window_size,
                                                       p_dropout=p_dropout, block_length=block_length))
            self.norm_layers_1.append(LayerNorm(hidden_channels))
            self.ffn_layers.append(FFN(hidden_channels, hidden_channels, filter_channels, kernel_size, p_dropout=p_dropout))
            self.norm_layers_2.append(LayerNorm(hidden_channels))
        if pre_ln:
            self.last_ln = LayerNorm(hidden_channels)
        if gin_channels is not None:
            self.pre_net = nn.Conv1d(gin_channels, hidden_channels, 1)
        self._vsg_pack = None
        self._vsg_key = None

    # -- native path -----------------------------------------------------------------------------
    def _native_supported(self):
        return not self.pre_ln and self.block_length is None and self.window_size is not None and self.kernel_size % 2 == 1

    def _pack(self):
        from .. import _lib
        params = list(self.parameters())
        dev = params[0].device
        key = (str(dev),) + tuple((p.data_ptr(), p._version) for p in params)
        if self._vsg_pack is None or self._vsg_key != key:
            c = _lib.VsgRelEncConfig(self.hidden_channels, self.filter_channels, self.n_heads, self.n_layers, self.kernel_size,
                                     self.window_size, self.gin_channels or 0)
            self._vsg_pack = _lib.RelEncPack(c, dict(self.state_dict()), "", dev)
            self._vsg_key = key
        return self._vsg_pack

    @torch.no_grad()
    def forward_native(self, x, x_mask, g=None):
        from .. import _lib
        if x.dim() != 3 or x.shape[1] != self.hidden_channels:
            raise RuntimeError(f"expected x of shape [B, {self.hidden_channels}, T], got {tuple(x.shape)}")
        B, _, T = x.shape
        if x_mask.numel() != B * T:
            raise RuntimeError(f"expected x_mask of shape [B, 1, T] = [{B}, 1, {T}], got {tuple(x_mask.shape)}")
        g_t = 0
        if g is not None:
            if self.gin_channels is None:
                raise RuntimeError("this encoder was built without gin_channels; g must be None")
            if g.dim() != 3 or g.shape[0] != B or g.shape[1] != self.gin_channels or g.shape[2] not in (1, T):
                raise RuntimeError(f"expected g of shape [B, {self.gin_channels}, 1 or T], got {tuple(g.shape)}")
            g_t = 1 if (g.shape[2] == T and T > 1) else 0
        pack = self._pack()
        prec = _lib.precision_code(self.precision)
        xc, mc = _lib.as_f32c(x), _lib.as_f32c(x_mask)
        gc = _lib.as_f32c(g) if g is not None else None
        y = torch.empty_like(xc)
        if B and T:
            with torch.cuda.device(x.device):
                ws = _lib.workspace(x.device, pack.workspace_bytes(B, T, g_t, prec))
                rc = _lib.lib().vsg_relenc_forward(pack.handle, xc.data_ptr(), mc.data_ptr(),
                                                   gc.data_ptr() if gc is not None else None, g_t, y.data_ptr(), B, T, prec,
                                                   ws.data_ptr(), ws.numel(), _lib.stream_ptr(x.device))
            _lib.check(rc, "vsg_relenc_forward")
        return y

    def forward(self, x, x_mask, g=None):
        if x.is_cuda and self.native and not self.training:
            if not self._native_supported():      # no silent fallback on the GPU: say what is missing
                raise RuntimeError("visinger_b200 RelativeEncoder: the native kernels implement post-LN (pre_ln=False), "
                                   "block_length=None, odd FFN kernel sizes; set `native = False` for the PyTorch statement")
            return self.forward_native(x, x_mask, g)
        return self.forward_torch(x, x_mask, g)

    # -- PyTorch statement of the same arithmetic --------------------------------------------------
    def forward_torch(self, x, x_mask, g=None):
        attn_mask = x_mask.unsqueeze(2) * x_mask.unsqueeze(-1)
        if g is not None:
            g = self.pre_net(g)
        for i in range(self.n_layers):
            if g is not None:
                x = x + g
            x = x * x_mask
            h = self.norm_layers_1[i](x) if self.pre_ln else x
            x = x + self.attn_layers[i](h, h, attn_mask)
            if not self.pre_ln:
                x = self.norm_layers_1[i](x)
            h = self.norm_layers_2[i](x) if self.pre_ln else x
            x = x + self.ffn_layers[i](h, x_mask)
            if not self.pre_ln:
                x = self.norm_layers_2[i](x)
        if self.pre_ln:
            x = self.last_ln(x)
        return x * x_mask
