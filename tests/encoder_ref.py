"""Float64 restatement of the voice-cloning encoder (DESIGN.md §4.6), the spec the device encoder is tested against.

Written the plain way, structurally unlike the CUDA path: convolutions are `F.conv1d(stride=...)` over channel-first [C, L] tensors, the
attention is a masked softmax over every key (computed in query blocks only to bound memory). It rounds where the engine rounds: conv
operands to f16, linear operands to bf16, q / k / v and the softmax probabilities to bf16; residual streams and accumulations stay wide.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

HOP = 1920
WINDOW = 250
ENC = "mimi.encoder.model."
ENC_TR = "mimi.encoder_transformer.transformer.layers."


def f16(x):
    return x.to(torch.float16).to(torch.float64)


def bf16(x):
    return x.to(torch.bfloat16).to(torch.float64)


def elu(x):
    return torch.where(x > 0, x, torch.expm1(x))


def gelu_ggml(x):
    """ggml's tanh GELU through f16 (input and output rounded to f16), as the engine's epilogue computes it."""
    xf = f16(x)
    return f16(0.5 * xf * (1.0 + torch.tanh(0.7978845608028654 * xf * (1.0 + 0.044715 * xf * xf))))


class EncoderRef:
    def __init__(self, weights: dict, device="cpu"):
        self.dev = torch.device(device)
        self.W = {k: torch.as_tensor(np.asarray(v), dtype=torch.float64, device=self.dev) for k, v in weights.items()
                  if k.startswith(("mimi.encoder", "mimi.downsample", "flow_lm.speaker_proj"))}
        i = np.arange(32, dtype=np.float32)
        self.freq = torch.as_tensor(np.exp(np.float32(-np.log(np.float32(10000.0))) * i / np.float32(32)).astype(np.float32), dtype=torch.float64, device=self.dev)

    def conv(self, x, name, stride=1):
        """Causal conv over x [C, L] (already rounded to f16): K - S zero samples of left padding, f16 weights."""
        w = f16(self.W[name + ".conv.weight"])
        b = self.W.get(name + ".conv.bias")
        k = w.shape[-1]
        return F.conv1d(F.pad(x[None], (k - stride, 0)), w, b, stride=stride)[0]

    def seanet(self, pcm):
        """pcm float [n] -> [16T, 512] (output of conv 11)."""
        x = torch.as_tensor(np.asarray(pcm, np.float32), dtype=torch.float64, device=self.dev)
        T = -(-len(x) // HOP)
        x = F.pad(x, (0, T * HOP - len(x)))[None]
        y = self.conv(f16(x), ENC + "0")
        for blk, conv, stride in ((1, 3, 4), (4, 6, 5), (7, 9, 6)):
            h = f16(elu(self.conv(f16(elu(y)), ENC + f"{blk}.block.1")))
            y = y + self.conv(h, ENC + f"{blk}.block.3")
            y = self.conv(f16(elu(y)), ENC + f"{conv}", stride)
        return self.conv(f16(elu(y)), ENC + "11").T.contiguous()

    @staticmethod
    def ln(x, w, b):
        mu = x.mean(-1, keepdim=True)
        var = ((x - mu) ** 2).mean(-1, keepdim=True)
        return bf16((x - mu) / torch.sqrt(var) * w + (0 if b is None else b))

    def rope(self, x):
        """Interleaved RoPE on pairs (2i, 2i+1) of every 64-wide head, angle = position * freq_mimi[i]."""
        R = x.shape[0]
        ang = torch.arange(R, dtype=torch.float64, device=self.dev)[:, None] * self.freq[None, :]
        c, s = torch.cos(ang)[:, None, :], torch.sin(ang)[:, None, :]
        xh = x.reshape(R, 8, 32, 2)
        re, im = xh[..., 0], xh[..., 1]
        return torch.stack([re * c - im * s, re * s + im * c], -1).reshape(R, 512)

    def attention(self, q, k, v, block=512, window=WINDOW):
        R = q.shape[0]
        qh, kh, vh = (t.reshape(R, 8, 64).transpose(0, 1) for t in (q, k, v))
        out = torch.empty(8, R, 64, dtype=torch.float64, device=self.dev)
        j = torch.arange(R, device=self.dev)
        for i0 in range(0, R, block):
            i = torch.arange(i0, min(R, i0 + block), device=self.dev)
            d = i[:, None] - j[None, :]
            s = (qh[:, i] @ kh.transpose(1, 2)) * 0.125
            s = s.masked_fill(~((d >= 0) & (d < window))[None], float("-inf"))
            p = torch.exp(s - s.amax(-1, keepdim=True))
            out[:, i] = (bf16(p) @ vh) / p.sum(-1, keepdim=True)
        return bf16(out.transpose(0, 1).reshape(R, 512))

    def transformer(self, x):
        W = self.W
        for l in range(2):
            p = ENC_TR + f"{l}."
            h = self.ln(x, W[p + "norm1.weight"], W.get(p + "norm1.bias"))
            qkv = h @ bf16(W[p + "self_attn.in_proj.weight"]).T
            q, k, v = qkv[:, :512], qkv[:, 512:1024], qkv[:, 1024:]
            a = self.attention(bf16(self.rope(q)), bf16(self.rope(k)), bf16(v))
            x = x + W[p + "layer_scale_1.scale"] * (a @ bf16(W[p + "self_attn.out_proj.weight"]).T)
            h = self.ln(x, W[p + "norm2.weight"], W.get(p + "norm2.bias"))
            g = bf16(gelu_ggml(h @ bf16(W[p + "linear1.weight"]).T))
            x = x + W[p + "layer_scale_2.scale"] * (g @ bf16(W[p + "linear2.weight"]).T)
        return x

    def downsample(self, x):
        """[16T, 512] -> [T, 512]: k32 s16, the 16 rows of causal padding replicate row 0."""
        xc = f16(x).T
        xc = torch.cat([xc[:, :1].expand(-1, 16), xc], 1)
        w = f16(self.W["mimi.downsample.conv.conv.weight"])
        return F.conv1d(xc[None], w, self.W.get("mimi.downsample.conv.conv.bias"), stride=16)[0].T.contiguous()

    def stages(self, pcm) -> dict:
        s = self.seanet(pcm)
        t = self.transformer(s)
        d = self.downsample(t)
        out = bf16(d) @ bf16(self.W["flow_lm.speaker_proj_weight"]).T
        return {"enc.seanet": s, "enc.transformer": t, "enc.downsample": d, "prompt": out}

    def embed(self, pcm) -> np.ndarray:
        return self.stages(pcm)["prompt"].cpu().numpy()


def strided_conv_reshape(x: np.ndarray, w: np.ndarray, b, r: int) -> np.ndarray:
    """The engine's formulation of a k = 2r, stride r causal conv: rows of r * C channels (one zero row-group in front), a 2-tap window
    over them against the weight laid out [co][tap][ci]. x [L][C] channel-last, w [co][ci][2r] -> [L / r][co]."""
    L, C = x.shape
    co = w.shape[0]
    g = np.concatenate([np.zeros((r, C)), x]).reshape(L // r + 1, r * C)
    win = np.concatenate([g[:-1], g[1:]], 1)                    # [L/r][2 r C]
    wk = w.transpose(0, 2, 1).reshape(co, 2 * r * C)
    return win @ wk.T + (0 if b is None else b)
