"""Whisper encoder/decoder on PyTorch + cuBLAS -- the part of the path that north_star
leaves on library GEMMs (SURVEY.md section 8 row a2).

`openai-whisper` is not installable offline, so the product carries its own module with
the published architecture and the published parameter names: a checkpoint's
`model_state_dict` (or the oracle's seeded random init) loads with `load_state_dict`.
Differences from the upstream module that matter for this path:

  * attention never materialises its maps (the reference's `disable_sdpa()` wraps the whole
    forward, timing.py:57-58, and pays for 24 x 144 MB of encoder maps nobody reads): on a GPU
    the encoder self-attention, the cross-attention output and the causal decoder self-attention
    run on the sm_100a kernel of csrc/enc_attn.cu, otherwise on `scaled_dot_product_attention`;
  * cross-attention logits are NOT produced here.  `timing.get_attentions` taps the
    outputs of `cross_attn.query` / `cross_attn.key` and hands them to the sm_100a
    capture kernel, so any module with this tree (including a stock upstream model)
    works as `model`;
  * the decoder accepts right-padded token batches (causal masking makes the padding
    invisible to the real positions).
"""
from __future__ import annotations

import math
import os
from dataclasses import asdict, dataclass

import torch
import torch.nn.functional as F
from torch import nn


@dataclass
class ModelDimensions:
    n_mels: int
    n_audio_ctx: int
    n_audio_state: int
    n_audio_head: int
    n_audio_layer: int
    n_vocab: int
    n_text_ctx: int
    n_text_state: int
    n_text_head: int
    n_text_layer: int


#: published sizes: (mels, audio ctx, width, heads, layers, vocab, text ctx, width, heads, layers)
SIZES = {
    "tiny": (80, 1500, 384, 6, 4, 51865, 448, 384, 6, 4),
    "base": (80, 1500, 512, 8, 6, 51865, 448, 512, 8, 6),
    "small": (80, 1500, 768, 12, 12, 51865, 448, 768, 12, 12),
    "medium": (80, 1500, 1024, 16, 24, 51865, 448, 1024, 16, 24),
    "large-v3": (128, 1500, 1280, 20, 32, 51866, 448, 1280, 20, 32),
}


def dims_for(name: str) -> ModelDimensions:
    return ModelDimensions(*SIZES[name])


#: "wca": unmasked attention (encoder self-attention, decoder cross-attention output) runs on csrc/enc_attn.cu;
#: "sdpa": torch SDPA (fp32 CUDA-core kernel).
ENCODER_ATTENTION = os.environ.get("WCA_ENCODER_ATTENTION", "wca")
#: "wca": the decoder's causal self-attention runs on the same kernel (wca_causal_attention); "sdpa": torch SDPA
CAUSAL_ATTENTION = os.environ.get("WCA_CAUSAL_ATTENTION", "wca")


class _Norm(nn.LayerNorm):
    def forward(self, x):
        return super().forward(x.float()).to(x.dtype)


class _Proj(nn.Linear):
    def forward(self, x):
        bias = self.bias if self.bias is None else self.bias.to(x.dtype)
        return F.linear(x, self.weight.to(x.dtype), bias)


class _Conv(nn.Conv1d):
    def _conv_forward(self, x, weight, bias):
        return super()._conv_forward(x, weight.to(x.dtype), None if bias is None else bias.to(x.dtype))


#: True: projections that read the same activations run as ONE cuBLAS GEMM against concatenated weights -- Q/K/V of a
#: self-attention (N = 3d) and the cross-attention K and V of ALL decoder layers (N = 2 * layers * d of the encoder
#: output).  Same products, fewer launches: with BF16x9 emulation every GEMM first scans its operands for Inf/NaN, and
#: `xa` (batch * 1500 rows) was scanned 2 * layers times.  False: one GEMM per nn.Linear, as the module tree suggests.
FUSED_PROJECTIONS = os.environ.get("WCA_FUSED_PROJECTIONS", "1") != "0"
#: decoder layers whose cross-attention K and V share one GEMM over the encoder output.  The output row pitch grows with
#: the group (2 * group * d floats), and the kernels that read one layer's K / V out of it walk rows that far apart.
#: Measured on a B200 (TIMIT-shaped batch of 32, one box, capture launch / attention / step): unfused 0.397 / 41.5 / 342.8 ms,
#: group 1: 0.407 / 41.7 / 340.6, group 4: 0.408 / 41.8 / 338.7, all 24 layers: 0.447 / 42.4 / 342.9.
CROSS_KV_GROUP = int(os.environ.get("WCA_CROSS_KV_GROUP", "4"))


class _FusedWeights:
    """Concatenation of several projections' weights (and biases, zeros where a projection has none), rebuilt when
    any parameter is reassigned, modified in place or moved."""

    def __init__(self):
        self.key = None
        self.weight = self.bias = None

    def get(self, projections, dtype):
        key = tuple((p.weight.data_ptr(), p.weight._version, None if p.bias is None else p.bias._version)
                    for p in projections) + (dtype,)
        if key != self.key:
            with torch.no_grad():
                self.weight = torch.cat([p.weight.detach().to(dtype) for p in projections], dim=0)
                self.bias = torch.cat([torch.zeros(p.weight.shape[0], dtype=dtype, device=p.weight.device)
                                       if p.bias is None else p.bias.detach().to(dtype) for p in projections])
            self.key = key
        return self.weight, self.bias


class Attention(nn.Module):
    """query/key/value/out projections (key without bias) around SDPA."""

    def __init__(self, width: int, heads: int):
        super().__init__()
        self.n_head = heads
        self.query = _Proj(width, width)
        self.key = _Proj(width, width, bias=False)
        self.value = _Proj(width, width)
        self.out = _Proj(width, width)
        self._qkv = _FusedWeights()

    def _split(self, t):
        return t.unflatten(-1, (self.n_head, -1)).transpose(1, 2)

    def forward(self, x, xa=None, causal: bool = False, kv=None, tap=None, cache=None, step: bool = False):
        """kv: (k, v) already projected (views into the decoder's all-layer K/V GEMM); tap: list that receives
        (q, k) of a cross-attention for the capture kernel.  step: one greedy decode step, x holds one new row per batch
        item and attends on the decode kernel (csrc/decode_attn.cu) -- a cross-attention over `kv`, a self-attention
        over its cache = (buffer (batch, n_text_ctx, 2d), pos): the row's K and V go to buffer[:, pos] (K then V), the
        query attends over buffer[:, :pos + 1]."""
        if step:
            from . import _cabi

            if cache is not None:
                buf, pos = cache
                w, b = self._qkv.get((self.query, self.key, self.value), x.dtype)
                d = x.shape[-1]
                qkv = F.linear(x, w, b)  # (batch, 1, 3d)
                buf[:, pos:pos + 1].copy_(qkv[..., d:])
                q, k, v = qkv[..., :d], buf[:, :pos + 1, :d], buf[:, :pos + 1, d:]
            else:
                q, (k, v) = self.query(x), kv
            return self.out(_cabi.decode_attention(q[:, 0], k, v, self.n_head).unsqueeze(1)), None
        fused = FUSED_PROJECTIONS and x.is_cuda and not torch.is_grad_enabled()
        if kv is not None:
            q, (k, v) = self.query(x), kv
        elif xa is None and fused:
            w, b = self._qkv.get((self.query, self.key, self.value), x.dtype)
            d = x.shape[-1]
            qkv = F.linear(x, w, b)  # (batch, n, 3d): q, k, v are strided views, read in place by the kernels
            q, k, v = qkv[..., :d], qkv[..., d:2 * d], qkv[..., 2 * d:]
        else:
            src = x if xa is None else xa
            q, k, v = self.query(x), self.key(src), self.value(src)
        if tap is not None:
            tap.append((q, k))
        if (ENCODER_ATTENTION == "wca" and q.is_cuda and q.dtype == torch.float32 and q.shape[-1] == 64 * self.n_head
                and (not causal or CAUSAL_ATTENTION == "wca")):
            # encoder self-attention, decoder cross-attention output and (causal) decoder self-attention: the sm_100a
            # tcgen05 kernel (csrc/enc_attn.cu) reads the projection outputs in place (no head split /
            # transposes) and keeps fp32 accuracy with 3 x tf32 products
            from . import _cabi

            return self.out(_cabi.full_attention(q, k, v, self.n_head, causal=causal and q.shape[1] > 1)), None
        q, k, v = self._split(q), self._split(k), self._split(v)  # views, also of the column slices of a fused projection
        # SDPA's default scale is d_head^-1/2 == (d_head^-1/4)^2, the published scaling
        ctx = F.scaled_dot_product_attention(q, k, v, is_causal=causal and q.shape[2] > 1)
        return self.out(ctx.transpose(1, 2).flatten(2)), None


#: "wca": residual add + LayerNorm pairs run as one sm_100a kernel (csrc/layernorm.cu); "torch": separate ops.
ADD_LAYERNORM = os.environ.get("WCA_ADD_LAYERNORM", "wca")


def _add_ln(x, h, ln):
    """(x + h, ln(x + h)); h None -> (x, ln(x)).  One fused kernel for fp32 CUDA tensors of a supported width."""
    if (ADD_LAYERNORM == "wca" and x.is_cuda and x.dtype == torch.float32 and x.shape[-1] % 128 == 0
            and x.shape[-1] // 128 in (1, 2, 3, 4, 6, 8, 10) and ln.weight.dtype == torch.float32):
        from . import _cabi

        x = x if x.is_contiguous() else x.contiguous()
        if h is not None and not h.is_contiguous():
            h = h.contiguous()
        return _cabi.add_layernorm(x, h, ln.weight, ln.bias, ln.eps)
    y = x if h is None else x + h
    return y, ln(y)


class Block(nn.Module):
    def __init__(self, width: int, heads: int, cross: bool):
        super().__init__()
        self.attn = Attention(width, heads)
        self.attn_ln = _Norm(width)
        self.cross_attn = Attention(width, heads) if cross else None
        self.cross_attn_ln = _Norm(width) if cross else None
        self.mlp = nn.Sequential(_Proj(width, 4 * width), nn.GELU(), _Proj(4 * width, width))
        self.mlp_ln = _Norm(width)

    def forward(self, x, xa=None, causal: bool = False, pending=None, kv=None, tap=None, cache=None):
        """Upstream: x += attn(ln(x)); x += cross_attn(ln(x), xa); x += mlp(ln(x)).  Every residual add is
        paired with the LayerNorm that follows it, so the last add of a block is handed to the next one
        (`pending`): returns (x, h) with the block's output being x + h.  cache: (buffer, pos) of the self-attention's
        K/V for one greedy decode step (Attention.forward)."""
        step = cache is not None
        x, n = _add_ln(x, pending, self.attn_ln)
        h = self.attn(n, causal=causal, cache=cache, step=step)[0]
        if self.cross_attn is not None:
            x, n = _add_ln(x, h, self.cross_attn_ln)
            h = self.cross_attn(n, xa, kv=kv, tap=tap, step=step)[0]
        x, n = _add_ln(x, h, self.mlp_ln)
        return x, self.mlp(n)


def _sinusoid_table(length: int, width: int, max_timescale: float = 10000.0):
    half = width // 2
    rates = torch.exp(-(math.log(max_timescale) / (half - 1)) * torch.arange(half))
    phase = torch.arange(length)[:, None] * rates[None, :]
    return torch.cat([phase.sin(), phase.cos()], dim=1)


class AudioEncoder(nn.Module):
    def __init__(self, n_mels, n_ctx, width, heads, layers):
        super().__init__()
        self.conv1 = _Conv(n_mels, width, kernel_size=3, padding=1)
        self.conv2 = _Conv(width, width, kernel_size=3, stride=2, padding=1)
        self.register_buffer("positional_embedding", _sinusoid_table(n_ctx, width))
        self.blocks = nn.ModuleList([Block(width, heads, cross=False) for _ in range(layers)])
        self.ln_post = _Norm(width)

    @staticmethod
    def _conv_as_gemm(x, conv):
        """Conv1d (kernel 3, padding 1, stride 1 or 2) over a (batch, frames, channels) tensor as ONE cuBLAS GEMM on
        unfolded windows: the same sums in another order, output again (batch, frames, channels) -- the layout the
        blocks want.  cuDNN's fp32 path for these shapes is a CUDA-core kernel and hands back (batch, channels,
        frames), which made every LayerNorm of the encoder copy a permuted residual stream."""
        b, _, c = x.shape
        cols = F.pad(x, (0, 0, 1, 1)).unfold(1, 3, conv.stride[0])       # (b, frames_out, c, 3) view
        cols = cols.reshape(b * cols.shape[1], c * 3)
        w = conv.weight.to(x.dtype).reshape(conv.out_channels, c * 3)
        return torch.addmm(conv.bias.to(x.dtype), cols, w.t()).view(b, -1, conv.out_channels)

    def forward(self, mel):
        if mel.is_cuda and mel.dtype == torch.float32:
            x = F.gelu(self._conv_as_gemm(mel.transpose(1, 2).contiguous(), self.conv1))
            x = F.gelu(self._conv_as_gemm(x, self.conv2))
        else:
            x = F.gelu(self.conv2(F.gelu(self.conv1(mel)))).transpose(1, 2).contiguous()
        if x.shape[1:] != self.positional_embedding.shape:
            raise ValueError(f"incorrect audio shape {tuple(mel.shape)}: expected {2 * self.positional_embedding.shape[0]} frames")
        x = (x + self.positional_embedding).to(x.dtype)
        pending = None
        for blk in self.blocks:
            x, pending = blk(x, pending=pending)
        return _add_ln(x, pending, self.ln_post)[1]


class TextDecoder(nn.Module):
    def __init__(self, n_vocab, n_ctx, width, heads, layers):
        super().__init__()
        self.token_embedding = nn.Embedding(n_vocab, width)
        self.positional_embedding = nn.Parameter(torch.empty(n_ctx, width))
        self.blocks = nn.ModuleList([Block(width, heads, cross=True) for _ in range(layers)])
        self.ln = _Norm(width)
        self._cross_kv = {}

    def cross_kv(self, xa, first, count):
        """K and V of the cross-attention of decoder layers [first, first + count) in ONE GEMM over the encoder output:
        (batch, n_ctx, 2 * count * d), layer first + i's K at columns [2i d, (2i+1) d), its V right after.  The kernels
        read the strided views in place."""
        projections = [p for blk in self.blocks[first:first + count] for p in (blk.cross_attn.key, blk.cross_attn.value)]
        w, b = self._cross_kv.setdefault((first, count), _FusedWeights()).get(projections, xa.dtype)
        return F.linear(xa, w, b)

    def cross_kv_group(self):
        """Decoder layers per cross_kv GEMM: the largest divisor of the layer count up to CROSS_KV_GROUP (equal groups
        only: the capture kernel reads every layer's K with ONE row pitch)."""
        return max(k for k in range(1, max(1, min(CROSS_KV_GROUP, len(self.blocks))) + 1) if len(self.blocks) % k == 0)

    def forward(self, tokens, xa, tap=None, cache=None):
        """tap: list that receives (q, k) of every layer's cross-attention (what timing.get_attentions captures).
        cache: a DecodeCache -- one greedy decode step: tokens (batch, 1) is position cache.pos, attention runs over
        the cached K/V, the step appends its own and advances cache.pos."""
        if cache is not None:
            return self._step(tokens, xa, cache)
        x = self.token_embedding(tokens) + self.positional_embedding[: tokens.shape[-1]]
        x = x.to(xa.dtype)
        d = x.shape[-1]
        fused = FUSED_PROJECTIONS and CROSS_KV_GROUP > 0 and xa.is_cuda and not torch.is_grad_enabled()
        group = self.cross_kv_group()
        kv_group = None
        pending = None
        for l, blk in enumerate(self.blocks):
            kv = None
            if fused:
                i = l % group
                if i == 0:
                    kv_group = self.cross_kv(xa, l, min(group, len(self.blocks) - l))
                kv = (kv_group[..., 2 * i * d:(2 * i + 1) * d], kv_group[..., (2 * i + 1) * d:(2 * i + 2) * d])
            x, pending = blk(x, xa, causal=True, pending=pending, kv=kv, tap=tap)
        x = _add_ln(x, pending, self.ln)[1]
        return self._vocab_logits(x)

    def _step(self, tokens, xa, cache):
        pos = cache.pos
        if tokens.shape[-1] != 1 or pos >= self.positional_embedding.shape[0]:
            raise ValueError(f"a decode step takes one token per row inside the text context (position {pos})")
        x = (self.token_embedding(tokens) + self.positional_embedding[pos: pos + 1]).to(xa.dtype)
        pending = None
        for l, blk in enumerate(self.blocks):
            x, pending = blk(x, xa, causal=True, pending=pending, kv=cache.cross[l], cache=(cache.self_kv[l], pos))
        cache.pos = pos + 1
        x = _add_ln(x, pending, self.ln)[1]
        return self._vocab_logits(x)

    def _vocab_logits(self, x):
        """x @ E^T.  n_vocab (51865 / 51866) is odd or not a multiple of 4, so the output rows are misaligned and
        cuBLAS falls back to a CUDA-core SGEMM; on the device the product is computed against a copy of E padded
        to a multiple of 16 rows (cached, rebuilt when the weight changes) and the padding columns are dropped."""
        w = self.token_embedding.weight
        if not (x.is_cuda and x.dtype == torch.float32 and w.dtype == torch.float32) or w.shape[0] % 16 == 0:
            return (x @ w.to(x.dtype).t()).float()
        key = (w.data_ptr(), w._version, w.device)
        if getattr(self, "_padded_key", None) != key:
            rows = (w.shape[0] + 15) // 16 * 16
            padded = torch.zeros(rows, w.shape[1], dtype=w.dtype, device=w.device)
            padded[: w.shape[0]] = w.detach()
            self._padded_vocab, self._padded_key = padded, key
        return F.linear(x, self._padded_vocab)[..., : w.shape[0]]


class DecodeCache:
    """K/V state of a cached greedy decode over audio features xa (batch, n_audio_ctx, d), CUDA fp32: the
    cross-attention K/V of every decoder layer, computed once with the grouped TextDecoder.cross_kv GEMMs (views into
    them), and per layer a (batch, n_text_ctx, 2d) self-attention cache, K then V, of which positions < pos are filled."""

    def __init__(self, decoder: TextDecoder, xa: torch.Tensor):
        from . import _cabi

        if not xa.is_cuda or xa.dtype != torch.float32:
            raise _cabi.WcaError("the cached decoder needs fp32 CUDA audio features (no CPU fallback exists)")
        n_layers, (n_ctx, d) = len(decoder.blocks), decoder.positional_embedding.shape
        group = decoder.cross_kv_group()
        self.cross = []
        for first in range(0, n_layers, group):
            kv = decoder.cross_kv(xa, first, group)
            self.cross += [(kv[..., 2 * i * d:(2 * i + 1) * d], kv[..., (2 * i + 1) * d:(2 * i + 2) * d]) for i in range(group)]
        self.self_kv = [torch.empty(xa.shape[0], n_ctx, 2 * d, dtype=xa.dtype, device=xa.device) for _ in range(n_layers)]
        self.pos = 0


class Whisper(nn.Module):
    def __init__(self, dims: ModelDimensions):
        super().__init__()
        self.dims = dims
        self.encoder = AudioEncoder(dims.n_mels, dims.n_audio_ctx, dims.n_audio_state, dims.n_audio_head,
                                    dims.n_audio_layer)
        self.decoder = TextDecoder(dims.n_vocab, dims.n_text_ctx, dims.n_text_state, dims.n_text_head,
                                   dims.n_text_layer)
        upper = torch.zeros(dims.n_text_layer, dims.n_text_head, dtype=torch.bool)
        upper[dims.n_text_layer // 2:] = True
        self.register_buffer("alignment_heads", upper.to_sparse(), persistent=False)

    def embed_audio(self, mel):
        return self.encoder(mel)

    def logits(self, tokens, audio_features):
        return self.decoder(tokens, audio_features)

    def forward(self, mel, tokens):
        return self.decoder(tokens, self.encoder(mel))

    def forward_with_cross_qk(self, mel, tokens, audio_features=None):
        """(logits, [q_l (batch, T, d)], [k_l (batch, n_ctx, d)]): the teacher-forced forward plus the cross-attention
        projections of every decoder layer, as the capture kernel reads them (k_l may be a strided view of the all-layer
        K/V GEMM).  timing.get_attentions uses this when the model offers it; any other module tree (a stock
        openai-whisper model) is tapped with forward hooks on cross_attn.query / cross_attn.key instead.
        audio_features: the encoder output of `mel`, already computed (mel is then not read)."""
        tap = []
        xa = self.encoder(mel) if audio_features is None else audio_features
        logits = self.decoder(tokens, xa, tap=tap)
        return logits, [q for q, _ in tap], [k for _, k in tap]

    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def is_multilingual(self):
        return self.dims.n_vocab >= 51865

    @property
    def num_languages(self):
        return self.dims.n_vocab - 51765 - int(self.is_multilingual)


#: tiny dims for smoke runs: 30 s context and head width 64 like the published models
TEST_SIZES = {
    "micro": (80, 1500, 128, 2, 2, 51865, 448, 128, 2, 2),
    "mini": (80, 1500, 256, 4, 2, 51865, 448, 256, 4, 3),
}


def load_model(name_or_path: str, device=None, *, seed: int = 0, qk_gain: float = 1.0) -> Whisper:
    """A checkpoint file ({"dims", "model_state_dict"}, the published openai-whisper format) if `name_or_path` is a
    path; `random:<size>` (e.g. `random:medium`, `random:micro`) for a SEEDED RANDOM-INIT model of that size.  A bare
    size name is refused: no checkpoint can be downloaded offline, and aligning with random weights must be asked for
    explicitly -- the results look like a real run but mean nothing.  The returned model carries `.model_source`."""
    if os.path.isfile(name_or_path):
        ckpt = torch.load(name_or_path, map_location="cpu", weights_only=True)
        model = Whisper(ModelDimensions(**ckpt["dims"]))
        model.load_state_dict(ckpt["model_state_dict"])
        model.model_source = f"checkpoint:{os.path.abspath(name_or_path)}"
    elif name_or_path.startswith("random:"):
        size = name_or_path.split(":", 1)[1]
        if size in TEST_SIZES:
            dims = ModelDimensions(*TEST_SIZES[size])
        elif size in SIZES:
            dims = dims_for(size)
        else:
            raise ValueError(f"unknown model size {size!r}: one of {sorted(SIZES) + sorted(TEST_SIZES)}")
        model = random_init(dims, seed=seed, qk_gain=qk_gain)
        model.model_source = f"random-init:{size}:seed{seed}:qk_gain{qk_gain:g}"
    else:
        raise FileNotFoundError(
            f"{name_or_path!r} is not a checkpoint file, and openai-whisper (which would download it) is not installed. "
            f"Pass a checkpoint path, or `random:{name_or_path}` to align with a seeded RANDOM-INIT model "
            "(synthetic benchmarks / smoke runs only: its alignments are meaningless).")
    model.eval()
    return model if device is None else model.to(device)


def random_init(dims: ModelDimensions, seed: int = 0, qk_gain: float = 1.0, device=None) -> Whisper:
    """Seeded synthetic weights.  `qk_gain` scales the cross-attention query/key projections
    so that the maps are peaky enough for alignment paths to be data-driven.  With `device` the parameters are created
    (and drawn) directly there -- seconds instead of a minute for large-v3 -- from that device's generator, i.e. NOT the
    weights the same seed gives on the CPU (throughput runs only; parity runs share CPU-initialised weights with the oracle)."""
    if device is not None and torch.device(device).type == "cuda":
        with torch.device(device):
            torch.cuda.manual_seed(seed)
            model = Whisper(dims)
            with torch.no_grad():
                model.decoder.positional_embedding.normal_(0, 0.02)
                for blk in model.decoder.blocks:
                    blk.cross_attn.query.weight.mul_(qk_gain)
                    blk.cross_attn.query.bias.mul_(qk_gain)
                    blk.cross_attn.key.weight.mul_(qk_gain)
        return model.eval()
    keep = torch.random.get_rng_state()
    torch.manual_seed(seed)
    model = Whisper(dims)
    with torch.no_grad():
        model.decoder.positional_embedding.normal_(0, 0.02)
        for blk in model.decoder.blocks:
            blk.cross_attn.query.weight.mul_(qk_gain)
            blk.cross_attn.query.bias.mul_(qk_gain)
            blk.cross_attn.key.weight.mul_(qk_gain)
    torch.random.set_rng_state(keep)
    return model.eval()


@torch.no_grad()
def greedy_decode(model: Whisper, mel: torch.Tensor, tokenizer, max_tokens: int = 224) -> list:
    """Greedy transcription without timestamps -- what the reference obtains from
    `whisper.decode(model, mel, DecodingOptions(language="en"))` (infer_ali.py:60) for the text it then
    aligns.  mel: (n_mels, 3000) or (B, n_mels, 3000).  Returns one list of text tokens per utterance.
    The prefix is re-run every step (no KV cache): the decoder context is at most 448 tokens and this
    step is outside the alignment hot path."""
    single = mel.dim() == 2
    if single:
        mel = mel.unsqueeze(0)
    xa = model.encoder(mel)
    b = mel.shape[0]
    prefix = [*tokenizer.sot_sequence, tokenizer.no_timestamps]
    tokens = torch.tensor([prefix] * b, device=mel.device)
    done = torch.zeros(b, dtype=torch.bool, device=mel.device)
    limit = min(max_tokens, model.dims.n_text_ctx - len(prefix) - 1)
    for _ in range(limit):
        logits = model.decoder(tokens, xa)[:, -1]
        logits[:, tokenizer.eot + 1:] = -float("inf")  # no special tokens / timestamps in the text
        nxt = logits.argmax(-1)
        nxt = torch.where(done, torch.full_like(nxt, tokenizer.eot), nxt)
        tokens = torch.cat([tokens, nxt[:, None]], dim=1)
        done |= nxt == tokenizer.eot
        if bool(done.all()):
            break
    out = []
    for row in tokens[:, len(prefix):].tolist():
        out.append(row[: row.index(tokenizer.eot)] if tokenizer.eot in row else row)
    return out[0] if single else out


@torch.no_grad()
def greedy_decode_cached(model: Whisper, audio_features: torch.Tensor, tokenizer, max_tokens: int = 224) -> list:
    """greedy_decode on a KV cache: the same procedure (prefix, limit, last-position logits, ids above EOT masked,
    first arg-max, finished rows emit EOT, stop when every row is done, cut at the first EOT) over encoder output that is
    already computed, audio_features (B, n_audio_ctx, d) fp32 CUDA.  The cross-attention K/V of every layer are
    projected once per call; each step projects one new token per row, appends its K/V to the layer's cache and attends
    on wca_decode_attention.  The prefix is fed one token per step.  Returns one list of text tokens per row."""
    dec = model.decoder
    cache = DecodeCache(dec, audio_features)
    b = audio_features.shape[0]
    prefix = [*tokenizer.sot_sequence, tokenizer.no_timestamps]
    tokens = torch.tensor([prefix] * b, device=audio_features.device)
    done = torch.zeros(b, dtype=torch.bool, device=audio_features.device)
    limit = min(max_tokens, model.dims.n_text_ctx - len(prefix) - 1)
    for p in range(len(prefix) - 1 if limit > 0 else 0):
        dec(tokens[:, p:p + 1], audio_features, cache=cache)
    for _ in range(limit):
        logits = dec(tokens[:, -1:], audio_features, cache=cache)[:, -1]
        logits[:, tokenizer.eot + 1:] = -float("inf")  # no special tokens / timestamps in the text
        nxt = logits.argmax(-1)
        nxt = torch.where(done, torch.full_like(nxt, tokenizer.eot), nxt)
        tokens = torch.cat([tokens, nxt[:, None]], dim=1)
        done |= nxt == tokenizer.eot
        if bool(done.all()):
            break
    out = []
    for row in tokens[:, len(prefix):].tolist():
        out.append(row[: row.index(tokenizer.eot)] if tokenizer.eot in row else row)
    return out


def save_checkpoint(model: Whisper, path: str):
    torch.save({"dims": asdict(model.dims), "model_state_dict": model.state_dict()}, path)
