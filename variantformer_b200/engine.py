"""Forward schedule of the hot path on top of the C-ABI kernels.

What runs here (reference sites in brackets):
  seq2reg window encoder      [seq2reg/model.py:193-279, seq2reg/modules.py:149-191]
  cre_map / gene_map          [seq2gene/model_combined_modulator.py:610-612]
  registry token + tissue axis [layers.py:508-521, model_combined_modulator.py:622-666]
  CombinedModulator           [model_combined_modulator.py:137-328, layers.py:88-165]
  head + Softplus             [layers.py:1078-1087, 1113-1144]

Schedule differences from the reference (results identical, oracle/model_fp32.py proves it):
  * the CRE stream is computed once per gene, not once per (gene, tissue) — tissue only enters
    through the registry token of the gene stream;
  * all tissue copies of a gene share one K/V projection of the CRE stream: their queries are
    stacked on the M axis of a single cross-attention problem;
  * the CRE x label cross-attention is collapsed to the 9 label classes;
  * only valid (unpadded) tokens are ever materialised.
  * every LayerNorm that feeds a Linear is folded into that GEMM: gamma into the weight, beta into the bias, and
    the per-row mean / rstd applied in the GEMM epilogue from (sum, sum of squares) that the epilogue of the GEMM
    which produced the row accumulated.  No LayerNorm pass reads the streams.
  * residual streams are stored row-centred (x - c_r, c_r = the row mean where the stream is assembled): exact, because
    every consumer is a LayerNorm or a residual add; raw values are rebuilt where they are needed (cross-attention
    context, pooled windows, returned embeddings).  Keeps the LayerNorm fold accurate when |mean| >> std.
Numerics: bf16 GEMM/attention operands, fp32 accumulation, fp32 residual stream and LayerNorm statistics.
"""
import math
import os

import numpy as np
import torch

from . import ops
from ._lib import EPI_BIAS_BF16, EPI_BIAS_F32, EPI_BIAS_GEGLU_BF16, EPI_BIAS_GELU_BF16, EPI_BIAS_RESID_F32
from .utils.alibi import alibi_slopes

NUM_REF_CRES = 9
# "coarse" (default): the forward of a slab is three calls into the library (vf_seq2reg_forward x2, vf_seq2gene_forward)
# with the layer loop in C++; "fine": one Python call per kernel — the same kernels in the same order, bit-identical
# results; used when a launch profiler is attached (bench.py's per-kernel pass) and for A/B runs (VF_ENGINE=fine).
COARSE = os.environ.get("VF_ENGINE", "coarse") != "fine"
# x1 = x + MHA(..) exists only as a bf16 mirror (its consumers are a LayerNorm-folded GEMM and the next residual add), so
# the out_proj epilogue may read its residual from the bf16 mirror of x instead of the fp32 stream: half the residual
# bytes of the most HBM-bound GEMMs of the layer.  The fp32 stream itself is untouched (the layer's own residual add reads
# it in full precision).  VF_RESID16_OUTPROJ=0: fp32 residual there too (A/B).
OUT_PROJ_RESID16 = os.environ.get("VF_RESID16_OUTPROJ", "1") != "0"
# run the CRE stack on its own CUDA stream, concurrently with the gene stack ("0": one stream, for A/B and debugging)
CRE_STREAM = os.environ.get("VF_CRE_STREAM", "1") != "0"


class AttnPlan:
    """Host-built work decomposition of one attention problem (all sequences of a slab, one launch of
    vf_attention_mc_varlen).  The decomposition depends on the sequence lengths only, never on how genes are batched,
    so results do not depend on the batching."""

    def __init__(self, q_lens, device, head_dim, k_lens=None, units=None):
        if head_dim not in (48, 64):
            raise NotImplementedError(f"attention head size {head_dim}: the B200 kernel is built for 48 and 64 "
                                      "(vf_model.yaml: 1536/32 = 48; seq2reg 512/8 = 64)")
        self.slots = ops.SlotMap.from_units(units, device) if units is not None else \
            ops.SlotMap(q_lens, device, k_lens=k_lens)

    def device_tensors(self):
        return [self.slots.table]

    def run(self, q, k, v, heads, head_dim, slopes, out):
        return ops.attention_mc(q, k, v, self.slots, heads, head_dim, slopes, out=out)


def sinusoidal_pe(d_model: int, length: int) -> torch.Tensor:
    """Same arithmetic as seq2reg/model.py:15-37 (computed once on the host in fp32)."""
    pe = torch.zeros(length, d_model)
    position = torch.arange(0, length).unsqueeze(1).float()
    div = torch.exp(torch.arange(0, d_model, 2, dtype=torch.float) * -(math.log(10000.0) / d_model))
    pe[:, 0::2] = torch.sin(position * div)
    pe[:, 1::2] = torch.cos(position * div)
    return pe


def interleave_geglu(w: torch.Tensor) -> torch.Tensor:
    """Reorder linear_geglu_1 rows so each 256-row tile holds 128 `u` rows followed by their 128 `gate`
    rows (u, gate = chunk(2, -1): layers.py:159-160).  Works for weights [2h, K] and biases [2h]."""
    h = w.shape[0] // 2
    assert h % 128 == 0, "GeGLU hidden size must be a multiple of 128"
    u = w[:h].reshape(h // 128, 128, *w.shape[1:])
    g = w[h:].reshape(h // 128, 128, *w.shape[1:])
    return torch.cat([u, g], dim=1).reshape(w.shape).contiguous()


class _Linear:
    __slots__ = ("w", "b")

    def __init__(self, sd, name, device, geglu=False):
        w, b = sd[name + ".weight"].float(), sd[name + ".bias"].float()
        if geglu:
            w, b = interleave_geglu(w), interleave_geglu(b)
        self.w = w.to(device=device, dtype=torch.bfloat16).contiguous()
        self.b = b.to(device=device, dtype=torch.float32).contiguous()


class _LnLinear:
    """Linear(LayerNorm(x)) with the norm folded in (vf_gemm.cu header): w = bf16(W * gamma), cs = row sums of that
    bf16 weight (what the tensor cores will actually multiply the row mean by), b = bias + W beta."""
    __slots__ = ("w", "b", "cs", "dim", "eps")

    def __init__(self, sd, name, norm, device, geglu=False, eps=1e-5):
        w, b = sd[name + ".weight"].float(), sd[name + ".bias"].float()
        g, beta = sd[norm + ".weight"].float(), sd[norm + ".bias"].float()
        wf = (w * g[None, :]).to(torch.bfloat16)
        cs = wf.float().sum(1)
        bf = b + w @ beta
        if geglu:
            wf, cs, bf = interleave_geglu(wf), interleave_geglu(cs), interleave_geglu(bf)
        self.w = wf.to(device).contiguous()
        self.cs = cs.to(device=device, dtype=torch.float32).contiguous()
        self.b = bf.to(device=device, dtype=torch.float32).contiguous()
        self.dim, self.eps = w.shape[1], eps

    def ln(self, stats):
        return (stats, self.cs, self.dim, self.eps)


class _Norm:
    __slots__ = ("g", "b")

    def __init__(self, sd, name, device):
        self.g = sd[name + ".weight"].to(device=device, dtype=torch.float32).contiguous()
        self.b = sd[name + ".bias"].to(device=device, dtype=torch.float32).contiguous()


class Workspace:
    """Grow-only named device buffers, reused across layers and batches."""

    def __init__(self, device):
        self.device = device
        self._buf = {}

    def get(self, name, shape, dtype):
        n = int(np.prod(shape))
        b = self._buf.get(name)
        if b is None or b.numel() < n or b.dtype != dtype:
            b = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._buf[name] = b
        return b[:n].view(*shape)


class Seq2RegWeights:
    """Device copy of one Seq2RegPredictor (`use_context=False`, the configuration both tokenizers use)."""

    def __init__(self, sd, prefix, hp, device):
        if hp.get("use_context", False):
            raise NotImplementedError("seq2reg use_context=True checkpoints are not supported on the B200 path yet")
        self.d = hp["embedding_dim"]; self.H = hp["num_heads"]; self.L = hp["num_layers"]
        self.hd = self.d // self.H
        self.token_length = hp.get("token_length") or 200
        self.emb = sd[prefix + "token_embedding.weight"].to(device=device, dtype=torch.float32).contiguous()
        if hp.get("positional_encoding", "sinusoidal") == "sinusoidal":
            self.pe = sinusoidal_pe(self.d, self.token_length).to(device)
            self.slopes = None
        else:
            self.pe = None
            self.slopes = alibi_slopes(self.H).to(device)
        self.layers = []
        for l in range(self.L):
            p = f"{prefix}transformer_encoder.{l}."
            self.layers.append(seq2reg_layer_weights(sd, p, device))
        self._abi = None

    def abi(self):
        """Weight-pointer table of vf_seq2reg_forward (built once; the ctypes arrays are kept alive here)."""
        if self._abi is None:
            from . import _abi
            self._abi = _abi.seq2reg_table(self)
        return self._abi[0]


def seq2reg_layer_weights(sd, p, device, mha="MHA."):
    """Device weights of one FlashTransformerLayer (seq2reg/modules.py:129-147), LayerNorms folded.  mha="mixer.MHA.":
    the same layer shape under seq2gene's names (FlashAttentionEncoderLayer, layers.py:166-228)."""
    return dict(qkv=_LnLinear(sd, p + mha + "Wqkv", p + "norm1", device), out=_Linear(sd, p + mha + "out_proj", device),
                g1=_LnLinear(sd, p + "linear_geglu_1", p + "norm2", device, geglu=True),
                g2=_Linear(sd, p + "linear_geglu_2", device))


def context_layer_weights(sd, p, device, emb9=None):
    """Device weights of one ContextFlashAttentionEncoderLayer (layers.py:47-86), LayerNorms folded.  emb9 (bf16 [9, D],
    the label embedding table): the layer's cross-attention context is a label embedding, so K/V of the 9 classes are
    computed once here (weights only) and `kv` is dropped."""
    L = dict(qkv=_LnLinear(sd, p + "mixer.MHA.Wqkv", p + "norm1", device),
             out=_Linear(sd, p + "mixer.MHA.out_proj", device),
             q=_LnLinear(sd, p + "crossMHA.MHA.Wq", p + "norm2", device),
             kv=_Linear(sd, p + "crossMHA.MHA.Wkv", device),
             out2=_Linear(sd, p + "crossMHA.MHA.out_proj", device),
             g1=_LnLinear(sd, p + "linear_geglu_1", p + "norm3", device, geglu=True),
             g2=_Linear(sd, p + "linear_geglu_2", device))
    if emb9 is not None:
        L["kv9"] = ops.gemm(emb9.contiguous(), L["kv"].w, EPI_BIAS_F32, bias=L["kv"].b)
        L["kv"] = None
    return L


def cross_layer_weights(sd, p, device):
    """Device weights of one ContextFlashCrossAttentionEncoderLayer (layers.py:231-265): cross-attention + GeGLU FFN."""
    return dict(q=_LnLinear(sd, p + "crossMHA.MHA.Wq", p + "norm1", device), kv=_Linear(sd, p + "crossMHA.MHA.Wkv", device),
                out2=_Linear(sd, p + "crossMHA.MHA.out_proj", device),
                g1=_LnLinear(sd, p + "linear_geglu_1", p + "norm2", device, geglu=True),
                g2=_Linear(sd, p + "linear_geglu_2", device))


class Seq2GeneWeights:
    def __init__(self, sd, cfg, device):
        self.D = cfg["emb_dim"]; self.H = cfg["num_heads"]; self.NL = cfg["num_layers"]
        self.hd = self.D // self.H
        assert cfg.get("use_context", False) and not cfg.get("only_cross_attention", True) and \
            cfg.get("gene_pooling") == "multi_registry" and not cfg.get("add_context_to_cres", False) and \
            not cfg.get("use_res", False) and not cfg.get("cross_alibi", False) and \
            cfg.get("use_bigger_head", False) and not cfg.get("multi_head", True), \
            "only the configs/vf_model.yaml architecture variant is implemented on the B200 path"
        self.slopes = alibi_slopes(self.H).to(device) if cfg.get("use_alibi", True) else None
        self.registry = sd["start_tkn.registry_tokens.weight"].to(device=device, dtype=torch.float32).contiguous()
        self.gene_map = _Linear(sd, "gene_map", device)
        self.cre_map = _Linear(sd, "cre_map", device) if "cre_map.weight" in sd else None
        emb9 = sd["combined_modulator.second_level_context_embedding.weight"].to(device=device, dtype=torch.bfloat16)

        def layer(p, with_kv9):
            return context_layer_weights(sd, p, device, emb9 if with_kv9 else None)

        self.cre_layers = [layer(f"combined_modulator.cre_layers.{i}.", True) for i in range(self.NL - 1)]
        self.gene_layers = [layer(f"combined_modulator.gene_layers.{i}.", False) for i in range(self.NL)]
        p = "tissue_heads.tissue_expressions."
        self.h0 = _Linear(sd, p + "0", device); self.hn = _Norm(sd, p + "1", device); self.h4 = _Linear(sd, p + "4", device)
        self.h6_w = sd[p + "6.weight"].to(device=device, dtype=torch.float32).reshape(-1).contiguous()
        self.h6_b = sd[p + "6.bias"].to(device=device, dtype=torch.float32).contiguous()
        self.token_dim = self.gene_map.w.shape[1]
        self._abi = None

    def abi(self):
        """Weight-pointer table of vf_seq2gene_forward (built once; the ctypes arrays are kept alive here)."""
        if self._abi is None:
            from . import _abi
            self._abi = _abi.seq2gene_table(self, self.token_dim)
        return self._abi[0]


class Engine:
    """Batched inference over a slab of genes: tokens -> expression + embeddings."""

    def __init__(self, state_dict, cfg, seq2reg_hp, device="cuda", gene_seq2reg_hp=None):
        self.device = torch.device(device)
        self.cfg = dict(cfg)
        with torch.cuda.device(self.device):
            self.cre_tok = Seq2RegWeights(state_dict, "cre_tokenizer.", seq2reg_hp, self.device)
            self.gene_tok = Seq2RegWeights(state_dict, "gene_tokenizer.", gene_seq2reg_hp or seq2reg_hp, self.device)
            self.w = Seq2GeneWeights(state_dict, cfg, self.device)
        self.ws = Workspace(self.device)

    # ---------------------------------------------------------------- seq2reg
    def seq2reg(self, W: Seq2RegWeights, tokens_i32, mask_u8, lens_host, cu, plan: AttnPlan):
        """tokens/mask: device [n_win, L]; lens_host: numpy valid-token counts; cu: their prefix sums on the device;
        plan: the windows' attention work decomposition.  -> bf16 [n_win, d] masked mean of the last layer."""
        ws = self.ws
        n_win = tokens_i32.shape[0]
        n_tok = int(lens_host.sum())
        if COARSE and ops.PROFILER is None and hasattr(W, "abi"):
            import ctypes as C
            from . import _lib
            nbytes = int(_lib.lib().vf_seq2reg_workspace_bytes(C.addressof(W.abi()), n_tok))
            return ops.seq2reg_forward(W.abi(), tokens_i32, mask_u8, cu, n_tok, plan.slots,
                                       ws.get("coarse_r", (nbytes,), torch.uint8), W.d)
        ids, pos = ops.compact_tokens(tokens_i32, mask_u8, cu, n_tok)
        x = ops.embed_tokens(ids, pos, W.emb, W.pe)
        d, H, hd = W.d, W.H, W.hd
        xb = ws.get("r_xb", (n_tok, d), torch.bfloat16)                  # bf16 mirror of x / of x1
        P = ops.stats_parts(d)
        xs0 = ws.get("r_xs0", (n_tok, 1, 2), torch.float32)              # row (sum, sum of squares) of the embeddings
        xs = ws.get("r_xs", (n_tok, P, 2), torch.float32)                # ... of x as the FFN GEMM epilogue leaves them
        s1 = ws.get("r_s1", (n_tok, P, 2), torch.float32)                # ... of x1
        qkv = ws.get("r_qkv", (n_tok, 3 * d), torch.bfloat16)
        a = ws.get("r_a", (n_tok, d), torch.bfloat16)
        f = ws.get("r_f", (n_tok, W.layers[0]["g2"].w.shape[1]), torch.bfloat16)
        # the stream is kept row-centred (x - mean of the embedding row): LayerNorm does not see the shift, residual adds
        # carry it, and the bf16 mirror then spends its 8 bits on the normalised signal (vf_center_rows)
        piv = ws.get("r_piv", (n_tok,), torch.float32)
        ops.center_rows(x, piv, xs0, xb)
        for li, L in enumerate(W.layers):
            ops.gemm(xb, L["qkv"].w, EPI_BIAS_BF16, bias=L["qkv"].b, out=qkv,
                     ln=L["qkv"].ln(xs0 if li == 0 else xs))                                           # Wqkv(norm1(x))
            plan.run(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], H, hd, W.slopes, a)
            # x1 = x + MHA(..) is consumed only through norm2 -> linear_geglu_1 (the layer's residual is its INPUT,
            # modules.py:189): it exists as a bf16 mirror + row statistics only
            ops.gemm(a, L["out"].w, EPI_BIAS_RESID_F32, bias=L["out"].b, resid=xb if OUT_PROJ_RESID16 else x, out2=xb,
                     stats_out=s1, mirror_only=True)
            ops.gemm(xb, L["g1"].w, EPI_BIAS_GEGLU_BF16, bias=L["g1"].b, out=f, ln=L["g1"].ln(s1))      # GeGLU(norm2(x1))
            ops.gemm(f, L["g2"].w, EPI_BIAS_RESID_F32, bias=L["g2"].b, resid=x, out=x, out2=xb, stats_out=xs)  # + layer input
        return ops.masked_meanpool(x, cu, n_win, pivot=piv)

    # ---------------------------------------------------------------- one encoder layer of seq2gene
    def _layer(self, L, x, xb, xs, M, self_attn, cross_attn, tag, xb_out=None):
        """ContextFlashAttentionEncoderLayer on an unpadded fp32 stream x [M, D] with its bf16 mirror xb and row
        statistics xs (x updated in place; the mirror of the output goes to xb_out, by default xb itself)."""
        ws, D = self.ws, self.w.D
        hb = ws.get(tag + "_hb", (M, D), torch.bfloat16)                 # bf16 mirror of x1
        s1 = ws.get(tag + "_s1", (M, ops.stats_parts(D), 2), torch.float32)     # row statistics of x1
        xs_out = ws.get(tag + "_xs", (M, ops.stats_parts(D), 2), torch.float32)  # ... of the layer output
        qkv = ws.get(tag + "_qkv", (M, 3 * D), torch.bfloat16)
        a = ws.get(tag + "_a", (M, D), torch.bfloat16)
        f = ws.get(tag + "_f", (M, L["g2"].w.shape[1]), torch.bfloat16)
        ops.gemm(xb, L["qkv"].w, EPI_BIAS_BF16, bias=L["qkv"].b, out=qkv, ln=L["qkv"].ln(xs))          # Wqkv(norm1(x))
        self_attn(qkv, a)
        # x1 = x + selfMHA(..) and x1' = x1 + crossMHA(..) are consumed only through norm2 / norm3 -> bf16 GEMM and as
        # each other's residual (the layer's own residual is its INPUT, layers.py:163): bf16 mirror + statistics only
        ops.gemm(a, L["out"].w, EPI_BIAS_RESID_F32, bias=L["out"].b, resid=xb if OUT_PROJ_RESID16 else x, out2=hb,
                 stats_out=s1, mirror_only=True)
        q = qkv[:, :D]                                                  # reuse the qkv buffer for the cross query
        ops.gemm(hb, L["q"].w, EPI_BIAS_BF16, bias=L["q"].b, out=q, ln=L["q"].ln(s1))                  # Wq(norm2(x1))
        cross_attn(q, a)
        ops.gemm(a, L["out2"].w, EPI_BIAS_RESID_F32, bias=L["out2"].b, resid=hb, out2=hb, stats_out=s1, mirror_only=True)
        ops.gemm(hb, L["g1"].w, EPI_BIAS_GEGLU_BF16, bias=L["g1"].b, out=f, ln=L["g1"].ln(s1))         # GeGLU(norm3(x1))
        ops.gemm(f, L["g2"].w, EPI_BIAS_RESID_F32, bias=L["g2"].b, resid=x, out=x,
                 out2=xb if xb_out is None else xb_out, stats_out=xs_out)
        return xs_out

    # ---------------------------------------------------------------- last gene layer, needed rows only
    def _gene_layer_last(self, L, s, x, xb, xs, kv):
        """The last ContextFlashAttentionEncoderLayer of the gene stream restricted to the rows whose output is read
        (registry rows + VEP token rows): K/V of the self-attention still come from every row, all the rest runs on
        `need` rows.  Same arithmetic as _layer on those rows.  -> fp32 [n_need, D], still row-centred."""
        ws, w = self.ws, self.w
        D, H, hd = w.D, w.H, w.hd
        M, R = x.shape[0], s["n_need"]
        rows = s["last_rows"]
        qkvw = L["qkv"]
        kvs = ws.get("g_qkv", (M, 3 * D), torch.bfloat16)[:, D:]            # K | V of every row (Q columns unused)
        ops.gemm(xb, qkvw.w[D:], EPI_BIAS_BF16, bias=qkvw.b[D:], out=kvs, ln=(xs, qkvw.cs[D:], qkvw.dim, qkvw.eps))
        xR, xbR = ops.gather_rows(x, None, rows, want_f32=True, want_bf16=True)
        P = xs.shape[1]
        stR, _ = ops.gather_rows(xs.view(M, 2 * P), None, rows)
        stR = stR.view(R, P, 2)
        q = ops.gemm(xbR, qkvw.w[:D], EPI_BIAS_BF16, bias=qkvw.b[:D], ln=(stR, qkvw.cs[:D], qkvw.dim, qkvw.eps))
        a = torch.empty((R, D), dtype=torch.bfloat16, device=x.device)
        s["plan_last_self"].run(q, kvs[:, :D], kvs[:, D:], H, hd, w.slopes, a)
        hb = torch.empty((R, D), dtype=torch.bfloat16, device=x.device)
        s1 = torch.empty((R, ops.stats_parts(D), 2), dtype=torch.float32, device=x.device)
        ops.gemm(a, L["out"].w, EPI_BIAS_RESID_F32, bias=L["out"].b, resid=xbR if OUT_PROJ_RESID16 else xR, out2=hb,
                 stats_out=s1, mirror_only=True)
        ops.gemm(hb, L["q"].w, EPI_BIAS_BF16, bias=L["q"].b, out=q, ln=L["q"].ln(s1))
        s["plan_last_cross"].run(q, kv[:, :D], kv[:, D:], H, hd, None, a)
        ops.gemm(a, L["out2"].w, EPI_BIAS_RESID_F32, bias=L["out2"].b, resid=hb, out2=hb, stats_out=s1, mirror_only=True)
        f = ops.gemm(hb, L["g1"].w, EPI_BIAS_GEGLU_BF16, bias=L["g1"].b, ln=L["g1"].ln(s1))
        return ops.gemm(f, L["g2"].w, EPI_BIAS_RESID_F32, bias=L["g2"].b, resid=xR, out=xR)

    # ---------------------------------------------------------------- slab preparation (host bookkeeping + H2D)
    def prepare(self, cre_tokens, cre_masks, gene_tokens, gene_masks, tissues, ref_labels,
                cre_token_position=None, gene_token_position=None, lens=None):
        """Lists (one entry per gene) of: cre_tokens [C,L] int, cre_masks [C,L] bool (True = pad), gene_tokens
        [G,L], gene_masks [G,L], tissues [T] int, ref_labels [C] int (CPU or CUDA tensors).  Builds every index
        structure the kernels need and moves the token windows to the device (pinned staging for CPU inputs).
        `lens` = optional (cre_lens, gene_lens) host arrays to skip the valid-token count."""
        dev = self.device
        B = len(cre_tokens)
        C = np.array([t.shape[0] for t in cre_tokens]); G = np.array([t.shape[0] for t in gene_tokens])

        def stage(tok_list, mask_list, known):
            tok = torch.cat([t.reshape(-1, t.shape[-1]) for t in tok_list]).to(torch.int32)
            msk = torch.cat([m.reshape(-1, m.shape[-1]) for m in mask_list]).to(torch.uint8)
            if tok.is_cuda:
                ln = known if known is not None else ops.window_lengths(msk).cpu().numpy().astype(np.int64)
                return tok, msk, ln
            ln = known if known is not None else (msk == 0).sum(1).numpy().astype(np.int64)
            return tok.pin_memory().to(dev, non_blocking=True), msk.pin_memory().to(dev, non_blocking=True), ln

        s = {}
        s["ctok"], s["cmsk"], s["clens"] = stage(cre_tokens, cre_masks, None if lens is None else lens[0])
        s["gtok"], s["gmsk"], s["glens"] = stage(gene_tokens, gene_masks, None if lens is None else lens[1])
        for tag, ln, W in (("c", s["clens"], self.cre_tok), ("g", s["glens"], self.gene_tok)):
            s[tag + "_cu_tok"] = ops.cu_seqlens(ln, dev)
            s[tag + "_plan_tok"] = AttnPlan(ln, dev, W.hd)
        g_off = np.concatenate([[0], np.cumsum(G)])
        gene_rows = [np.arange(g_off[g], g_off[g + 1], dtype=np.int64) for g in range(B)]
        return self._prepare_seq2gene(s, C, gene_rows, int(G.sum()), tissues, ref_labels, cre_token_position,
                                      gene_token_position)

    def prepare_shared(self, cre_rows, gene_rows, n_gene_chunks, tissues, ref_labels):
        """Slab of items whose windows are encoded once and shared between items (saturation mutagenesis: every
        mutant of a gene reuses the reference item's unchanged windows).  cre_rows / gene_rows: one int array per item,
        the rows of the item's CRE windows / gene chunks (in batch order) in the pooled outputs of the unique windows;
        n_gene_chunks = number of unique gene chunks.  A window's pooled vector depends on its tokens alone, so the
        result of an item equals its result in a slab built by `prepare` from its own tokens.  -> a slab for
        run_pooled(slab, unique CRE pooled rows, unique gene pooled rows)."""
        C = np.array([len(r) for r in cre_rows])
        s = {"cre_rows": torch.from_numpy(np.concatenate(cre_rows).astype(np.int64)).to(self.device, non_blocking=True)}
        return self._prepare_seq2gene(s, C, [np.asarray(r, np.int64) for r in gene_rows], int(n_gene_chunks), tissues,
                                      ref_labels)

    def _prepare_seq2gene(self, s, C, gene_rows, n_gene_chunks, tissues, ref_labels, cre_token_position=None,
                          gene_token_position=None):
        """Index structures of stages 3-4: gene_rows[g] = rows of gene g's chunk embeddings in gene_map's output."""
        dev = self.device
        B = len(gene_rows)
        G = np.array([len(r) for r in gene_rows])
        T = np.array([len(t) for t in tissues])
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev, non_blocking=True)
        s.update({"B": B, "C": C, "G": G, "T": T, "n_gene_chunks": n_gene_chunks})
        # gene stream layout: per (gene, tissue): [registry(tissue); the gene's chunk embeddings]
        idx, seq_lens = [], []
        for g in range(B):
            tis = tissues[g].detach().cpu().numpy().astype(np.int64).reshape(-1)
            body = gene_rows[g]
            for t in tis:
                idx.append(np.concatenate([[-(t + 1)], body]))
                seq_lens.append(G[g] + 1)
        idx = np.concatenate(idx)
        seq_lens = np.asarray(seq_lens)
        s["Mg"] = int(idx.shape[0])
        s["gene_idx"] = up(idx, np.int32)
        s["plan_gself"] = AttnPlan(seq_lens, dev, self.w.hd)            # one sequence per (gene, tissue): self-attention
        s["plan_gcross"] = AttnPlan(T * (G + 1), dev, self.w.hd, k_lens=C)   # per gene: stacked tissue queries x its CREs
        s["plan_cself"] = AttnPlan(C, dev, self.w.hd)
        s["row_seq"] = up(np.repeat(np.arange(B), C), np.int32)
        lab = torch.cat([l.reshape(-1) for l in ref_labels]).detach().cpu().numpy().astype(np.int64)
        counts = np.zeros((B, NUM_REF_CRES), np.float64)
        np.add.at(counts, (np.repeat(np.arange(B), C), lab), 1.0)
        with np.errstate(divide="ignore"):
            s["logc"] = up(np.log(counts), np.float32)
        reg_rows = np.cumsum(seq_lens) - seq_lens
        s["reg_idx"] = up(reg_rows, np.int32)
        # Last gene layer: only the registry rows (and the VEP token rows) of its output are ever read, so everything
        # after the K/V projection of its self-attention runs on those rows alone (exact).  `need` lists them; each is a
        # one-row query tile against its own sequence (ALiBi position = its offset), and the rows of one gene form
        # query tiles of the stacked cross-attention.
        n_seq = len(seq_lens)
        need_seq = np.arange(n_seq); need_off = np.zeros(n_seq, np.int64)
        if gene_token_position is not None:
            gp = np.repeat(np.asarray([int(p) for p in gene_token_position]) + 1, T)      # +1: registry token
            need_seq = np.concatenate([need_seq, np.arange(n_seq)]); need_off = np.concatenate([need_off, gp])
        s["last_rows"] = up(reg_rows[need_seq] + need_off, np.int32)
        s["n_need"] = int(len(need_seq))
        k = np.arange(len(need_seq))
        s["plan_last_self"] = AttnPlan(None, dev, self.w.hd, units=np.stack(
            [k, np.ones_like(k), reg_rows[need_seq], seq_lens[need_seq], need_off], 1))
        gene_of = np.repeat(np.arange(B), T)[need_seq]                                  # gene of every needed row
        cu_cre_np = np.concatenate([[0], np.cumsum(C)])
        units = []
        start = 0
        for i in range(1, len(k) + 1):                                                 # runs of one gene, <= 128 rows
            if i == len(k) or gene_of[i] != gene_of[start] or i - start == 128:
                g = gene_of[start]
                units.append([start, i - start, cu_cre_np[g], C[g], 0])
                start = i
        s["plan_last_cross"] = AttnPlan(None, dev, self.w.hd, units=np.asarray(units))
        if gene_token_position is not None:
            s["gene_pos_idx"] = up(reg_rows + gp, np.int32)                                 # (:665-666)
        if cre_token_position is not None:
            c_off = np.concatenate([[0], np.cumsum(C)])[:-1]
            s["cre_pos_idx"] = up(np.repeat(c_off + np.asarray([int(p) for p in cre_token_position]), T), np.int32)
        return s

    # ---------------------------------------------------------------- device work for one prepared slab
    @torch.no_grad()
    def run(self, s):
        """-> dict(pred fp32 [sum T], emb fp32 [sum T, D], T list, optional token embeddings); device tensors."""
        return self.run_pooled(s, *self.pool_windows(s))

    @torch.no_grad()
    def pool_windows(self, s):
        """Stage 2 of a slab built by `prepare`: the window encoders.  -> (CRE pooled bf16 [sum C, d], gene pooled bf16
        [sum G, d])."""
        cre_pooled = self.seq2reg(self.cre_tok, s["ctok"], s["cmsk"], s["clens"], s["c_cu_tok"], s["c_plan_tok"])
        gene_pooled = self.seq2reg(self.gene_tok, s["gtok"], s["gmsk"], s["glens"], s["g_cu_tok"], s["g_plan_tok"])
        return cre_pooled, gene_pooled

    @torch.no_grad()
    def run_pooled(self, s, cre_pooled, gene_pooled):
        """Stages 3-4 of a slab from its pooled window vectors (pool_windows, or the unique windows of a slab built by
        prepare_shared).  -> the dict of `run`."""
        w, ws = self.w, self.ws
        D, H, hd = w.D, w.H, w.hd
        nC, Mg = int(s["C"].sum()), s["Mg"]
        if "cre_rows" in s:                                  # shared windows: each item's CRE rows (1 KB per row)
            cre_pooled = cre_pooled.index_select(0, s["cre_rows"])
        if COARSE and ops.PROFILER is None and w.cre_map is not None:
            return self._run_coarse(s, cre_pooled, gene_pooled)
        if w.cre_map is None:
            raise NotImplementedError("token_dim == emb_dim (no cre_map) is not wired on the B200 path")
        # Both streams are row-centred (see the module docstring): cx / gx hold x - pivot_r, cxb / gxb their bf16 mirrors.
        # The gene stack's cross-attention reads the RAW CRE stream (the context is not normalised, layers.py:142-150):
        # `ctx` is its bf16 copy, written by the cre_map epilogue for gene layer 0 and rebuilt (x + pivot) after every
        # CRE layer, right before the K/V projection that consumes it on the same stream.
        ctx = ws.get("cre_ctx", (nC, D), torch.bfloat16)
        cxb = ws.get("cxb", (nC, D), torch.bfloat16)
        cx = ops.gemm(cre_pooled, w.cre_map.w, EPI_BIAS_F32, bias=w.cre_map.b, out=ws.get("cx", (nC, D), torch.float32),
                      out2=ctx)
        cpiv, cxs = ops.center_rows(cx, ws.get("cpiv", (nC,), torch.float32), ws.get("cxs0", (nC, 1, 2), torch.float32), cxb)
        gene_emb = ops.gemm(gene_pooled, w.gene_map.w, EPI_BIAS_F32, bias=w.gene_map.b)
        gx, _ = ops.gather_rows(gene_emb, w.registry, s["gene_idx"])
        gxb = ws.get("gxb", (Mg, D), torch.bfloat16)
        gpiv, gxs = ops.center_rows(gx, ws.get("gpiv", (Mg,), torch.float32), ws.get("gxs0", (Mg, 1, 2), torch.float32), gxb)
        st = {"g": gxs, "c": cxs}                                      # current row statistics of each stream
        # K/V of the gene stack's cross-attention, one buffer per gene layer: they depend on the CRE stack only, so the
        # projection of layer i+1 is issued on the CRE stream right behind CRE layer i
        kvs = [ws.get(f"g_kv{i}", (nC, 2 * D), torch.bfloat16) for i in range(w.NL)]

        def gene_self(qkv, out):
            s["plan_gself"].run(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H, hd, w.slopes, out)

        def cre_self(qkv, out):
            s["plan_cself"].run(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H, hd, w.slopes, out)

        def project_kv(i):
            L = w.gene_layers[i]
            ops.gemm(ctx, L["kv"].w, EPI_BIAS_BF16, bias=L["kv"].b, out=kvs[i])          # shared by every tissue copy

        def gene_layer(i):
            L, kv = w.gene_layers[i], kvs[i]

            def cross(q, out):
                s["plan_gcross"].run(q, kv[:, :D], kv[:, D:], H, hd, None, out)
            st["g"] = self._layer(L, gx, gxb, st["g"], Mg, gene_self, cross, "g")

        def cre_layer(i):
            L = w.cre_layers[i]

            def cross(q, out):
                ops.label_attention(q, L["kv9"], s["logc"], s["row_seq"], H, hd, out=out)
            st["c"] = self._layer(L, cx, cxb, st["c"], nC, cre_self, cross, "c")
            ops.uncenter_rows(cx, cpiv, want_f32=False, out_bf16=ctx)                    # context of gene layer i + 1

        # The CRE stack does not depend on the gene stack (gene layer i+1 reads the output of CRE layer i, never the
        # other way round): it runs on a second CUDA stream and its short kernels (8 192 rows) fill the tails of the
        # gene stack's persistent kernels.  Gene layer i+1 waits for the event recorded after CRE layer i.
        prune_last = "plan_last_self" in s and w.NL > 1
        two_streams = self.device.type == "cuda" and CRE_STREAM and w.NL > 1
        done = []
        if two_streams:
            main = torch.cuda.current_stream(self.device)
            if getattr(self, "_cre_stream", None) is None:
                self._cre_stream = torch.cuda.Stream(self.device)
            side = self._cre_stream
            for t in (s["logc"], s["row_seq"], *s["plan_cself"].device_tensors()):
                t.record_stream(side)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                project_kv(0)
                ev = torch.cuda.Event(); ev.record(side)
                done.append(ev)
                for i in range(w.NL - 1):
                    cre_layer(i)
                    project_kv(i + 1)
                    ev = torch.cuda.Event(); ev.record(side)
                    done.append(ev)
        for i in range(w.NL):                                  # done[i]: context and K/V of gene layer i are ready
            if two_streams:
                main.wait_event(done[i])
            else:
                if i > 0:
                    cre_layer(i - 1)
                project_kv(i)
            if i < w.NL - 1 or not prune_last:
                gene_layer(i)
        n_reg = s["reg_idx"].numel()
        if prune_last:
            last = self._gene_layer_last(w.gene_layers[w.NL - 1], s, gx, gxb, st["g"], kvs[w.NL - 1])
            last, last_bf = ops.uncenter_rows(last, gpiv, idx=s["last_rows"], want_bf16=True)
            emb, emb_bf = last[:n_reg], last_bf[:n_reg]
        else:
            last = None
            emb, _ = ops.gather_rows(gx, None, s["reg_idx"])
            emb, emb_bf = ops.uncenter_rows(emb, gpiv, idx=s["reg_idx"], want_bf16=True)

        # ---- registry rows -> embeddings -> head ----
        h1 = ops.gemm(emb_bf, w.h0.w, EPI_BIAS_F32, bias=w.h0.b)
        h1n = ops.layernorm(h1, w.hn.g, w.hn.b, gelu=True)
        h2 = ops.gemm(h1n, w.h4.w, EPI_BIAS_GELU_BF16, bias=w.h4.b)
        pred = ops.head_out(h2, w.h6_w, w.h6_b, softplus=True)
        out = {"pred": pred, "emb": emb, "T": s["T"].tolist()}
        if "gene_pos_idx" in s:
            if last is not None:
                out["gene_token_embedding"] = last[n_reg:]
            else:
                t, _ = ops.gather_rows(gx, None, s["gene_pos_idx"])
                out["gene_token_embedding"], _ = ops.uncenter_rows(t, gpiv, idx=s["gene_pos_idx"])
        if "cre_pos_idx" in s:
            t, _ = ops.gather_rows(cx, None, s["cre_pos_idx"])
            out["cre_token_embedding"], _ = ops.uncenter_rows(t, cpiv, idx=s["cre_pos_idx"])
        return out

    def _run_coarse(self, s, cre_pooled, gene_pooled):
        """Stages 3-4 of a prepared slab through vf_seq2gene_forward (layer loop in the library)."""
        import ctypes as C
        from . import _abi, _lib
        w = self.w
        if "_abi_slab" not in s:
            tab = lambda k: (s[k].slots.table.data_ptr(), s[k].slots.n_items)
            n_reg = s["reg_idx"].numel()
            cpos = s.get("cre_pos_idx")
            s["_abi_slab"] = _abi.Seq2GeneSlab(
                int(s["C"].sum()), s["n_gene_chunks"], s["Mg"], n_reg, s["n_need"], 0,
                s["gene_idx"].data_ptr(), s["row_seq"].data_ptr(), s["logc"].data_ptr(), s["last_rows"].data_ptr(),
                None if cpos is None else cpos.data_ptr(), *tab("plan_gself"), *tab("plan_gcross"), *tab("plan_cself"),
                *tab("plan_last_self"), *tab("plan_last_cross"))
        slab = s["_abi_slab"]
        slab.single_stream = 0 if (CRE_STREAM and self.device.type == "cuda") else 1
        nbytes = int(_lib.lib().vf_seq2gene_workspace_bytes(C.addressof(w.abi()), C.addressof(slab)))
        pred, emb, gtok, ctok = ops.seq2gene_forward(w.abi(), slab, cre_pooled, gene_pooled,
                                                     self.ws.get("coarse_g", (nbytes,), torch.uint8), slab.n_reg,
                                                     slab.n_need - slab.n_reg, w.D, "cre_pos_idx" in s)
        out = {"pred": pred, "emb": emb, "T": s["T"].tolist()}
        if "gene_pos_idx" in s:
            out["gene_token_embedding"] = gtok
        if ctok is not None:
            out["cre_token_embedding"] = ctok
        return out

    def forward_tokens(self, cre_tokens, cre_masks, gene_tokens, gene_masks, tissues, ref_labels, **kw):
        return self.run(self.prepare(cre_tokens, cre_masks, gene_tokens, gene_masks, tissues, ref_labels, **kw))
