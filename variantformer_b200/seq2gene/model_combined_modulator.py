"""Seq2GenePredictorCombinedModulator — the configured `model_class` (configs/vf_model.yaml:10) behind the
reference's signatures (seq2gene/model_combined_modulator.py:411-435 ctor, :540-552 forward, :857 predict_step,
:909 variant_prediction).  All tensor math runs in libvf_b200.so through variantformer_b200.engine.Engine.
"""
import logging
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn

from .._params import Affine, Table
from ..utils.functions import precision2dtype
from .modules.layers import (AddContext, ContextFlashAttentionEncoderLayer, ContextFlashCrossAttentionEncoderLayer,
                             FlashAttentionEncoderLayer, MultiRegistry, StartToken, TissueExpressionHeads)

logger = logging.getLogger(__name__)
NUM_REF_CRES = 9


class _HParams(dict):
    __getattr__ = dict.get


class CombinedModulator(nn.Module):
    """Interleaved CRE / gene encoder stacks: gene_0(g, cre_in); for i: cre_i(cre, label ctx); gene_{i+1}(g, cre)."""

    def __init__(self, emb_dim, num_heads, num_layers, use_alibi, mlp_dout, use_context, num_ref_cres=None,
                 only_cross_attention=True, use_res=False, cross_alibi=False, flash_attn_3=False):
        """Layer variants exactly as the reference builds them (model_combined_modulator.py:69-135): CRE layers with the
        label cross-attention (use_context) or self-attention only; gene layers with self + cross attention or cross
        attention only (only_cross_attention); use_res adds the gene input after every gene layer.  The batched engine
        implements the vf_model.yaml combination (use_context, full gene layers, no use_res); the other combinations
        run layer by layer through `forward`."""
        super().__init__()
        if flash_attn_3:
            raise NotImplementedError("flash_attn_3=True is not implemented (the reference itself rejects it for cross attention)")
        self.emb_dim, self.num_heads, self.num_layers = emb_dim, num_heads, num_layers
        self.use_context, self.only_cross_attention, self.use_res, self.cross_alibi = \
            use_context, only_cross_attention, use_res, cross_alibi
        if use_context:
            assert num_ref_cres is not None, "num_ref_cres must be provided when use_context is True"
            self.second_level_context_embedding = Table(num_ref_cres, emb_dim)
            mk_cre = lambda: ContextFlashAttentionEncoderLayer(d_model=emb_dim, nhead=num_heads, batch_first=True,
                                                               use_alibi=use_alibi, mlp_dout=mlp_dout)
        else:
            mk_cre = lambda: FlashAttentionEncoderLayer(d_model=emb_dim, nhead=num_heads, batch_first=True,
                                                        use_alibi=use_alibi, mlp_dout=mlp_dout)
        if only_cross_attention:
            mk_gene = lambda: ContextFlashCrossAttentionEncoderLayer(d_model=emb_dim, nhead=num_heads, batch_first=True,
                                                                     use_alibi=use_alibi, mlp_dout=mlp_dout,
                                                                     cross_alibi=cross_alibi)
        else:
            mk_gene = lambda: ContextFlashAttentionEncoderLayer(d_model=emb_dim, nhead=num_heads, batch_first=True,
                                                                use_alibi=use_alibi, mlp_dout=mlp_dout,
                                                                cross_alibi=cross_alibi)
        self.cre_layers = nn.ModuleList([mk_cre() for _ in range(num_layers - 1)])
        self.gene_layers = nn.ModuleList([mk_gene() for _ in range(num_layers)])

    @torch.no_grad()
    def forward(self, cre_x, gene_x, context=None, cre_padding_mask=None, gene_padding_mask=None,
                context_padding_mask=None, precision=None, cre_token_position=None, gene_token_position=None):
        """model_combined_modulator.py:137-148: cre_x [batch, cre_seq_len, emb_dim], gene_x [batch, gene_seq_len, emb_dim],
        context int [batch, cre_seq_len] (reference cCRE labels), masks True = padding -> (gene_output [batch,
        gene_seq_len, emb_dim], gene_token_embedding, cre_token_embedding).  Layer by layer through the layers' own
        forwards; the batched engine (Seq2GenePredictorCombinedModulator.forward) is the fast path."""
        from ..layer_ops import combined_modulator_forward
        assert context is not None or not self.use_context, \
            "context (reference cCRE labels) is required when use_context is True"
        return combined_modulator_forward(self, cre_x, gene_x, context, cre_padding_mask, gene_padding_mask,
                                          context_padding_mask, cre_token_position, gene_token_position)


class Seq2GenePredictorCombinedModulator(nn.Module):
    def __init__(self, num_tissues: int, emb_dim: int, gene_emb_dim: int, num_heads: int, num_layers: int,
                 use_alibi: bool = True, mlp_dout: float = 0.1, weight_decay: float = 0.0, learning_rate: float = 1e-4,
                 lr_scale: float = 1, use_context: bool = False, token_dim: int = 128, cre_tokenizer=None,
                 gene_tokenizer=None, cre_tokenizer_train_mode="val", cre_tokenizer_val_mode="val",
                 gene_tokenizer_train_mode="val", gene_tokenizer_val_mode="val", tissues: list = None,
                 optimizer="adam", gene_pooling="mean", flash_attn_3=False, **kwargs):
        super().__init__()
        assert gene_pooling in ["mean", "max", "start_token", "multi_registry"], \
            "gene_pooling must be one of mean, max, start_token, or multi_registry"
        if gene_pooling == "mean":
            # the reference's own 'mean' branch never reduces over the sequence axis (pool_outputs :372-377 returns a
            # [batch, seq, emb] tensor that the head cannot consume): there is no behaviour to reproduce
            raise NotImplementedError("gene_pooling='mean' is broken upstream (pool_outputs does not reduce); not implemented")
        self.hparams = _HParams(dict(num_tissues=num_tissues, emb_dim=emb_dim, gene_emb_dim=gene_emb_dim,
                                     num_heads=num_heads, num_layers=num_layers, use_alibi=use_alibi, mlp_dout=mlp_dout,
                                     use_context=use_context, token_dim=token_dim, gene_pooling=gene_pooling, **kwargs))
        self.precision = None
        self.gene_pooling = gene_pooling
        self.start_tkn = (MultiRegistry(num_tissues, emb_dim) if gene_pooling == "multi_registry" else
                          StartToken(emb_dim) if gene_pooling == "start_token" else None)
        self.add_context_to_cres = kwargs.get("add_context_to_cres", False)
        self.add_context = AddContext(num_tissues, emb_dim) if self.add_context_to_cres else None
        self.cre_tokenizer, self.gene_tokenizer = cre_tokenizer, gene_tokenizer
        self.emb_dim, self.use_context, self.tissues = emb_dim, use_context, tissues
        self.use_res = kwargs.get("use_res", False)
        self.loss_fn = kwargs.get("loss_fn", "poisson")
        self.use_bigger_head = kwargs.get("use_bigger_head", False)
        self.multi_head = kwargs.get("multi_head", True)
        self.only_cross_attention = kwargs.get("only_cross_attention", True)
        self.cross_alibi = kwargs.get("cross_alibi", False) and use_alibi
        self.gene_map = Affine(emb_dim, gene_emb_dim)
        if token_dim != emb_dim:
            self.cre_map = Affine(emb_dim, token_dim)
        self.combined_modulator = CombinedModulator(
            emb_dim=emb_dim, num_heads=num_heads, num_layers=num_layers, use_alibi=use_alibi, mlp_dout=mlp_dout,
            use_context=use_context, num_ref_cres=NUM_REF_CRES if use_context else None,
            only_cross_attention=self.only_cross_attention, use_res=self.use_res, cross_alibi=self.cross_alibi,
            flash_attn_3=flash_attn_3)
        self.tissue_heads = TissueExpressionHeads(emb_dim, num_tissues, use_bigger_head=self.use_bigger_head,
                                                  multi_head=self.multi_head, mlp_dout=mlp_dout, loss_fn=self.loss_fn,
                                                  head_type=kwargs.get("head_type", "mlp"))
        self.vep = False
        self.trainer = None
        self._engine = None

    # -- engine plumbing ---------------------------------------------------------------------------
    def engine(self):
        from ..engine import Engine
        dev = self.gene_map.weight.device
        if self._engine is None or self._engine.device != dev:
            if dev.type != "cuda":
                raise RuntimeError("this model runs on a B200 only: call .to('cuda') first (there is no CPU path)")
            cfg = dict(self.hparams)
            self._engine = Engine(self.state_dict(), cfg, dict(self.cre_tokenizer.hparams), device=dev,
                                  gene_seq2reg_hp=dict(self.gene_tokenizer.hparams))
        return self._engine

    def load_state_dict(self, *a, **k):
        self._engine = None
        return super().load_state_dict(*a, **k)

    def _apply(self, fn, *a, **k):
        self._engine = None
        return super()._apply(fn, *a, **k)

    def _check_precision(self):
        """model_combined_modulator.py:736-744: bf16/fp16 trainers run the mixed path; anything else asked the
        reference for its fp16-cast attention path, which this implementation does not reproduce."""
        try:
            p = precision2dtype(self.trainer.precision)
        except Exception:
            p = torch.bfloat16 if self.trainer is None else torch.float32
        if p not in (torch.float16, torch.bfloat16):
            raise NotImplementedError("the B200 path computes in bf16 (fp32 accumulate); use precision='bf16-mixed'")

    # -- reference forward signature ----------------------------------------------------------------
    @torch.no_grad()
    def forward(self, inp, attention_mask, tissue_vector, cre_context, strand, gene_embedding, gene_att_mask,
                return_embedding=False, get_all=False, **kwargs):
        """inp / gene_embedding: lists of int64 [n,1,L]; masks bool (True = pad); tissue_vector: list of [T_i];
        cre_context: list of ref-cCRE label ids [C_i].  -> (pred [sum T,1], donors[, emb [sum T, D], gene_token_emb,
        cre_token_emb]) exactly like the reference (:705-720)."""
        self._check_precision()
        if not self._engine_variant():
            return self._forward_generic(inp, attention_mask, tissue_vector, cre_context, gene_embedding, gene_att_mask,
                                         return_embedding, **kwargs)
        sq = lambda xs: [x[:, 0, :] if x.dim() == 3 else x for x in xs]
        cpos, gpos = kwargs.get("cre_token_position"), kwargs.get("gene_token_position")
        out = self.engine().forward_tokens(
            sq(inp), sq(attention_mask), sq(gene_embedding), sq(gene_att_mask), list(tissue_vector), list(cre_context),
            cre_token_position=None if cpos is None else [int(p) for p in cpos],
            gene_token_position=None if gpos is None else [int(p) for p in gpos])
        donors = list(range(len(inp)))
        emb = out["emb"]
        if kwargs.get("only_embedding", False):
            return {"embedding": emb, "donors": donors}
        pred = out["pred"].unsqueeze(1)
        if not return_embedding:
            return pred, donors
        zeros = lambda: torch.zeros(emb.shape[0], emb.shape[1], device=emb.device)
        return (pred, donors, emb, out.get("gene_token_embedding", zeros()), out.get("cre_token_embedding", zeros()))

    def _engine_variant(self):
        """True for the architecture the batched engine implements (configs/vf_model.yaml): label-context CRE layers, full
        gene layers, per-tissue registry token, shared bigger head, no use_res / cross_alibi / add_context_to_cres."""
        cm = self.combined_modulator
        return (self.gene_pooling == "multi_registry" and cm.use_context and not cm.only_cross_attention and
                not cm.use_res and not cm.cross_alibi and not self.add_context_to_cres and
                not self.cre_tokenizer.use_context and not self.gene_tokenizer.use_context)

    @torch.no_grad()
    def _forward_generic(self, inp, attention_mask, tissue_vector, cre_context, gene_embedding, gene_att_mask,
                         return_embedding=False, **kwargs):
        """The reference's forward (model_combined_modulator.py:540-720) step by step for the configurations the batched
        engine does not cover (gene_pooling start_token / max, add_context_to_cres, only_cross_attention, use_res,
        use_context=False, cross_alibi): window encoders, cre_map / gene_map, per-tissue replication, AddContext,
        prepare_input, CombinedModulator.forward, pool_outputs, head — every layer through the modules' own forwards
        (same kernels).  No tissue de-duplication here: this path serves correctness, not the benchmark."""
        from .. import ops
        from .._lib import EPI_BIAS_F32
        dev = self.gene_map.weight.device
        D = self.emb_dim

        def encode(tok_list, mask_list, labels, tokenizer):
            """-> padded [n_items, max_windows, d], mask [n_items, max_windows] (True = pad)"""
            embs = []
            for i, (t, m) in enumerate(zip(tok_list, mask_list)):
                t = t if t.dim() == 3 else t[:, None, :]
                m = m if m.dim() == 3 else m[:, None, :]
                ctx = None if labels is None else torch.as_tensor(labels[i]).to(dev)
                embs.append(tokenizer(t.to(dev), m.to(dev), None, context=ctx, only_embed=True)[:, 0, :])
            n = max(e.shape[0] for e in embs)
            x = torch.zeros(len(embs), n, embs[0].shape[1], device=dev)
            mask = torch.ones(len(embs), n, dtype=torch.bool, device=dev)
            for i, e in enumerate(embs):
                x[i, :e.shape[0]] = e; mask[i, :e.shape[0]] = False
            return x, mask

        def linear(x, lin):
            y = ops.gemm(ops.cast_bf16(x.reshape(-1, x.shape[-1]).float().contiguous()),
                         lin.weight.to(torch.bfloat16).contiguous(), EPI_BIAS_F32, bias=lin.bias.float().contiguous())
            return y.view(*x.shape[:-1], -1)
        cre_labels = list(cre_context) if self.cre_tokenizer.use_context else None
        x, mask_c = encode(inp, attention_mask, cre_labels, self.cre_tokenizer)
        gene_labels = [torch.zeros(g.shape[0], dtype=torch.long) for g in gene_embedding] \
            if self.gene_tokenizer.use_context else None
        xg, mask_g = encode(gene_embedding, gene_att_mask, gene_labels, self.gene_tokenizer)
        n_c = x.shape[1]
        context = torch.zeros(len(inp), n_c, dtype=torch.long, device=dev)
        for i, c in enumerate(cre_context):
            context[i, :len(c)] = torch.as_tensor(c).to(dev).long()
        if x.shape[-1] != D:
            x = linear(x, self.cre_map)
        xg = linear(xg, self.gene_map)
        T = [len(t) for t in tissue_vector]
        rep = torch.repeat_interleave(torch.arange(len(T), device=dev), torch.tensor(T, device=dev))
        x, mask_c, context, xg, mask_g = x[rep], mask_c[rep], context[rep], xg[rep], mask_g[rep]
        tv = torch.cat([torch.as_tensor(t).reshape(-1) for t in tissue_vector]).to(dev).long()[:, None]
        cpos, gpos = kwargs.get("cre_token_position"), kwargs.get("gene_token_position")
        rp = lambda p: None if p is None else torch.repeat_interleave(
            torch.as_tensor([int(v) for v in p], device=dev), torch.tensor(T, device=dev))
        cpos, gpos = rp(cpos), rp(gpos)
        if gpos is not None and self.start_tkn is not None:
            gpos = gpos + 1
        if self.add_context_to_cres:
            x = self.add_context(x, tv)
        g = xg
        if self.gene_pooling == "start_token":
            g = torch.cat((self.start_tkn(g), g), dim=1)
        elif self.gene_pooling == "multi_registry":
            g, _ = self.start_tkn(g, tv)
        if self.start_tkn is not None:
            mask_g = torch.cat((torch.zeros(mask_g.shape[0], 1, dtype=torch.bool, device=dev), mask_g), dim=1)
        g, gtok, ctok = self.combined_modulator(cre_x=x, gene_x=g, context=context, cre_padding_mask=mask_c,
                                                gene_padding_mask=mask_g, context_padding_mask=mask_c,
                                                cre_token_position=cpos, gene_token_position=gpos)
        if self.gene_pooling == "max":
            g = g.masked_fill(mask_g[:, :, None], float("-inf")).max(dim=1).values
        else:
            g = g[:, 0, :]
        donors = list(range(len(inp)))
        if kwargs.get("only_embedding", False):
            return {"embedding": g, "donors": donors}
        pred = self.tissue_heads(g.contiguous(), tv)
        return (pred, donors, g, gtok, ctok) if return_embedding else (pred, donors)

    def predict_step(self, batch, batch_idx, dataloader_idx=None):
        """:857-907 — one batch of genes -> per-gene numpy predictions and registry-token embeddings."""
        if self.vep:
            return self.variant_prediction(batch)
        pred, donors, embd, _, _ = self(batch["cre_sequences"], batch["cre_attention_masks"], batch["tissue_context"],
                                        batch["ref_cre_labels"], batch["strand_val"], batch["gene_embeddings"],
                                        batch["gene_attention_masks"], return_embedding=True)
        assert len(donors) == len(batch["cre_sequences"]), "Number of donors and CREs do not match"
        pred = pred.cpu().float().numpy(); embd = embd.cpu().float().numpy()
        preds, embs, s = [], [], 0
        for i in donors:
            e = s + len(batch["tissue_context"][i])
            preds.append(pred[s:e]); embs.append(embd[s:e]); s = e
        return {"pred_gene_exp": preds, "embeddings": embs, "batch_idx": batch_idx, "dataloader_idx": dataloader_idx}

    @torch.no_grad()
    def predict_cre_attention(self, batch):
        """predict_step with the gene -> CRE cross-attention maps of every prediction (Engine.run_pooled):
        -> {"pred_gene_exp": [np (T_i, 1)], "cre_attention": [np fp32 (T_i, num_layers, num_heads, C_i)]}, CREs in
        the batch order of the item.  Predictions are bit-identical to predict_step's."""
        self._check_precision()
        if not self._engine_variant():
            raise NotImplementedError("cross-attention maps are implemented for the configs/vf_model.yaml architecture")
        sq = lambda xs: [x[:, 0, :] if x.dim() == 3 else x for x in xs]
        out = self.engine().forward_tokens(sq(batch["cre_sequences"]), sq(batch["cre_attention_masks"]),
                                           sq(batch["gene_embeddings"]), sq(batch["gene_attention_masks"]),
                                           list(batch["tissue_context"]), list(batch["ref_cre_labels"]),
                                           cre_attention=True)
        pred = out["pred"].cpu().numpy(); flat = out["cre_attention"].cpu().numpy(); off = out["cre_attention_off"]
        L, H = self.combined_modulator.num_layers, self.combined_modulator.num_heads
        preds, maps, r = [], [], 0
        for g, tis in enumerate(batch["tissue_context"]):
            T, C = len(tis), batch["cre_sequences"][g].shape[0]
            preds.append(pred[r:r + T, None])
            maps.append(np.stack([flat[off[r + t]:off[r + t] + L * H * C].reshape(L, H, C) for t in range(T)]))
            r += T
        return {"pred_gene_exp": preds, "cre_attention": maps}

    def variant_prediction(self, batch):
        """:909-1004 — (ref, het, hom) triplet; the three samples run as ONE batched pass instead of three
        sequential batch-1 forwards (identical results: items are independent)."""
        x = batch["cre_sequences"]
        n = len(x)
        if n == 0:
            return {"pred_gene_exp": [], "embd": [], "variant_type": batch["variant_type"],
                    "gene_token_embedding": [], "cre_token_embedding": []}
        cpos, gpos = batch["cre_token_position"], batch["gene_token_position"]
        assert len(cpos) == 3 and len(gpos) == 3, "there should be 3 samples in the batch for ref, het, hom"
        cpos = None if torch.isnan(torch.as_tensor(cpos, dtype=torch.float)).any() else cpos
        gpos = None if torch.isnan(torch.as_tensor(gpos, dtype=torch.float)).any() else gpos
        pred, _, embd, gtok, ctok = self(x, batch["cre_attention_masks"], batch["tissue_context"], batch["ref_labels"],
                                         batch["strand"], batch["gene_embeddings"], batch["gene_attention_masks"],
                                         return_embedding=True, cre_token_position=cpos, gene_token_position=gpos)
        arrs = [t.cpu().float().numpy() for t in (pred, embd, gtok, ctok)]
        outs = [[], [], [], []]
        s = 0
        for i in range(n):
            e = s + len(batch["tissue_context"][i])
            for o, a in zip(outs, arrs):
                o.append(a[s:e])
            s = e
        return {"pred_gene_exp": outs[0], "embd": outs[1], "variant_type": batch["variant_type"],
                "gene_token_embedding": outs[2], "cre_token_embedding": outs[3]}


def attach_trainer(model, precision="bf16-mixed"):
    """Mimic Lightning's `model.trainer` attribute (read at model_combined_modulator.py:736)."""
    model.trainer = SimpleNamespace(precision=precision)
    return model
