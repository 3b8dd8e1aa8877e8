"""Gene -> CRE cross-attention maps on the GPU: vf_cross_attention_probs against float64 on the same bf16 operands, the
engine's maps against the fp32 oracle, bit-identity of every other output, coarse vs fine engine, batching invariance,
and VCFProcessor.cre_attention."""
import math

import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import model_fp32  # noqa: E402  (checker only)
from tests.common import GOLD_CFG, GOLD_HP, GOLD_SEED, load_model_golden, parity_report, synth_batch  # noqa: E402
from variantformer_b200 import _lib, ops  # noqa: E402
from variantformer_b200 import engine as engine_mod  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.utils import random_init  # noqa: E402

SENTINEL = -12345.5
U = 2.0 ** -24                                       # fp32 unit roundoff


# ---- kernel ------------------------------------------------------------------------------------------------------------
def _probs_case(hd, heads, key_counts, query_counts, seed):
    """Groups of the given sizes; q rows scattered through a [n, 3D] buffer (ldq = 3D, middle third), K the first half of
    a [keys, 2D] buffer (ldk = 2D); output blocks of 2 layers per query with sentinel gaps between them."""
    g = torch.Generator().manual_seed(seed)
    D = heads * hd
    nq_tot, nk_tot = sum(query_counts), sum(key_counts)
    qbuf = torch.randn(nq_tot + 17, 3 * D, generator=g).to(torch.bfloat16).cuda()
    kbuf = (torch.randn(nk_tot, 2 * D, generator=g) * 1.5).to(torch.bfloat16).cuda()
    q, k = qbuf[:, D:2 * D], kbuf[:, :D]
    q_rows = torch.randperm(nq_tot + 17, generator=g)[:nq_tot].to(torch.int32)
    group_q = np.stack([np.cumsum(query_counts) - query_counts, query_counts], 1).astype(np.int32)
    group_k = np.stack([np.cumsum(key_counts) - key_counts, key_counts], 1).astype(np.int32)
    sizes = np.repeat(key_counts, query_counts) * 2 * heads
    gap = 13
    off = (np.cumsum(sizes + gap) - sizes).astype(np.int64)
    total = int(off[-1] + sizes[-1] + gap)
    return dict(q=q, k=k, q_rows=q_rows.cuda(), group_q=torch.from_numpy(group_q).cuda(),
                group_k=torch.from_numpy(group_k).cuda(), off=torch.from_numpy(off).cuda(), off_h=off, total=total,
                q_rows_h=q_rows.numpy(), gq=group_q, gk=group_k, heads=heads, hd=hd)


def _ref(c, i, g, scale_mult=1.0, drop_last=False):
    """float64 softmax of query i of group g, [heads, keys]; with its row bound (fp32 scores, exp, sum and division)."""
    H, hd = c["heads"], c["hd"]
    k0, nk = c["gk"][g]
    q = c["q"][int(c["q_rows_h"][i])].double().cpu().view(H, hd)
    k = c["k"][k0:k0 + nk].double().cpu().view(nk, H, hd)
    if drop_last:
        k = k[:-1]
    scale = scale_mult / math.sqrt(hd)
    s = torch.einsum("hd,chd->hc", q, k) * scale
    p = torch.softmax(s, -1)
    mag = torch.einsum("hd,chd->hc", q.abs(), k.abs()).max(-1).values * scale        # [H]
    rel = 2 * (hd + 4) * U * mag + (nk / 8 + 64) * U                                  # |d s| twice + sum and exp/div
    return p.numpy(), rel.numpy()[:, None]


@pytest.mark.parametrize("hd", [48, 64])
def test_kernel_against_float64(hd):
    keys = [1, 63, 64, 65, 1000, 3000, 130]
    qs = [5, 63, 1, 17, 63, 33, 130]                 # the last group spans three 64-row chunks
    c = _probs_case(hd, 3, np.asarray(keys), np.asarray(qs), seed=hd)
    H = c["heads"]
    out = torch.full((c["total"],), SENTINEL, dtype=torch.float32, device="cuda")
    n0 = ops.launch_count()
    ops.cross_attention_probs(c["q"], c["k"], c["q_rows"], c["group_q"], c["group_k"], H, hd, out, c["off"], 1)
    torch.cuda.synchronize()
    assert ops.launch_count() == n0 + 1
    got = out.cpu().numpy()
    written = np.zeros(c["total"], bool)
    i = 0
    for g, (nk, nq) in enumerate(zip(keys, qs)):
        wrong_scale_passes = one_short_passes = True
        for _ in range(nq):
            blk = got[c["off_h"][i]:c["off_h"][i] + 2 * H * nk].reshape(2, H, nk)
            written[c["off_h"][i] + H * nk:c["off_h"][i] + 2 * H * nk] = True
            want, rel = _ref(c, i, g)
            p = blk[1]
            assert np.abs(p.astype(np.float64).sum(-1) - 1).max() <= 1e-5
            assert (np.abs(p - want) <= rel * want + 1e-30).all(), (g, i, np.abs(p - want).max())
            if nk > 1:
                bad, _ = _ref(c, i, g, scale_mult=1.001)
                wrong_scale_passes &= bool((np.abs(p - bad) <= rel * bad + 1e-30).all())
                bad, _ = _ref(c, i, g, drop_last=True)
                one_short_passes &= bool((np.abs(p[:, :-1] - bad) <= rel * bad + 1e-30).all())
            i += 1
        # the bound is tight enough to reject a reference with a 0.1 % wrong scale or one key short
        assert nk == 1 or not (wrong_scale_passes or one_short_passes), (g, wrong_scale_passes, one_short_passes)
    # layer 0 of every block and the gaps between blocks keep their sentinel bits
    assert (got.view(np.int32)[~written] == np.float32(SENTINEL).view(np.int32)).all()
    # the same operands as layer 0: the same bits
    ops.cross_attention_probs(c["q"], c["k"], c["q_rows"], c["group_q"], c["group_k"], H, hd, out, c["off"], 0)
    got0 = out.cpu().numpy()
    for i in range(len(c["off_h"])):
        nk = keys[np.searchsorted(np.cumsum(qs), i, side="right")]
        a = got0[c["off_h"][i]:c["off_h"][i] + 2 * H * nk].reshape(2, H, nk)
        assert np.array_equal(a[0].view(np.int32), a[1].view(np.int32))


def test_kernel_rows_do_not_depend_on_their_group():
    """A query row's probabilities are the same bits alone, at any position of a 63-row group, and in any launch."""
    c = _probs_case(48, 4, np.array([777]), np.array([63]), seed=3)
    H = 4
    out = torch.zeros(c["total"], device="cuda")
    ops.cross_attention_probs(c["q"], c["k"], c["q_rows"], c["group_q"], c["group_k"], H, 48, out, c["off"], 0)
    for i in (0, 9, 62):
        one = torch.zeros(2 * H * 777, device="cuda")
        ops.cross_attention_probs(c["q"], c["k"], c["q_rows"][i:i + 1].contiguous(), torch.tensor([[0, 1]], dtype=torch.int32,
                                  device="cuda"), c["group_k"], H, 48, one, torch.zeros(1, dtype=torch.int64, device="cuda"), 0)
        o = c["off_h"][i]
        assert torch.equal(one[:H * 777], out[o:o + H * 777])


def test_kernel_rejects_malformed_arguments_without_a_launch():
    lib = _lib.lib()
    c = _probs_case(48, 2, np.array([10]), np.array([3]), seed=1)
    out = torch.zeros(c["total"] + 4, device="cuda")
    n0 = lib.vf_launch_count()
    p = lambda t: t.data_ptr()
    base = [p(c["q"]), c["q"].stride(0), p(c["q_rows"]), p(c["group_q"]), 1, p(c["k"]), c["k"].stride(0), p(c["group_k"]), 2,
            48, p(out), p(c["off"]), 0, torch.cuda.current_stream().cuda_stream]
    for idx, val in ((0, p(c["q"]) + 2), (5, p(c["k"]) + 8), (1, 97), (9, 40), (4, -1), (8, 0), (12, -3), (10, p(out) + 2),
                     (11, p(c["off"]) + 4)):
        args = list(base); args[idx] = val
        assert lib.vf_cross_attention_probs(*args) < 0, (idx, val)
    torch.cuda.synchronize()
    assert lib.vf_launch_count() == n0


# ---- engine ------------------------------------------------------------------------------------------------------------
def _run(engine, batch, **kw):
    sq = lambda xs: [x[:, 0, :] for x in xs]
    out = engine.forward_tokens(sq(batch["cre_sequences"]), sq(batch["cre_attention_masks"]), sq(batch["gene_embeddings"]),
                                sq(batch["gene_attention_masks"]), batch["tissue_context"], batch["ref_cre_labels"], **kw)
    torch.cuda.synchronize()
    return out


def _maps(out, T, C, L, H):
    """Engine output -> list (per prediction) of [L, H, C] numpy arrays."""
    flat = out["cre_attention"].cpu().numpy(); off = out["cre_attention_off"]
    Cs = np.repeat(C, T)
    assert len(off) == len(Cs)
    return [flat[o:o + L * H * c].reshape(L, H, c) for o, c in zip(off, Cs)]


def _oracle_maps(monkeypatch, sd, cfg, hp, batch):
    """Registry-row probabilities of every gene layer's cross-attention, recorded from the oracle's own q and k
    (schedule="reference": one query sequence and one CRE copy per tissue).  -> {(gene, layer): [T, H, C]}."""
    rec, gene = {}, [0]
    orig = model_fp32._mha_cross

    def spy(num, sd_, pre, x, ctx, cu_q, cu_k, H):
        if "gene_layers." in pre:
            layer = int(pre.split("gene_layers.")[1].split(".")[0])
            n, d = x.shape
            q = num.linear(x, sd_[pre + "Wq.weight"], sd_[pre + "Wq.bias"]).view(n, H, d // H).double()
            k = num.linear(ctx, sd_[pre + "Wkv.weight"], sd_[pre + "Wkv.bias"]).view(ctx.shape[0], 2, H, d // H)[:, 0].double()
            P = [torch.softmax(torch.einsum("hd,chd->hc", q[cu_q[t]], k[cu_k[t]:cu_k[t + 1]]) / math.sqrt(d // H), -1)
                 for t in range(len(cu_q) - 1)]
            if layer == 0 and rec:
                gene[0] += 1
            rec[(gene[0], layer)] = torch.stack(P).numpy()
        return orig(num, sd_, pre, x, ctx, cu_q, cu_k, H)
    monkeypatch.setattr(model_fp32, "_mha_cross", spy)
    want = model_fp32.predict_step(sd, cfg, hp, batch, schedule="reference")
    monkeypatch.setattr(model_fp32, "_mha_cross", orig)
    return rec, want


@pytest.mark.parametrize("fixture", ["model_golden.npz", "model_golden_large.npz"])
def test_maps_against_the_fp32_oracle(monkeypatch, fixture):
    batch, _, _ = load_model_golden(fixture)
    sd = random_init.make_state_dict(GOLD_CFG, GOLD_HP, seed=GOLD_SEED)
    rec, _ = _oracle_maps(monkeypatch, sd, GOLD_CFG, GOLD_HP, batch)
    L, H = GOLD_CFG["num_layers"], GOLD_CFG["num_heads"]
    T = [len(t) for t in batch["tissue_context"]]; C = [x.shape[0] for x in batch["cre_sequences"]]
    maps = _maps(_run(Engine(sd, GOLD_CFG, GOLD_HP), batch, cre_attention=True), T, C, L, H)
    bad = []
    for layer in range(L):
        got = np.concatenate([m[layer].ravel() for m in maps])
        want = np.concatenate([rec[(g, layer)][t].ravel() for g in range(len(T)) for t in range(T[g])])
        rep = parity_report(got, want)
        print(f"{fixture} layer {layer}: {rep}")
        if not rep["ok"]:
            bad.append((layer, rep))
    for m in maps:
        assert np.abs(m.astype(np.float64).sum(-1) - 1).max() <= 1e-5
    assert not bad, bad


MID_CFG = dict(random_init.V4_PCG_MODEL, emb_dim=512, gene_emb_dim=256, num_heads=8, num_layers=3, token_dim=256)   # hd 64
MID_HP = dict(random_init.SEQ2REG_HP, embedding_dim=256, num_heads=4, num_layers=2)


@pytest.fixture(scope="module")
def mid():
    sd = random_init.make_state_dict(MID_CFG, MID_HP, seed=11)
    batch = synth_batch(31, 3, [150, 40, 300], [5, 2, 9], [[62, 0, 14, 7], [3], [5, 9]])
    return Engine(sd, MID_CFG, MID_HP), batch


@pytest.mark.parametrize("cre_stream", [True, False])
def test_other_outputs_unchanged_and_coarse_equals_fine(monkeypatch, mid, cre_stream):
    eng, batch = mid
    monkeypatch.setattr(engine_mod, "CRE_STREAM", cre_stream)
    kw = dict(cre_token_position=[7, 0, 299], gene_token_position=[4, 1, 0])
    res = {}
    for coarse in (True, False):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        plain = _run(eng, batch, **kw)
        plain = {k: plain[k].clone() for k in ("pred", "emb", "gene_token_embedding", "cre_token_embedding")}
        with_maps = _run(eng, batch, cre_attention=True, **kw)
        for k, v in plain.items():
            assert torch.equal(v, with_maps[k]), (coarse, k)
        res[coarse] = with_maps
    assert np.array_equal(res[True]["cre_attention_off"], res[False]["cre_attention_off"])
    a, b = res[True]["cre_attention"], res[False]["cre_attention"]
    assert a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_batching_invariance_and_determinism():
    cfg = dict(GOLD_CFG); hp = dict(GOLD_HP)
    sd = random_init.make_state_dict(cfg, hp, seed=5)
    eng = Engine(sd, cfg, hp)
    L, H = cfg["num_layers"], cfg["num_heads"]
    C = [300, 64, 1000, 65, 1, 130, 12, 500]
    T = [[62, 3], [1], [7, 8, 9], [0], [5], [62, 40, 2], [11], [30]]
    slab = synth_batch(41, 8, C, [4, 2, 6, 1, 3, 2, 5, 7], T)
    out = _run(eng, slab, cre_attention=True)
    whole = _maps(out, [len(t) for t in T], C, L, H)
    again = _maps(_run(eng, slab, cre_attention=True), [len(t) for t in T], C, L, H)
    assert all(np.array_equal(x.view(np.int32), y.view(np.int32)) for x, y in zip(whole, again))
    r = 0
    for g in range(8):
        one = {k: ([v[g]] if isinstance(v, list) else v[g:g + 1]) for k, v in slab.items()}
        alone = _maps(_run(eng, one, cre_attention=True), [len(T[g])], [C[g]], L, H)
        for t in range(len(T[g])):
            assert np.array_equal(alone[t].view(np.int32), whole[r + t].view(np.int32)), (g, t)
        r += len(T[g])
    # a tissue at T = 1 and inside all 63 tissues of its gene
    one = {k: ([v[0]] if isinstance(v, list) else v[0:1]) for k, v in slab.items()}
    one["tissue_context"] = [torch.arange(63)]
    all63 = _maps(_run(eng, one, cre_attention=True), [63], [C[0]], L, H)
    for t in (0, 31, 62):
        one["tissue_context"] = [torch.tensor([t])]
        single = _maps(_run(eng, one, cre_attention=True), [1], [C[0]], L, H)[0]
        assert np.array_equal(single.view(np.int32), all63[t].view(np.int32)), t


# ---- public surface ----------------------------------------------------------------------------------------------------
def test_vcfprocessor_cre_attention(tmp_path):
    from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    chroms, var, genes = _world(seed=83, n_genes=2, n_cres=30)
    assert genes[1].strand == "-"
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    query = pd.DataFrame({"gene_id": [r["gene_id"] for r in rows], "tissues": ["whole blood,thyroid", "K562"]})
    vcf = str(tmp_path / "sample.vcf")
    before = sorted(p.name for p in tmp_path.rglob("*"))
    df, maps = vp.cre_attention(vcf, query)
    assert sorted(p.name for p in tmp_path.rglob("*")) == before              # writes no file
    L, H = CFG["num_layers"], CFG["num_heads"]
    assert set(maps) == {(rows[0]["gene_id"], "whole blood"), (rows[0]["gene_id"], "thyroid"), (rows[1]["gene_id"], "K562")}
    assert len(df) == 3 * L * 30
    ds, dl = vp.create_data(vcf, query)
    model, ckpt, trainer = vp.load_model()
    pred = vp.predict(model, ckpt, trainer, dl, ds)
    ds2, dl2 = vp.create_data(vcf, query)
    model.trainer = trainer
    batch_maps = [m for b in dl2 for m in model.predict_cre_attention(b)["cre_attention"]]
    for gi, (r, names) in enumerate(zip(rows, (["whole blood", "thyroid"], ["K562"]))):
        manifest = pd.read_csv(tmp_path / "_artifacts" / "gene_cre_manifests" / f"{r['gene_id']}.csv")
        _, order = ds.cre_manifest(r["gene_id"])
        if gi == 1:                                                            # minus strand: descending start
            assert (np.diff(manifest["start_cre"].to_numpy()[order]) <= 0).all()
        for t, name in enumerate(names):
            m = maps[(r["gene_id"], name)]
            assert m.shape == (L, H, 30) and m.dtype == np.float32
            assert np.array_equal(m[..., order], batch_maps[gi][t])
            for layer in range(L):
                sub = df[(df["gene_id"] == r["gene_id"]) & (df["tissue"] == name) & (df["layer"] == layer)]
                assert sub[["chromosome", "start_cre", "end_cre", "cre_name"]].reset_index(drop=True).equals(manifest)
                assert np.array_equal(sub["attention"].to_numpy(), m[layer].mean(0))
                assert (sub["predicted_expression"] == pred["predicted_expression"].iloc[gi][t, 0]).all()
