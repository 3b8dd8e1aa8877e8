"""Host side of the gene -> CRE cross-attention maps: the slab layout, the manifest-order long format of
VCFProcessor.cre_attention, and argument checks of vf_cross_attention_probs that fail before any launch (no GPU)."""
import ctypes as C

import numpy as np
import pandas as pd
import pytest

from variantformer_b200 import _lib
from variantformer_b200.engine import cre_attention_layout
from variantformer_b200.processors.vcfprocessor import cre_attention_frame


def test_layout_of_a_slab():
    gq, gk, off, total = cre_attention_layout([2, 1, 3], [5, 0, 7], n_layers=4, heads=3)
    assert gq.dtype == np.int32 and gq.tolist() == [[0, 2], [2, 1], [3, 3]]
    assert gk.dtype == np.int32 and gk.tolist() == [[0, 5], [5, 0], [5, 7]]
    size = [60, 60, 0, 84, 84, 84]
    assert off.dtype == np.int64 and off.tolist() == list(np.cumsum(size) - size) and total == sum(size)


def test_frame_undoes_the_minus_strand_batch_order():
    manifest = pd.DataFrame({"chromosome": "chr2", "start_cre": [500, 100, 300, 100], "end_cre": [600, 150, 420, 180],
                             "cre_name": ["dELS", "PLS", "pELS", "CTCF-only"]})
    order = np.argsort(manifest["start_cre"].to_numpy() - 50, kind="stable")[::-1]      # '-' gene: descending start
    assert order.tolist() == [0, 2, 3, 1]
    T, L, H, Cn = 2, 3, 4, 4
    rng = np.random.default_rng(0)
    batch = rng.random((T, L, H, Cn)).astype(np.float32)
    pred = np.array([[1.5], [0.25]], np.float32)
    df, maps = cre_attention_frame("G", ["thyroid", "whole blood"], manifest, order, batch, pred)
    assert len(df) == T * L * Cn and set(maps) == {("G", "thyroid"), ("G", "whole blood")}
    for t, name in enumerate(["thyroid", "whole blood"]):
        m = maps[("G", name)]
        assert np.array_equal(m[..., order], batch[t])          # batch position k = manifest row order[k]
        for layer in range(L):
            sub = df[(df["tissue"] == name) & (df["layer"] == layer)]
            assert sub[["chromosome", "start_cre", "end_cre", "cre_name"]].reset_index(drop=True).equals(manifest)
            assert np.array_equal(sub["attention"].to_numpy(), m[layer].mean(0))
            assert (sub["predicted_expression"] == pred[t, 0]).all() and (sub["gene_id"] == "G").all()


def test_malformed_arguments_fail_before_any_launch():
    lib = _lib.load()
    n0 = lib.vf_launch_count()
    A = 1 << 20                                     # aligned stand-in addresses: nothing is dereferenced on error

    def call(q=A, ldq=96, q_rows=A, group_q=A, n_groups=1, k=A, ldk=96, group_k=A, heads=2, hd=48, out=A, off=A, layer=0):
        return lib.vf_cross_attention_probs(q, ldq, q_rows, group_q, n_groups, k, ldk, group_k, heads, hd, out, off, layer,
                                            None)
    bad = [dict(hd=32), dict(hd=96, ldq=192, ldk=192), dict(q=A + 2), dict(k=A + 8), dict(ldq=100), dict(ldk=44),
           dict(ldq=88), dict(n_groups=-1), dict(heads=0), dict(heads=-2), dict(layer=-1), dict(out=A + 2),
           dict(off=A + 4), dict(q_rows=A + 1), dict(group_q=A + 2), dict(group_k=A + 3), dict(q=0), dict(out=0)]
    for kw in bad:
        assert call(**kw) < 0, kw
        assert _lib.load().vf_last_error().decode().startswith("cross_attention_probs"), kw
    assert call(n_groups=0) == 0                    # nothing to do: no launch, no device access
    assert lib.vf_launch_count() == n0
    assert lib.vf_seq2gene_forward_attn(None, None, None, None, None, 0, None, None, None, None, None, None) < 0
    assert lib.vf_launch_count() == n0


@pytest.mark.parametrize("name", ["vf_cross_attention_probs", "vf_seq2gene_forward_attn"])
def test_new_symbols_are_exported(name):
    assert name in _lib.SIGNATURES and hasattr(C.CDLL(_lib.LIB_PATH), name)
