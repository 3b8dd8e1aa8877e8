"""ctypes mirrors of the weight-pointer / slab tables of the coarse entry points (include/vf_b200.h:
vf_seq2reg_forward, vf_seq2gene_forward, vf_seq2gene_forward_attn) and their builders from the engine's device-side weight objects."""
import ctypes as C

_vp, _i, _f = C.c_void_p, C.c_int, C.c_float


class Linear(C.Structure):
    _fields_ = [("w", _vp), ("b", _vp), ("cs", _vp)]


class Seq2RegLayer(C.Structure):
    _fields_ = [("qkv", Linear), ("out", Linear), ("g1", Linear), ("g2", Linear)]


class Seq2RegWeights(C.Structure):
    _fields_ = [("d", _i), ("heads", _i), ("n_layers", _i), ("ffn_hidden", _i), ("token_length", _i), ("ln_eps", _f),
                ("emb", _vp), ("pe", _vp), ("slopes", _vp), ("layers", C.POINTER(Seq2RegLayer))]


class ContextLayer(C.Structure):
    _fields_ = [("qkv", Linear), ("out", Linear), ("q", Linear), ("kv", Linear), ("out2", Linear), ("g1", Linear),
                ("g2", Linear), ("kv9", _vp)]


class Seq2GeneWeights(C.Structure):
    _fields_ = [("D", _i), ("heads", _i), ("n_layers", _i), ("ffn_hidden", _i), ("token_dim", _i), ("ln_eps", _f),
                ("slopes", _vp), ("registry", _vp), ("cre_map", Linear), ("gene_map", Linear),
                ("cre_layers", C.POINTER(ContextLayer)), ("gene_layers", C.POINTER(ContextLayer)),
                ("h0", Linear), ("h4", Linear), ("hn_g", _vp), ("hn_b", _vp), ("h6_w", _vp), ("h6_b", _vp)]


class Seq2GeneSlab(C.Structure):
    _fields_ = [("n_cre", _i), ("n_gene_chunks", _i), ("n_gene_rows", _i), ("n_reg", _i), ("n_need", _i),
                ("single_stream", _i), ("gene_idx", _vp), ("row_seq", _vp), ("logc", _vp), ("last_rows", _vp),
                ("cre_pos_idx", _vp),
                ("slots_gself", _vp), ("n_gself", _i), ("slots_gcross", _vp), ("n_gcross", _i),
                ("slots_cself", _vp), ("n_cself", _i), ("slots_last_self", _vp), ("n_last_self", _i),
                ("slots_last_cross", _vp), ("n_last_cross", _i)]


class CreAttention(C.Structure):
    _fields_ = [("n_groups", _i), ("group_q", _vp), ("group_k", _vp), ("reg_rows", _vp), ("out", _vp), ("out_off", _vp)]


def _ptr(t):
    return None if t is None else t.data_ptr()


def linear(L):
    """engine._Linear / engine._LnLinear (or None) -> Linear."""
    if L is None:
        return Linear(None, None, None)
    return Linear(_ptr(L.w), _ptr(L.b), _ptr(getattr(L, "cs", None)))


def seq2reg_table(W, eps=1e-5):
    """engine.Seq2RegWeights -> (Seq2RegWeights, keep-alive list)."""
    layers = (Seq2RegLayer * W.L)(*[Seq2RegLayer(linear(L["qkv"]), linear(L["out"]), linear(L["g1"]), linear(L["g2"]))
                                     for L in W.layers])
    ffn = W.layers[0]["g1"].w.shape[0]
    t = Seq2RegWeights(W.d, W.H, W.L, ffn, W.token_length, eps, _ptr(W.emb), _ptr(W.pe), _ptr(W.slopes), layers)
    return t, [layers]


def _context_layer(L):
    return ContextLayer(linear(L["qkv"]), linear(L["out"]), linear(L["q"]), linear(L.get("kv")), linear(L["out2"]),
                        linear(L["g1"]), linear(L["g2"]), _ptr(L.get("kv9")))


def seq2gene_table(w, token_dim, eps=1e-5):
    """engine.Seq2GeneWeights -> (Seq2GeneWeights, keep-alive list)."""
    cre = (ContextLayer * max(len(w.cre_layers), 1))(*[_context_layer(L) for L in w.cre_layers])
    gene = (ContextLayer * len(w.gene_layers))(*[_context_layer(L) for L in w.gene_layers])
    ffn = w.gene_layers[0]["g1"].w.shape[0]
    t = Seq2GeneWeights(w.D, w.H, w.NL, ffn, token_dim, eps, _ptr(w.slopes), _ptr(w.registry), linear(w.cre_map),
                        linear(w.gene_map), cre, gene, linear(w.h0), linear(w.h4), _ptr(w.hn.g), _ptr(w.hn.b),
                        _ptr(w.h6_w), _ptr(w.h6_b))
    return t, [cre, gene]
