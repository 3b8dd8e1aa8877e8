"""Host-side arithmetic of bench.py (no GPU, no model): the CPU arm's cost line, the per-config metric table and the
output dump."""
import numpy as np

import bench


def test_cost_line_recovers_base_and_marginal_cost():
    # cost(T) = base + T * marginal exactly (the reference schedule repeats both streams per tissue)
    pts = [(1, 5.0 + 3.0), (2, 5.0 + 6.0), (4, 5.0 + 12.0)]
    rate, base, marginal = bench.fit_rate(pts, stage1_s=0.5, T=63)
    assert abs(marginal - 3.0) < 1e-9 and abs(base - 5.5) < 1e-9
    assert abs(rate - 63 / (5.5 + 63 * 3.0)) < 1e-12


def test_cost_line_with_noise_is_least_squares_not_a_two_point_difference():
    rng = np.random.default_rng(0)
    pts = [(t, 4.0 + 2.5 * t + rng.normal(0, 0.05)) for t in (1, 2, 4, 1, 2, 4)]
    _, base, marginal = bench.fit_rate(pts, stage1_s=0.0, T=63)
    assert abs(marginal - 2.5) < 0.1 and abs(base - 4.0) < 0.3


def test_a_single_tissue_count_does_not_pretend_to_know_the_base_cost():
    # one point cannot separate base from marginal: the fallback attributes everything to the marginal cost (a LOWER CPU
    # rate) — which is why run_reference adds a warm-up sample at a second tissue count before it fits
    rate1, base, marginal = bench.fit_rate([(1, 8.0)], stage1_s=0.0, T=63)
    assert base == 0.0 and abs(marginal - 8.0) < 1e-12
    rate2, _, _ = bench.fit_rate([(1, 8.0), (2, 11.0)], stage1_s=0.0, T=63)
    assert rate2 > 2 * rate1


def test_dump_outputs_writes_float_arrays_and_a_seeded_row_sample_above_the_cap(tmp_path, monkeypatch):
    import torch
    pred = torch.arange(100, dtype=torch.float32)
    emb = torch.arange(100 * 8, dtype=torch.float32).view(100, 8).bfloat16()      # bf16 has no numpy dtype
    bench.dump_outputs(str(tmp_path / "all"), {"pred": pred, "emb": emb, "f64": np.ones(3)})
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in ("pred", "emb", "f64")}
    assert got["pred"].dtype == np.float32 and got["emb"].dtype == np.float32 and got["f64"].dtype == np.float64
    assert (got["pred"] == pred.numpy()).all() and (got["emb"] == emb.float().numpy()).all()

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1800)                          # 3600 bytes in all -> half the rows
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"pred": pred, "emb": emb})
    a = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("pred", "emb")}
    b = {k: np.load(tmp_path / "b" / f"{k}.npy") for k in ("pred", "emb")}
    assert sum(x.nbytes for x in a.values()) <= 1800
    assert a["pred"].shape == (50,) and a["emb"].shape == (50, 8)
    rows = a["pred"].astype(int)                                                  # pred[i] == i: the rows it kept
    assert (np.diff(rows) > 0).all() and (a["emb"] == emb.float().numpy()[rows]).all()
    assert all((a[k] == b[k]).all() for k in a)


def test_every_config_has_a_metric_and_unit():
    for c in (1, 2, 3, 4, 5):
        metric, unit = bench.METRICS[c]
        assert metric and unit
    assert bench.METRICS[3][0] == bench.METRIC
