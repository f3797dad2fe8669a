"""The oracle (torch restatement, numpy equations, plain-C restatement) against the golden fixtures
produced by the unmodified reference (tests/golden/make_golden.py).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

import golden_cases
import oracle_c
from oracle import bigru_oracle as bo
from oracle import loader_oracle as lo
import fake_db

CASES = ["c0", "small_l2", "small_uni_bce", "small_bi_h0_mlsm", "ragged"]


def load(golden_dir, name):
    z = golden_cases.load(golden_dir, name)
    B, T, F, H, L, C, bidir = [int(v) for v in z["meta"]]
    return z, dict(B=B, T=T, F=F, H=H, L=L, C=C, D=2 if bidir else 1, bidir=bool(bidir))


def params_of(z, prefix="p:"):
    return {k[len(prefix):]: z[k] for k in z if k.startswith(prefix)}


def test_kat_torch_oracle(golden_dir):
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    m = bo.OracleBiGRU(8, 108, 4, 1, 50, 0.2, False, True)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params_of(z).items()})
    m.eval()
    for i in (1, 2, 3):
        with torch.no_grad():
            y = m(torch.from_numpy(z[f"x{i}"])).numpy()
        np.testing.assert_allclose(y, z[f"y{i}"], atol=1e-6, rtol=0)
    # SURVEY.md section 8(c) known-answer vectors
    np.testing.assert_allclose(z["y1"][0], [0.96302879, -1.16067171, -4.01751852, -4.27485228], atol=1e-5)
    np.testing.assert_allclose(z["y2"][0], [0.69684184, -1.72828078, -3.58145571, -3.75949073], atol=1e-5)


def test_kat_numpy_and_c(golden_dir):
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    P = params_of(z)
    flat = oracle_c.flatten_params(P, 1, 2)
    assert flat.size == oracle_c.lib().bigru_ref_param_count(108, 8, 1, 4, 2)
    for i in (1, 2, 3):
        y_np = bo.gru_forward_np(P, z[f"x{i}"], 8, 1, True)
        np.testing.assert_allclose(y_np, z[f"y{i}"], atol=2e-6, rtol=0)
        y_c, _ = oracle_c.forward(flat, z[f"x{i}"], 8, 1, 4, 2)
        np.testing.assert_allclose(y_c, z[f"y{i}"], atol=2e-6, rtol=0)


def _loss_and_dlogits(z, logits):
    kind = str(z["loss_kind"])
    if kind == "ce":
        return oracle_c.loss_ce(logits, z["target"])
    if kind == "bce":
        return oracle_c.loss_bce(logits, z["target"], z["loss_weight"], z["loss_pos_weight"])
    return oracle_c.loss_bce(logits, z["target"])


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_forward_backward(golden_dir, name):
    z, d = load(golden_dir, name)
    P = params_of(z)
    flat = oracle_c.flatten_params(P, d["L"], d["D"])
    h0 = z["h0"] if "h0" in z else None
    logits, hn, stash = oracle_c.forward(flat, z["x"], d["H"], d["L"], d["C"], d["D"], h0, keep=True)
    scale = np.abs(z["logits"]).max()
    assert np.abs(logits - z["logits"]).max() / scale < 2e-6
    loss, dlog = _loss_and_dlogits(z, z["logits"])
    assert abs(loss - float(z["loss"])) < 2e-6 * max(1.0, abs(float(z["loss"])))
    grads, dx, dh0 = oracle_c.backward(flat, z["x"], stash, dlog, d["H"], d["L"], d["C"], d["D"])
    gflat = oracle_c.flatten_params(params_of(z, "g:"), d["L"], d["D"])
    assert np.linalg.norm(grads - gflat) / np.linalg.norm(gflat) < 2e-5
    assert np.linalg.norm(dx - z["dx"]) / np.linalg.norm(z["dx"]) < 2e-5
    if h0 is not None:
        assert np.linalg.norm(dh0 - z["dh0"]) / np.linalg.norm(z["dh0"]) < 2e-5
    # clip + Adam
    p = flat.copy(); m = np.zeros_like(p); v = np.zeros_like(p); g = gflat.copy()
    norm = oracle_c.clip_adam(p, g, m, v, 50.0, 1e-3, 0.9, 0.999, 1e-8, 1)
    assert abs(norm - float(z["grad_norm"])) < 1e-5 * float(z["grad_norm"])
    q = oracle_c.flatten_params(params_of(z, "q:"), d["L"], d["D"])
    np.testing.assert_allclose(p, q, atol=1e-5, rtol=0)


@pytest.mark.parametrize("name", ["small_l2", "small_uni_bce", "small_bi_h0_mlsm", "ragged"])
def test_numpy_equations(golden_dir, name):
    z, d = load(golden_dir, name)
    P = params_of(z)
    h0 = z["h0"] if "h0" in z else None
    logits, cache = bo.gru_forward_np(P, z["x"], d["H"], d["L"], d["bidir"], h0, keep=True)
    np.testing.assert_allclose(logits, z["logits"], atol=3e-6, rtol=0)
    _, dlog = _loss_and_dlogits(z, z["logits"])
    g, dx, dh0 = bo.gru_backward_np(cache, dlog)
    for k in g:
        np.testing.assert_allclose(g[k], z["g:" + k], atol=3e-6, rtol=1e-4)
    np.testing.assert_allclose(dx, z["dx"], atol=3e-6, rtol=1e-4)
    if h0 is not None:
        np.testing.assert_allclose(dh0, z["dh0"], atol=3e-6, rtol=1e-4)


@pytest.mark.parametrize("name", ["c0", "small_uni_bce"])
def test_torch_oracle_train_step(golden_dir, name):
    z, d = load(golden_dir, name)
    m = bo.OracleBiGRU(d["H"], d["F"], d["C"], d["L"], 50, 0.0, False, d["bidir"])
    m.load_state_dict({k: torch.from_numpy(v) for k, v in params_of(z).items()})
    if name == "c0":
        loss_fn, tgt = nn.CrossEntropyLoss(), torch.from_numpy(z["target"])
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        loss = bo.train_step(m, opt, loss_fn, torch.from_numpy(z["x"]), tgt)
        assert abs(float(loss) - float(z["loss"])) < 1e-6
        for k, v in m.state_dict().items():
            np.testing.assert_allclose(v.numpy(), z["q:" + k], atol=1e-5, rtol=0)   # Adam amplifies 1-ulp grad noise
    else:
        y = m(torch.from_numpy(z["x"]), torch.from_numpy(z["h0"]))
        np.testing.assert_allclose(y.detach().numpy(), z["logits"], atol=1e-6, rtol=0)


def test_loader_oracle(golden_dir):
    z = np.load(os.path.join(golden_dir, "loader.npz"))
    cols, targets, fields, query = fake_db.make_table(n_rows=250)
    ranges = lo.chunk_ranges(250, 100, 30)
    assert len(ranges) == int(z["n_chunks"])
    X = np.stack([np.nan_to_num(cols[f], nan=0.0) for f in fields], 1)
    Xraw = np.stack([cols[f] for f in fields], 1)
    Y = np.stack([targets[f"t{i}"] for i in range(4)], 1).astype(np.float32)
    for i, r in enumerate(ranges):
        np.testing.assert_array_equal(np.array(r), z[f"chunk{i}_ids"])
        rows = np.array(r) - 1
        mn, mx = lo.guard_min_max(np.nanmin(Xraw[rows], 0), np.nanmax(Xraw[rows], 0))
        mn, mx = lo.share_order_book(fields, mn, mx, 2, 2)
        np.testing.assert_array_equal(mn, z[f"chunk{i}_min"][0])
        np.testing.assert_array_equal(mx, z[f"chunk{i}_max"][0])
    tr, va, te = lo.split_sizes(len(ranges))
    assert [len(r) for r in ranges[tr]] == list(z["split_train"])
    assert [len(r) for r in ranges[va]] == list(z["split_val"])
    assert [len(r) for r in ranges[te]] == list(z["split_test"])
    rows = np.array(ranges[1]) - 1
    xn = lo.normalise(X[rows], z["chunk1_min"][0], z["chunk1_max"][0])
    np.testing.assert_array_equal(xn, z["bs2_xnorm"])
    for bs in (2, 8):
        batches = lo.delivered_batches(len(rows), 30, bs)
        assert len(batches) == int(z[f"bs{bs}_nbatches"])
        xb = np.concatenate([lo.collate(xn, Y[rows], s, 30)[0] for s in batches])
        yb = np.concatenate([lo.collate(xn, Y[rows], s, 30)[1] for s in batches])
        np.testing.assert_array_equal(xb, z[f"bs{bs}_x"])
        np.testing.assert_array_equal(yb, z[f"bs{bs}_y"])
        # C restatement of the gather
        xg = oracle_c.window_gather_norm(X[rows].astype(np.float32), z["chunk1_min"][0], z["chunk1_max"][0], 0, len(xb), 30)
        np.testing.assert_array_equal(xg, xb)
    assert lo.window_indices(5, 3) == [(0, 1, 2), (1, 2, 3), (2, 3, 4)]
    assert lo.window_indices(2, 3) == []


# ---- SURVEY.md 8(f) N4: window-function features (oracle/features_oracle.py) -----------------------------------------
def _market(n, seed=5):
    rng = np.random.default_rng(seed)
    close = 2900 + np.cumsum(rng.normal(0, 2.0, n))
    high = close + rng.uniform(0.1, 3.0, n)
    low = close - rng.uniform(0.1, 3.0, n)
    volume = rng.integers(100, 50000, n).astype(np.float64)
    delta = rng.normal(0, 300, n)
    return [np.float32(v).astype(np.float64) for v in (close, high, low, volume, delta)]


def test_features_oracle_against_pandas_rolling():
    import pandas as pd
    from oracle import features_oracle as fo
    close, high, low, volume, delta = _market(300)
    feats, tgt = fo.window_features(close, high, low, volume, delta)
    s = pd.Series(close)
    avg, sd = s.rolling(20, min_periods=1).mean(), s.rolling(20, min_periods=1).std(ddof=0)
    np.testing.assert_allclose(feats[:, 0], (avg + 2 * sd - s).values, rtol=0, atol=1e-7)
    np.testing.assert_allclose(feats[:, 1], (s - (avg - 2 * sd)).values, rtol=0, atol=1e-7)
    np.testing.assert_allclose(feats[:, 2], pd.Series(volume).rolling(6, min_periods=1).mean().values, rtol=1e-12)
    np.testing.assert_allclose(feats[:, 3], pd.Series(volume).rolling(20, min_periods=1).mean().values, rtol=1e-12)
    np.testing.assert_allclose(feats[:, 4], avg.values, rtol=1e-12)
    np.testing.assert_allclose(feats[:, 5], pd.Series(delta).rolling(12, min_periods=1).mean().values, rtol=1e-9, atol=1e-9)
    mn, mx = s.rolling(15, min_periods=1).min(), s.rolling(15, min_periods=1).max()
    stoch = ((s - mn) / (mx - mn)).values
    assert np.isnan(feats[0, 6]) and np.isnan(stoch[0])                       # one-row frame: max == min -> NULL
    np.testing.assert_allclose(feats[1:, 6], stoch[1:], rtol=1e-12)
    atr = pd.Series(high - low).rolling(15, min_periods=1).mean().values
    np.testing.assert_allclose(feats[:, 7], atr, rtol=1e-12)
    assert np.isnan(feats[0, 8])
    np.testing.assert_allclose(feats[1:, 8], np.diff(close), rtol=0, atol=0)
    # targets: LEAD(close, 8 / 15); NULL past the end -> 0
    p8, p15 = s.shift(-8).values, s.shift(-15).values
    np.testing.assert_array_equal(tgt[:, 0], np.nan_to_num(p8 >= close + 1.5 * atr, nan=0).astype(float) * ~np.isnan(p8))
    np.testing.assert_array_equal(tgt[:, 3], (np.where(np.isnan(p15), np.inf, p15) <= close - 3 * atr).astype(float))
    assert tgt[-8:, 0].sum() == 0 and tgt[-15:, 1].sum() == 0 and tgt[-8:, 2].sum() == 0 and tgt[-15:, 3].sum() == 0


def test_features_oracle_hand_rows_and_shapes():
    from oracle import features_oracle as fo
    close = np.array([10., 12., 11., 15.]); high = close + 1; low = close - 2
    feats, tgt = fo.window_features(close, high, low, np.ones(4), np.arange(4.), volume_MA_periods=[2], price_MA_periods=[3],
                                    delta_MA_periods=[], bollinger_bands_period=2, bollinger_bands_std=1, stochastic_oscillator=True)
    assert feats.shape == (4, 7) and tgt.shape == (4, 4) and not tgt.any()
    # row 2: BB over (12, 11): avg 11.5, pop-std 0.5 -> upper 12 - 11 = 1, lower 11 - 11 = 0
    np.testing.assert_allclose(feats[2, :2], [1.0, 0.0])
    np.testing.assert_allclose(feats[:, 3], [10, 11, 11, 38 / 3])             # price_MA3 with clipped frames
    np.testing.assert_allclose(feats[:, 5], [3, 3, 3, 3])                     # ATR: high - low == 3
    np.testing.assert_allclose(feats[1:, 6], [2, -1, 4])
    np.testing.assert_allclose(feats[1:, 4], [1.0, 0.5, 1.0])                 # stoch over all rows so far
    f0, t0 = fo.window_features(np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0), np.zeros(0))
    assert f0.shape == (0, 9) and t0.shape == (0, 4)


def test_features_oracle_against_reference_sql(golden_dir):
    """SURVEY.md 8(f) N4, pinned: the restatement equals what the reference's own CREATE VIEW statements
    (create_database.py:76-190, executed unmodified through the sqlite3 shim of tests/golden/make_features_golden.py)
    return - every feature column, the SQL NULLs and the four target labels."""
    from oracle import features_oracle as fo
    z = np.load(os.path.join(golden_dir, "features.npz"))
    cols = [z[k].astype(np.float64) for k in ("close", "high", "low", "volume", "delta")]
    f, t = fo.window_features(*cols, volume_MA_periods=list(z["volume_MA_periods"]), price_MA_periods=list(z["price_MA_periods"]),
                              delta_MA_periods=list(z["delta_MA_periods"]), bollinger_bands_period=int(z["bollinger_bands_period"]),
                              bollinger_bands_std=float(z["bollinger_bands_std"]), stochastic_oscillator=True)
    assert int(z["n_views"]) == 8 and f.shape == z["features"].shape
    assert np.array_equal(np.isnan(f), np.isnan(z["features"]))
    np.testing.assert_allclose(np.nan_to_num(f), np.nan_to_num(z["features"]), rtol=1e-12, atol=1e-9)
    assert np.array_equal(t, z["targets"])
