"""bigru_infer_cluster: the live predictor's forward for full-size models (long windows, hidden sizes up to 512), against
the C oracle, and LivePredictor's choice between it and the single-CTA kernel."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import oracle_c


@pytest.fixture(scope="module")
def pkg():
    import financial_market_data_analysis_b200 as p
    from financial_market_data_analysis_b200 import build as b
    if not os.path.exists(p._lib.LIB_PATH):
        b.build()
    return p


def _model(pkg, H, F, Cn, L, bidir, seed=5):
    torch.manual_seed(seed)
    return pkg.BiGRU(H, F, Cn, L, 50, 0.0, False, bidir, precision="fp32").cuda().eval()


def _infer_cluster(pkg, m, x, xmin=None, xmax=None):
    """bigru_infer_cluster on device tensors; returns (logits, probs) on the device."""
    _lib = pkg._lib
    lib = _lib.load()
    B, T, F = x.shape
    H, L, Cn, bi = m.hidden_size, m.n_layers, m.output_size, int(m.bidirectional)
    nbytes = C.c_size_t()
    _lib.check(lib.bigru_infer_cluster_workspace_bytes(B, T, F, H, L, bi, C.byref(nbytes)), "workspace")
    work = torch.empty(nbytes.value // 4, dtype=torch.float32, device="cuda")
    logits = torch.empty(B, Cn, device="cuda")
    probs = torch.empty(B, Cn, device="cuda")
    _lib.check(lib.bigru_infer_cluster(_lib.ptr(m.flat_parameters()), _lib.ptr(x), _lib.ptr(xmin), _lib.ptr(xmax), B, T, F, H, L, Cn,
                                       bi, _lib.ptr(work), _lib.ptr(logits), _lib.ptr(probs),
                                       torch.cuda.current_stream().cuda_stream), "bigru_infer_cluster")
    return logits, probs


def _oracle_logits(m, x):
    D = 2 if m.bidirectional else 1
    ref, _ = oracle_c.forward(m.flat_parameters().cpu().numpy(), x, m.hidden_size, m.n_layers, m.output_size, D)
    return ref


def _assert_close(logits, probs, ref):
    got = logits.cpu().numpy()
    scale = max(np.abs(ref).max(), 1e-3)
    assert np.abs(got - ref).max() / scale < 1e-5
    assert np.abs(probs.cpu().numpy() - 1 / (1 + np.exp(-got.astype(np.float64)))).max() < 1e-6


# ---- without a device ----------------------------------------------------------------------------------------------------
def test_workspace_query_without_device(pkg):
    lib = pkg._lib.load()
    n = C.c_size_t()
    assert lib.bigru_infer_cluster_workspace_bytes(1, 128, 64, 256, 2, 1, C.byref(n)) == 0
    # normalised input + gi of both directions + one layer output, each rounded up to 256 bytes
    assert n.value == 4 * (128 * 64 + 2 * 128 * 768 + 128 * 512)
    uni = C.c_size_t()
    assert lib.bigru_infer_cluster_workspace_bytes(1, 128, 64, 256, 2, 0, C.byref(uni)) == 0 and uni.value < n.value
    for bad in ((0, 5, 5, 8, 1, 1), (1, 0, 5, 8, 1, 1), (1, 5, 0, 8, 1, 1), (1, 5, 5, 0, 1, 1), (1, 5, 5, 8, 0, 1)):
        assert lib.bigru_infer_cluster_workspace_bytes(*bad, C.byref(n)) == pkg._lib.ERR_ARG
    assert lib.bigru_infer_cluster_workspace_bytes(1, 5, 5, 8, 1, 1, None) == pkg._lib.ERR_ARG


def test_argument_errors_without_device(pkg):
    """Arguments are checked before anything touches a device; both kinds of refusal surface as ValueError."""
    _lib = pkg._lib
    lib = _lib.load()
    p = C.c_void_p(256)                                   # never dereferenced: every call below is refused first

    def call(params=p, x=p, xmin=None, xmax=None, B=1, T=5, F=5, H=8, L=1, Cn=4, bi=1, work=p, logits=p):
        return lib.bigru_infer_cluster(params, x, xmin, xmax, B, T, F, H, L, Cn, bi, work, logits, None, None)

    for kw in (dict(params=None), dict(x=None), dict(work=None), dict(logits=None), dict(B=0), dict(T=0), dict(F=-1), dict(H=0),
               dict(L=0), dict(L=17), dict(Cn=0), dict(xmin=p), dict(work=C.c_void_p(260))):
        assert call(**kw) == _lib.ERR_ARG, kw
        with pytest.raises(ValueError, match="bad argument"):
            _lib.check(call(**kw), "bigru_infer_cluster")
    assert call(H=513) == _lib.ERR_UNSUPPORTED
    with pytest.raises(ValueError, match="not supported"):
        _lib.check(call(H=513), "bigru_infer_cluster")


def test_checkpoint_shape_is_read_from_the_state_dict(pkg):
    from financial_market_data_analysis_b200.predict import checkpoint_shape
    m = pkg.BiGRU(256, 64, 4, 2, 50, 0.0, False, True, precision="fp32")
    assert checkpoint_shape(m.state_dict()) == (256, 2)
    m = pkg.BiGRU(8, 108, 4, 1, 50, 0.0, False, True, precision="fp32")
    assert checkpoint_shape(m.state_dict()) == (8, 1)


# ---- on the GPU -----------------------------------------------------------------------------------------------------------
SWEEP = [  # B, T, F, H, L, bidirectional
    (1, 1, 5, 8, 1, True),
    (3, 5, 64, 33, 2, False),
    (17, 49, 108, 64, 1, True),          # 5 window groups per direction
    (2, 128, 64, 128, 2, True),
    (1, 49, 5, 200, 3, False),
    (3, 128, 64, 256, 2, True),          # T > 48 at H 256: bigru_infer_window refuses it
    (1, 128, 108, 256, 1, False),
    (1, 5, 108, 300, 1, True),           # ragged last slice
    (1, 49, 64, 512, 2, True),           # T > 23 at H 512: bigru_infer_window refuses it
    (17, 5, 5, 512, 1, False),
    (3, 1, 108, 512, 3, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", SWEEP, ids=lambda c: "B{}-T{}-F{}-H{}-L{}-{}".format(*c[:5], "bi" if c[5] else "uni"))
def test_sweep_against_c_oracle(pkg, cfg):
    B, T, F, H, L, bidir = cfg
    m = _model(pkg, H, F, 3, L, bidir)
    x = torch.randn(B, T, F, generator=torch.Generator().manual_seed(2))
    logits, probs = _infer_cluster(pkg, m, x.cuda())
    _assert_close(logits, probs, _oracle_logits(m, x.numpy()))


@pytest.mark.gpu
def test_configs4_model_one_window(pkg):
    """BASELINE configs[4] model (T 1024, F 128, H 512, L 2, bidirectional): needs 16-CTA clusters."""
    m = _model(pkg, 512, 128, 3, 2, True)
    x = torch.randn(1, 1024, 128, generator=torch.Generator().manual_seed(3))
    try:
        logits, probs = _infer_cluster(pkg, m, x.cuda())
    except ValueError as e:
        assert "16-CTA cluster" in str(e)
        return
    _assert_close(logits, probs, _oracle_logits(m, x.numpy()))


@pytest.mark.gpu
def test_raw_windows_with_min_max_match_normalised_windows(pkg):
    B, T, F, H = 3, 64, 108, 256
    m = _model(pkg, H, F, 4, 2, True)
    g = torch.Generator().manual_seed(4)
    mn = torch.rand(F, generator=g) * 100
    mx = mn + 1 + torch.rand(F, generator=g) * 50
    raw = (mn + torch.rand(B, T, F, generator=g) * (mx - mn)).cuda()
    mn, mx = mn.cuda(), mx.cuda()
    got, _ = _infer_cluster(pkg, m, raw, mn, mx)
    want, _ = _infer_cluster(pkg, m, ((raw - mn) / (mx - mn)).contiguous())
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_repeat_calls_are_bitwise_equal(pkg):
    m = _model(pkg, 256, 64, 4, 2, True)
    x = torch.randn(5, 128, 64, generator=torch.Generator().manual_seed(6)).cuda()
    a, _ = _infer_cluster(pkg, m, x)
    b, _ = _infer_cluster(pkg, m, x)
    assert torch.equal(a, b)


def _launches(pkg, fn):
    lib = pkg._lib.load()
    torch.cuda.synchronize()
    n0 = lib.bigru_launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, lib.bigru_launch_count() - n0


@pytest.mark.gpu
def test_live_predictor_configs1_checkpoint(pkg):
    """A configs[1]-shaped checkpoint (H 256, L 2, window 128, F 64, 4 labels) loads without restating its shape and is
    served by bigru_infer_cluster (2L+1 launches)."""
    from financial_market_data_analysis_b200.predict import LivePredictor
    src = _model(pkg, 256, 64, 4, 2, True, seed=11)
    state = {k: v.detach().cpu() for k, v in src.state_dict().items()}
    lp = LivePredictor(state, None, window=128)
    assert (lp.model.hidden_size, lp.model.n_layers) == (256, 2)
    x = torch.randn(128, 64, generator=torch.Generator().manual_seed(8))
    out, n = _launches(pkg, lambda: lp.predict(x.numpy(), "2020-03-02 10:05:00"))
    assert n == 5
    ref = _oracle_logits(lp.model, x.numpy()[None])[0]
    want = 1 / (1 + np.exp(-ref.astype(np.float64)))
    assert np.abs(out["probabilities"].numpy() - want).max() < 1e-5
    assert list(out["pred_indices"]) == list(np.where(out["probabilities"].numpy() > 0.5)[0])
    assert out["pred_labels"] == [lp.y_fields[i] for i in out["pred_indices"]] and out["timestamp"] == "2020-03-02 10:05:00"
    with torch.no_grad():
        same = torch.sigmoid(src.cuda().eval()(x[None].cuda()))[0].cpu().numpy()
    assert np.abs(out["probabilities"].numpy() - same).max() < 1e-5
    # several windows at once: as many window groups as needed, same answers per window
    xs = torch.randn(6, 128, 64, generator=torch.Generator().manual_seed(9))
    logits, _ = lp.forward_windows(xs.numpy())
    one, _ = lp.forward_windows(xs[4].numpy())
    assert np.abs(logits[4].cpu().numpy() - one[0].cpu().numpy()).max() < 1e-6


@pytest.mark.gpu
def test_live_predictor_keeps_small_models_on_one_launch(pkg, golden_dir):
    from financial_market_data_analysis_b200.predict import LivePredictor
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    state = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("p:")}
    lp = LivePredictor(state, None)
    assert (lp.model.hidden_size, lp.model.n_layers) == (8, 1)
    (logits, _), n = _launches(pkg, lambda: lp.forward_windows(z["x1"]))
    assert n == 1 and np.abs(logits.cpu().numpy() - z["y1"]).max() < 1e-5


@pytest.mark.gpu
def test_live_predictor_falls_back_to_the_model_above_hidden_512(pkg):
    from financial_market_data_analysis_b200.predict import LivePredictor
    src = _model(pkg, 520, 12, 4, 1, True)
    lp = LivePredictor({k: v.detach().cpu() for k, v in src.state_dict().items()}, None, window=3)
    x = torch.randn(1, 3, 12, generator=torch.Generator().manual_seed(1))
    logits, probs = lp.forward_windows(x.numpy())
    with torch.no_grad():
        want = src(x.cuda())
    assert torch.allclose(logits, want, rtol=0, atol=1e-6) and torch.allclose(probs, torch.sigmoid(want))
