"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.
Run on the B200 box:  python -m pytest tests -m gpu -x -q"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

import fake_db
import golden_cases
import oracle_c
from oracle import bigru_oracle as bo
from oracle import loader_oracle as lo

pytestmark = pytest.mark.gpu

# fp32 path: logits <= 1e-4 rel (BASELINE.json north_star); gradients rel-L2 <= 1e-3 (SURVEY.md 8(d))
# step: Adam divides by |g| so elements with |g| ~ eps flip freely; bound the element error by a
# fraction of lr (1e-3) and the whole update by rel-L2
# bf16 path: operands, the gate stash and dgi/dgh are bf16 (fp32 accumulate/state), so the error of BPTT grows
# with T and L; bounds: per-tensor rel-L2 "grads", whole flat gradient "gflat"
# bf16x3 path ("fp32-class" on tensor cores: split bf16 operand pairs, fp32 accumulate / gate math / stash): the SAME bounds as
# the fp32 path - it is the variant BASELINE.json configs[1] ("fp32 tolerance check") is measured on
TOL = {"fp32": dict(logits=1e-4, grads=1e-3, gflat=1e-3, kat=1e-5, step=2e-4, update=2e-2),
       "bf16x3": dict(logits=1e-4, grads=1e-3, gflat=1e-3, kat=1e-5, step=5e-4, update=2e-2),   # step: see above, half of lr
       "bf16": dict(logits=3e-2, grads=0.15, gflat=6e-2, kat=3e-2, step=2e-3, update=0.5)}


def _pkg():
    import financial_market_data_analysis_b200 as pkg
    return pkg


def precisions():
    pkg = _pkg()
    lib = pkg._lib.load()
    out = ["fp32"]
    h = pkg._lib.C.c_void_p()
    if lib.bigru_plan_create(128, 16, 64, 256, 1, 3, 1, pkg._lib.PREC_BF16X3, pkg._lib.C.byref(h)) == 0:
        lib.bigru_plan_destroy(h)
        out.append("bf16x3")
    if lib.bigru_plan_create(128, 16, 64, 256, 1, 3, 1, pkg._lib.PREC_BF16, pkg._lib.C.byref(h)) == 0:
        lib.bigru_plan_destroy(h)
        out.append("bf16")
    return out


def supported(precision, B, F, H, h0=False):
    """Through the Python mirror the tensor-core paths take any batch size (zero-padded to whole batch tiles), any feature count
    (layer-0 K extent padded to 8 inside the plan) and any hidden size up to 256 (bf16x3) / 512 (bf16) - smaller models run
    zero-padded to 128 / 256 / 512 hidden units; BIGRU_PREC_BF16 has no initial hidden state."""
    if precision == "fp32":
        return True
    if precision == "bf16x3":
        return H <= 256
    return H <= 512 and not h0


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def params_of(z, prefix="p:"):
    return {k[len(prefix):]: z[k] for k in z if k.startswith(prefix)}


def make_model(d, sd_np, precision, dropout=0.0, spatial=False):
    m = _pkg().BiGRU(d["H"], d["F"], d["C"], d["L"], 50, dropout, spatial, d["bidir"], precision=precision)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd_np.items()})
    return m.cuda()


def loss_from(z):
    kind = str(z["loss_kind"])
    if kind == "ce":
        return nn.CrossEntropyLoss(), torch.from_numpy(z["target"])
    if kind == "bce":
        return (nn.BCEWithLogitsLoss(weight=torch.from_numpy(z["loss_weight"]), pos_weight=torch.from_numpy(z["loss_pos_weight"])),
                torch.from_numpy(z["target"]))
    return nn.MultiLabelSoftMarginLoss(), torch.from_numpy(z["target"])


def test_library_is_native_and_device_ok():
    pkg = _pkg()
    lib = pkg._lib.load()
    assert os.path.basename(pkg._lib.LIB_PATH) == "libbigru_b200.so"
    assert lib.bigru_device_check(0) == 0, lib.bigru_last_error()


def test_known_answer_vectors(golden_dir):
    """Shipped model_params.pt through the CUDA path (SURVEY.md 8(c) KAT1/KAT2)."""
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    for precision in precisions():
        if not supported(precision, 1, 108, 8):
            continue                                   # the shipped checkpoint has H=8: fp32 path only
        m = make_model(dict(H=8, F=108, C=4, L=1, bidir=True), params_of(z), precision, dropout=0.2)
        m.eval()
        for i in (1, 2, 3):
            with torch.no_grad():
                y = m(torch.from_numpy(z[f"x{i}"])).cpu().numpy()      # CPU input: moved to the model's device
            assert np.abs(y - z[f"y{i}"]).max() < TOL[precision]["kat"] * max(1.0, np.abs(z[f"y{i}"]).max()), (precision, i)


@pytest.mark.parametrize("name", ["c0", "small_l2", "small_uni_bce", "small_bi_h0_mlsm", "ragged"])
def test_golden_forward_backward_autograd(golden_dir, name):
    """Logits, loss, every parameter gradient, dx and dh0 against the reference's own autograd."""
    z = golden_cases.load(golden_dir, name)
    B, T, F, H, L, C, bidir = [int(v) for v in z["meta"]]
    d = dict(B=B, T=T, F=F, H=H, L=L, C=C, bidir=bool(bidir))
    for precision in precisions():
        if not supported(precision, B, F, H, "h0" in z):
            continue
        tol = TOL[precision]
        m = make_model(d, params_of(z), precision)
        m.train()
        x = torch.from_numpy(z["x"]).cuda().requires_grad_(True)
        h0 = torch.from_numpy(z["h0"]).cuda().requires_grad_(True) if "h0" in z else None
        loss_fn, tgt = loss_from(z)
        loss_fn = loss_fn.cuda()
        pred = m(x, h0)
        assert rel(pred.detach().cpu().numpy(), z["logits"]) < tol["logits"], precision
        loss = loss_fn(pred, tgt.cuda())
        loss.backward()
        assert abs(loss.item() - float(z["loss"])) < 10 * tol["logits"] * max(1.0, abs(float(z["loss"])))
        errs = {k: rel_l2(p.grad.cpu().numpy(), z["g:" + k]) for k, p in m.named_parameters()
                if np.abs(p.grad.cpu().numpy() - z["g:" + k]).max() >= 1e-7}
        assert all(v < tol["grads"] for v in errs.values()), (precision, errs)
        got = np.concatenate([p.grad.cpu().numpy().ravel() for _, p in m.named_parameters()])
        ref = np.concatenate([z["g:" + k].ravel() for k, _ in m.named_parameters()])
        assert rel_l2(got, ref) < tol["gflat"], (precision, rel_l2(got, ref))
        assert rel_l2(x.grad.cpu().numpy(), z["dx"]) < tol["grads"], (precision, rel_l2(x.grad.cpu().numpy(), z["dx"]))
        if h0 is not None:
            assert rel_l2(h0.grad.cpu().numpy(), z["dh0"]) < tol["grads"]


@pytest.mark.parametrize("name", ["c0", "small_uni_bce", "small_bi_h0_mlsm"])
def test_golden_fused_train_step(golden_dir, name):
    """zero_grad -> forward -> loss -> backward -> clip_grad_norm_ -> Adam (biGRU_model.py:198-210):
    parameters after one fused step against the reference's."""
    z = golden_cases.load(golden_dir, name)
    B, T, F, H, L, C, bidir = [int(v) for v in z["meta"]]
    d = dict(B=B, T=T, F=F, H=H, L=L, C=C, bidir=bool(bidir))
    for precision in precisions():
        if not supported(precision, B, F, H, "h0" in z):
            continue
        tol = TOL[precision]
        m = make_model(d, params_of(z), precision)
        loss_fn, tgt = loss_from(z)
        m.add_loss_fn(loss_fn)
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
        m.train()
        h0 = torch.from_numpy(z["h0"]).cuda() if "h0" in z else None
        loss, logits = m.train_step(torch.from_numpy(z["x"]).cuda(), tgt.cuda(), h0)
        assert abs(float(loss) - float(z["loss"])) < 10 * tol["logits"] * max(1.0, abs(float(z["loss"])))
        assert rel(logits.cpu().numpy(), z["logits"]) < tol["logits"]
        gn = float(torch.sqrt(m._adam["scal"][1]))
        assert abs(gn - float(z["grad_norm"])) < tol["grads"] * float(z["grad_norm"])
        upd_got, upd_ref = [], []
        for k, v in m.state_dict().items():
            if "q:" + k not in z:
                continue
            assert np.abs(v.cpu().numpy() - z["q:" + k]).max() < tol["step"], (precision, k)
            if "q:" + k not in z:
                continue                                  # buffers of the attached loss module
            upd_got.append((v.cpu().numpy() - z["p:" + k]).ravel())
            upd_ref.append((z["q:" + k] - z["p:" + k]).ravel())
        assert rel_l2(np.concatenate(upd_got), np.concatenate(upd_ref)) < tol["update"], precision


SWEEP = [  # B, T, F, H, L, C, bidir, h0
    (1, 1, 1, 1, 1, 1, True, False),
    (2, 3, 5, 7, 1, 2, False, True),
    (5, 4, 9, 33, 2, 3, True, True),
    (17, 9, 12, 40, 3, 4, True, False),
    (33, 6, 64, 64, 2, 3, False, False),
    (64, 16, 32, 128, 2, 3, True, False),
    (48, 7, 40, 256, 2, 3, True, False),
    (32, 5, 8, 128, 1, 2, False, False),
    (32, 9, 64, 128, 2, 3, True, False),      # F == 64: layer-0 input projection fused into the forward scan (bf16 path)
    (16, 5, 64, 256, 1, 2, False, False),
    (32, 6, 16, 128, 2, 3, True, True),       # initial hidden state on the x3 tensor-core path (2-CTA clusters)
    (64, 11, 24, 256, 2, 4, True, True),      # ... and with 4-CTA clusters, two batch tiles
    (96, 3, 8, 256, 1, 2, False, False),
    (19, 6, 13, 128, 2, 3, True, True),       # batch not a whole tile (zero-padded rows), n_features % 8 != 0 (padded K extent), h0
    (40, 5, 108, 256, 1, 4, True, False),     # the reference's own feature count (108) at a tensor-core hidden size
    (3, 4, 5, 128, 2, 2, False, False),
    (32, 1, 16, 256, 1, 2, True, False),      # single time step / two time steps on the 4-CTA-cluster kernels (ping-pong forward)
    (64, 2, 16, 256, 2, 2, True, True),
    (32, 300, 8, 256, 1, 2, True, False),     # many steps: barrier phase bookkeeping of the ping-pong scans far beyond the ring depths
    (32, 1, 16, 512, 1, 2, True, False),
    (64, 6, 24, 512, 2, 3, True, False),      # hidden 512 (bf16 path: 8-CTA clusters, tc_scan_w.cuh), two batch tiles
    (40, 3, 128, 512, 1, 2, False, False),
]


@pytest.mark.parametrize("cfg", SWEEP)
def test_sweep_against_c_oracle(cfg):
    B, T, F, H, L, C, bidir, use_h0 = cfg
    D = 2 if bidir else 1
    for precision in precisions():
        if not supported(precision, B, F, H, use_h0):
            continue
        tol = TOL[precision]
        torch.manual_seed(3)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, bidir, precision=precision).cuda()
        g = torch.Generator().manual_seed(11)
        x = torch.randn(B, T, F, generator=g)
        h0 = torch.randn(L * D, B, H, generator=g) * 0.5 if use_h0 else None
        dl = torch.randn(B, C, generator=g)
        flat = m.flat_parameters().cpu().numpy()
        sd = {k: v.cpu().numpy() for k, v in m.state_dict().items()}
        assert np.array_equal(flat, oracle_c.flatten_params(sd, L, D))       # C-ABI parameter order
        ref_logits, ref_hn, stash = oracle_c.forward(flat, x.numpy(), H, L, C, D, None if h0 is None else h0.numpy(), keep=True)
        ref_g, ref_dx, ref_dh0 = oracle_c.backward(flat, x.numpy(), stash, dl.numpy(), H, L, C, D)
        xg = x.cuda().requires_grad_(True)
        hg = h0.cuda().requires_grad_(True) if use_h0 else None
        y = m(xg, hg)
        y.backward(dl.cuda())
        scale = max(np.abs(ref_logits).max(), 1e-3)
        assert np.abs(y.detach().cpu().numpy() - ref_logits).max() / scale < tol["logits"], (precision, cfg)
        assert rel(m._last_hidden.cpu().numpy(), ref_hn) < tol["logits"] * 10
        got = torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).cpu().numpy()
        assert rel_l2(got, ref_g) < tol["grads"], (precision, cfg)
        assert rel_l2(xg.grad.cpu().numpy(), ref_dx) < tol["grads"]
        if use_h0:
            assert rel_l2(hg.grad.cpu().numpy(), ref_dh0) < tol["grads"]


def test_c1_shape_against_torch_oracle():
    """BASELINE config 1 shape (B512,T128,F64,H256,L2): logits <= 1e-4 rel of the torch.nn.GRU CPU path, gradients by
    rel-L2.  The max-pool over T routes its gradient to ONE time step per (row, unit); among 131 072 such maxima a
    handful are ties to within fp32 rounding (top-2 gap ~1e-6), where any implementation's rounding decides the route.
    So: (1) every routing disagreement with the reference must be such a tie (the reference's own values at the two
    steps differ by <= 2e-5 of the output scale), and (2) gradients are compared with the reference autograd run under
    the routing the kernel took (bo.forward_routed)."""
    B, T, F, H, L, C = 512, 128, 64, 256, 2, 3
    torch.manual_seed(0)
    ref = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(B, T, F, generator=g)
    target = torch.randint(0, C, (B,), generator=g)
    ref.train()

    def ref_grads(idx):
        ref.zero_grad()
        pred, s = bo.forward_routed(ref, x, None, idx)
        loss = nn.CrossEntropyLoss()(pred, target)
        loss.backward()
        return pred.detach(), loss.item(), s.detach(), {k: q.grad.numpy().copy() for k, q in ref.named_parameters()}

    pred, loss, s_ref, g_own = ref_grads(None)
    ref_arg = s_ref.argmax(dim=1)
    scale = float(s_ref.abs().max())
    report = {}
    for precision in precisions():
        tol = TOL[precision]
        torch.manual_seed(0)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=precision).cuda()
        m.train()
        y = m(x.cuda())
        arg = m.pooled_argmax().cpu().long()
        l2 = nn.CrossEntropyLoss()(y, target.cuda())
        l2.backward()
        e_log = rel(y.detach().cpu().numpy(), pred.numpy())
        assert e_log < tol["logits"], (precision, e_log)
        assert abs(l2.item() - loss) < 10 * tol["logits"]
        flips = arg != ref_arg
        nflip = int(flips.sum())
        tie_tol = (2e-5 if precision != "bf16" else 2e-2) * scale
        if nflip:
            gap = (s_ref.gather(1, ref_arg.unsqueeze(1)) - s_ref.gather(1, arg.unsqueeze(1))).squeeze(1)[flips]
            assert float(gap.max()) <= tie_tol, (precision, nflip, float(gap.max()))
        want_g = ref_grads(arg)[3] if nflip else g_own
        errs = {k: rel_l2(p.grad.cpu().numpy(), want_g[k]) for k, p in m.named_parameters()}
        got = np.concatenate([p.grad.cpu().numpy().ravel() for _, p in m.named_parameters()])
        want = np.concatenate([want_g[k].ravel() for k, _ in m.named_parameters()])
        report[precision] = dict(logits_rel=e_log, grad_flat_rel_l2=rel_l2(got, want), grad_worst_tensor=max(errs.values()), pool_ties_rerouted=nflip)
        print(f"c1[{precision}] logits rel {e_log:.2e} flat-grad rel-L2 {rel_l2(got, want):.2e} worst tensor {max(errs.values()):.2e} "
              f"(max-pool ties routed differently: {nflip} of {flips.numel()})")
        assert all(v < tol["grads"] for v in errs.values()), (precision, errs)
        assert rel_l2(got, want) < tol["gflat"], (precision, rel_l2(got, want))
    out = os.environ.get("BIGRU_PARITY_REPORT")
    if out:
        import json
        with open(out, "w") as f:
            json.dump({"shape": dict(B=B, T=T, F=F, H=H, L=L, C=C), "reference": "oracle/bigru_oracle.OracleBiGRU (torch.nn.GRU CPU fp32)",
                       "errors": report}, f, indent=1)


def test_shard_gradients_sum_to_full_batch():
    """Data-parallel property: the shard gradients of the global-mean loss add up to the full-batch
    gradient (what the single all-reduce computes)."""
    B, T, F, H, L, C = 64, 10, 16, 128, 2, 3
    for precision in precisions():
        torch.manual_seed(1)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=precision).cuda()
        x = torch.randn(B, T, F, device="cuda")
        t = torch.randint(0, C, (B,), device="cuda")
        ce = nn.CrossEntropyLoss(reduction="sum")

        def grad(xs, ts):
            m.zero_grad()
            (ce(m(xs), ts) / B).backward()
            return torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).clone()

        full = grad(x, t)
        parts = grad(x[:32], t[:32]) + grad(x[32:], t[32:])
        assert rel_l2(parts.cpu().numpy(), full.cpu().numpy()) < (1e-5 if precision == "fp32" else 2e-2)


def test_linearity_in_upstream_gradient():
    """Size-independent property at a realistic size: backward is linear in dlogits."""
    B, T, F, H, L, C = 128, 32, 64, 256, 2, 3
    for precision in precisions():
        torch.manual_seed(2)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=precision).cuda()
        x = torch.randn(B, T, F, device="cuda")
        d1, d2 = torch.randn(B, C, device="cuda"), torch.randn(B, C, device="cuda")

        def grad(dl):
            m.zero_grad()
            m(x).backward(dl)
            return torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).clone()

        lhs = grad(d1 + 2 * d2)
        rhs = grad(d1) + 2 * grad(d2)
        assert rel_l2(lhs.cpu().numpy(), rhs.cpu().numpy()) < (1e-4 if precision == "fp32" else 2e-2)


def test_dropout_modes():
    """Train-mode dropout: elementwise and channel-wise ('spatial', one mask per (b, f) over T) input
    masks, inter-layer dropout; same mask in backward (dx is zero exactly where the input was dropped)."""
    for precision, spatial in [(p, s) for p in precisions() for s in (False, True)]:
        B, T, F, H, L, C = (16, 12, 24, 32, 2, 3) if precision == "fp32" else (32, 12, 24, 128, 2, 3)
        torch.manual_seed(4)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.5, spatial, True, precision=precision).cuda()
        m.train()
        x = (torch.rand(B, T, F, device="cuda") + 0.5).requires_grad_(True)
        y1 = m(x)
        y1.sum().backward()
        dx = x.grad.clone()
        zero = (dx == 0)
        frac = zero.float().mean().item()
        assert 0.35 < frac < 0.65, frac
        if spatial:
            per_channel = zero.all(dim=1) | (~zero).all(dim=1)          # a channel is dropped for all T or none
            assert per_channel.all()
        y2 = m(x)
        assert not torch.equal(y1, y2)                                   # fresh mask per call
        m.eval()
        with torch.no_grad():
            assert torch.equal(m(x), m(x))                               # eval: deterministic, no dropout


def test_window_gather_matches_reference_loader(golden_dir):
    """The gather/normalise kernel against batches delivered by the unmodified reference loader
    (bit-exact: float32 subtract and IEEE divide)."""
    z = np.load(os.path.join(golden_dir, "loader.npz"))
    cols, targets, fields, query = fake_db.make_table(n_rows=250)
    cur = fake_db.FakeCursor(cols, targets)
    pkg = _pkg()
    ids = tuple(int(v) for v in z["chunk1_ids"])
    norm = (torch.from_numpy(z["chunk1_min"]), torch.from_numpy(z["chunk1_max"]))
    for bs in (2, 8):
        ds = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 30)
        assert np.array_equal(ds.x.cpu().numpy(), z[f"bs{bs}_xnorm"])
        xs, ys = zip(*[(x.cpu().numpy(), y.cpu().numpy()) for x, y in ds.batches(bs)])
        assert len(xs) == int(z[f"bs{bs}_nbatches"])
        assert np.array_equal(np.concatenate(xs), z[f"bs{bs}_x"])
        assert np.array_equal(np.concatenate(ys), z[f"bs{bs}_y"])
        # per-sample drop-in path through torch's DataLoader
        ds2 = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 30)
        got = [(x.cpu().numpy(), y.cpu().numpy()) for x, y in torch.utils.data.DataLoader(ds2, batch_size=bs)]
        assert np.array_equal(np.concatenate([g[0] for g in got]), z[f"bs{bs}_x"])
        assert np.array_equal(np.concatenate([g[1] for g in got]), z[f"bs{bs}_y"])
    tail = list(ds.batches(8, drop_incomplete=False))
    assert sum(x.shape[0] for x, _ in tail) == 100


@pytest.mark.parametrize("shape", [(512, 128, 64), (256, 1024, 128), (7, 3, 5), (1, 1, 1), (0, 4, 8)])
def test_window_gather_property(shape):
    """Full-size property: the collated batch equals the strided view of the chunk (x.unfold)."""
    B, T, F = shape
    pkg = _pkg()
    lib = pkg._lib.load()
    N = B + T - 1 + 3
    src = torch.rand(max(N, 1), F, device="cuda")
    mn = src.min(0).values - 0.1
    mx = src.max(0).values + 0.1
    out = torch.empty(B, T, F, device="cuda")
    pkg._lib.check(lib.bigru_window_gather_norm(src.data_ptr(), mn.data_ptr(), mx.data_ptr(), 2, N, B, T, F,
                                                out.data_ptr(), torch.cuda.current_stream().cuda_stream), "gather")
    if B:
        ref = ((src - mn) / (mx - mn))[2:2 + B + T - 1].unfold(0, T, 1).permute(0, 2, 1)
        assert torch.equal(out, ref.contiguous())
        ref_c = oracle_c.window_gather_norm(src.cpu().numpy(), mn.cpu().numpy(), mx.cpu().numpy(), 2, min(B, 4), T)
        assert np.array_equal(out[:4].cpu().numpy(), ref_c)
    # out-of-range windows are an argument error, not a silent clamp
    with pytest.raises(ValueError):
        pkg._lib.check(lib.bigru_window_gather_norm(src.data_ptr(), None, None, N, N, 1, T, F, out.data_ptr(), 0), "gather")


def test_train_and_evaluate_model_surface():
    """train_model / evaluate_model return tuples (biGRU_model.py:224, :286); device metric counters
    against sklearn on the same logits."""
    from sklearn.metrics import accuracy_score, fbeta_score, hamming_loss
    cols, targets, fields, query = fake_db.make_table(n_rows=120, with_nulls=False)
    cur = fake_db.FakeCursor(cols, targets)
    pkg = _pkg()
    cl = pkg.MySQLChunkLoader(cur, "stock_data_joined", query, 60, 10, norm_params_path=None)
    ids, norm = cl[1]
    torch.manual_seed(0)
    m = pkg.BiGRU(16, len(fields), 4, 1, 50, 0.0, False, True).cuda()
    m.add_loss_fn(nn.BCEWithLogitsLoss(pos_weight=torch.tensor([2.0, 1.0, 3.0, 1.5])))
    m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
    m.add_device(torch.device("cuda"))
    assert m.can_fuse_step()
    ds = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 10)
    acc, ham, loss, fb = m.train_model(ds.batches(8))
    assert 0 <= acc <= 1 and 0 <= ham <= 1 and np.isfinite(loss) and fb.shape == (4,)
    ds = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 10)
    batches = list(ds.batches(8))
    acc, ham, fb, pred_total, target_total = m.evaluate_model(batches)
    assert pred_total.dtype == torch.int64 and pred_total.shape == target_total.shape == (len(batches) * 8, 4)
    accs, hams, fbs = [], [], []
    m.eval()
    with torch.no_grad():
        for x, y in batches:
            p = (torch.sigmoid(m(x)) > 0.5).cpu().numpy()
            t = y.squeeze(1).cpu().numpy()
            accs.append(accuracy_score(t, p)); hams.append(hamming_loss(t, p))
            fbs.append(fbeta_score(t, p, beta=0.5, average=None, zero_division=0))
    assert abs(acc - np.mean(accs)) < 1e-12 and abs(ham - np.mean(hams)) < 1e-12
    np.testing.assert_allclose(fb, np.mean(fbs, axis=0), atol=1e-12)
    # generic (non-fusable) optimiser goes through autograd and the same kernels
    m.add_optimizer(torch.optim.SGD(m.parameters(), lr=1e-2))
    assert not m.can_fuse_step()
    ds = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 10)
    out = m.train_model(torch.utils.data.DataLoader(ds, batch_size=4))
    assert np.isfinite(out[2])
    # class-index targets cannot feed the multilabel metrics (sklearn raises ValueError in the reference)
    m.add_loss_fn(nn.CrossEntropyLoss())
    with pytest.raises(ValueError):
        m.train_model([(torch.rand(4, 10, len(fields)), torch.zeros(4, 1, dtype=torch.long))])


def test_fused_step_matches_generic_step():
    """train_step (C-ABI calls only) and the autograd + torch.optim path give the same parameters."""
    B, T, F, H, L, C = 32, 8, 16, 32, 2, 4
    pkg = _pkg()
    x = torch.randn(B, T, F, device="cuda")
    t = (torch.rand(B, C, device="cuda") < 0.3).float()
    outs = []
    for fused in (True, False):
        torch.manual_seed(5)
        m = pkg.BiGRU(H, F, C, L, 1, 0.0, False, True).cuda()           # clip=1 so that clipping is active
        m.add_loss_fn(nn.MultiLabelSoftMarginLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-2))
        m.train()
        for _ in range(3):
            if fused:
                m.train_step(x, t)
            else:
                m._generic_step(x, t)
        outs.append(m.flat_parameters().clone())
    assert rel_l2(outs[0].cpu().numpy(), outs[1].cpu().numpy()) < 1e-5


def test_error_conventions():
    pkg = _pkg()
    lib = pkg._lib.load()
    h = pkg._lib.C.c_void_p()
    assert lib.bigru_plan_create(0, 4, 4, 4, 1, 2, 1, 0, pkg._lib.C.byref(h)) == pkg._lib.ERR_ARG
    assert b"bad shape" in lib.bigru_last_error()
    m = pkg.BiGRU(8, 4, 2, 1).cuda()
    with pytest.raises(ValueError):
        m(torch.zeros(2, 3, 5))                       # wrong feature count
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 3, 4), torch.zeros(1, 2, 8))  # wrong hidden shape
    with pytest.raises(RuntimeError):
        pkg.BiGRU(8, 4, 2, 1)(torch.zeros(2, 3, 4))    # parameters on CPU: no CPU path


def test_auto_precision_and_batch_padding():
    """precision="auto" runs the fp32-class tensor-core path for H in {128, 256}; batch sizes that are not whole batch tiles
    run zero-padded (the padded rows get a zero upstream gradient).  Logits, loss, input gradient and every parameter gradient
    of an odd batch must match the oracle like a whole-tile batch does; the fused train step (plain and CUDA graph) too."""
    pkg = _pkg()
    T, F, H, L, C = 12, 16, 128, 2, 3
    for prec, b in (("auto", 64), ("auto", 61), ("bf16", 19), ("auto", 1)):
        torch.manual_seed(3)
        ref = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
        m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision=prec)
        m.load_state_dict(ref.state_dict())
        m = m.cuda()
        tol_l, tol_g = ((1e-4, 1e-3) if prec == "auto" else (3e-2, 6e-2))
        assert m.resolved_precision(b) == ("bf16x3" if prec == "auto" else "bf16")
        g = torch.Generator().manual_seed(b)
        x = torch.randn(b, T, F, generator=g)
        y = torch.randint(0, C, (b,), generator=g)
        xr = x.clone().requires_grad_(True)
        lr_ = nn.functional.cross_entropy(ref(xr), y)
        lr_.backward()
        xg = x.cuda().requires_grad_(True)
        out = m(xg)
        assert out.shape == (b, C)
        lg = nn.functional.cross_entropy(out, y.cuda())
        lg.backward()
        with torch.no_grad():
            want = ref(x)
        assert float((out.detach().cpu() - want).abs().max() / want.abs().max()) <= tol_l
        assert abs(float(lg.detach()) - float(lr_.detach())) <= tol_l * max(1.0, abs(float(lr_.detach())))
        assert rel_l2(xg.grad.cpu().numpy(), xr.grad.numpy()) <= tol_g
        for (k, p_ref), (_, p_gpu) in zip(ref.named_parameters(), m.named_parameters()):
            assert rel_l2(p_gpu.grad.cpu().numpy(), p_ref.grad.numpy()) <= tol_g * 3, k
        assert m.pooled_argmax().shape == (b, H)
        # fused step on the odd batch: loss and logits of the real rows, plain launches and graph replay
        m.add_loss_fn(nn.CrossEntropyLoss()); m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
        for it in range(3):
            loss, logits = m.train_step(x.cuda(), y.cuda())
            assert logits.shape == (b, C) and bool(torch.isfinite(loss).all())
            if it == 0:
                assert abs(float(loss) - float(lr_.detach())) <= tol_l * max(1.0, abs(float(lr_.detach())))


def test_fused_adam_state_lives_in_the_optimizer():
    """The fused train step keeps Adam's moments in flat buffers; optimizer.state mirrors them (views + step counters) in
    torch.optim.Adam's own format: a checkpoint of optimizer.state_dict() resumes the fused step, and the generic autograd step
    (any loss / optimiser route) continues from the same moments."""
    import copy
    pkg = _pkg()
    B, T, F, H, L, C = 8, 5, 6, 12, 1, 3
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, T, F, generator=g).cuda()
    y = torch.randint(0, C, (B,), generator=g).cuda()

    def fresh(state=None):
        torch.manual_seed(2)
        m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision="fp32").cuda()
        if state is not None:
            m.load_state_dict(state)
        m.add_loss_fn(nn.CrossEntropyLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-2))
        return m.train()

    m1 = fresh()
    for _ in range(3):
        m1.train_step(x, y)
    sd_opt = copy.deepcopy(m1.optimizer.state_dict())
    sd_model = {k: v.clone() for k, v in m1.state_dict().items()}
    st = sd_opt["state"]
    assert len(st) == len(list(m1.parameters())) and all(int(float(v["step"])) == 3 for v in st.values())
    assert all(float(v["exp_avg"].abs().max()) > 0 for v in st.values())
    for _ in range(2):
        m1.train_step(x, y)
    want = torch.cat([p.detach().reshape(-1) for p in m1.parameters()]).cpu()
    # (b) resume from the checkpoint, fused
    m2 = fresh(sd_model)
    m2.optimizer.load_state_dict(sd_opt)
    for _ in range(2):
        m2.train_step(x, y)
    got = torch.cat([p.detach().reshape(-1) for p in m2.parameters()]).cpu()
    assert float((got - want).abs().max()) < 1e-6
    assert all(int(float(v["step"])) == 5 for v in m2.optimizer.state_dict()["state"].values())
    # (c) resume from the checkpoint, generic autograd step with torch's own Adam arithmetic
    m3 = fresh(sd_model)
    m3.optimizer.load_state_dict(sd_opt)
    for _ in range(2):
        m3._generic_step(x, y)
    got3 = torch.cat([p.detach().reshape(-1) for p in m3.parameters()]).cpu()
    assert float((got3 - want).abs().max()) < 2e-4
    # a per-element BCE weight cannot be fused: the step falls back to autograd instead of raising
    mb = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision="fp32").cuda().train()
    mb.add_loss_fn(nn.BCEWithLogitsLoss(weight=torch.rand(B, C).cuda()))
    mb.add_optimizer(torch.optim.Adam(mb.parameters(), lr=1e-3))
    assert not mb.can_fuse_step()


def test_model_on_a_device_that_is_not_current():
    """A model on cuda:1 while cuda:0 is the current device: every C-ABI call must run on the model's device and stream (per-device
    shared-memory opt-ins, device guards in the mirror); results equal the same model on cuda:0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    pkg = _pkg()
    B, T, F, H, L, C = 32, 6, 16, 128, 2, 3
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, T, F, generator=g)
    y = torch.randint(0, C, (B,), generator=g)
    torch.cuda.set_device(0)
    for prec in precisions():
        outs = []
        for dev in (0, 1):
            torch.manual_seed(4)
            m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision=prec).to(f"cuda:{dev}").train()
            m.add_loss_fn(nn.CrossEntropyLoss()); m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
            assert torch.cuda.current_device() == 0
            for _ in range(3):
                loss, logits = m.train_step(x.to(f"cuda:{dev}"), y.to(f"cuda:{dev}"))
            outs.append((float(loss), logits.cpu(), m.flat_parameters().cpu()))
        tol = 1e-6 if prec != "bf16" else 5e-3
        assert abs(outs[0][0] - outs[1][0]) <= tol and float((outs[0][1] - outs[1][1]).abs().max()) <= tol * 10
        assert float((outs[0][2] - outs[1][2]).abs().max()) <= tol * 10


def test_long_sequence_config_reduced():
    """BASELINE config 4 (B256,T1024,F128,H512,L2) at reduced batch/length on the exact FFMA path (logits <= 1e-4 rel of the
    torch.nn.GRU CPU path); the bf16x3 path must refuse H = 512 loudly (its split weights do not fit tensor memory)."""
    B, T, F, H, L, C = 16, 256, 128, 512, 2, 3
    torch.manual_seed(0)
    ref = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(B, T, F, generator=g)
    ref.eval()
    with torch.no_grad():
        want = ref(x).numpy()
    torch.manual_seed(0)
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision="fp32").cuda()
    m.eval()
    with torch.no_grad():
        got = m(x.cuda()).cpu().numpy()
    assert rel(got, want) < 1e-4
    if "bf16x3" in precisions():
        mb = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision="bf16x3").cuda()
        with pytest.raises(ValueError, match="hidden_size 128 or 256"):
            mb(x.cuda())


def test_long_sequence_config_on_tensor_cores():
    """BASELINE configs[4] at its FULL sequence length, feature count and hidden size (T1024, F128, H512, L2, bidirectional) on the
    persistent 8-CTA-cluster tensor-core kernels (precision="bf16", tc_scan_w.cuh), batch 64 so that the torch.nn.GRU CPU
    oracle (forward + autograd) finishes in about a minute: logits and every gradient against the oracle at the bf16 path's
    tolerances, the training step against the exact FFMA path's loss."""
    if "bf16" not in precisions():
        pytest.skip("tensor-core path not built")
    B, T, F, H, L, C = 64, 1024, 128, 512, 2, 3
    tol = TOL["bf16"]
    torch.manual_seed(0)
    ref = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
    g = torch.Generator().manual_seed(99)
    x = torch.randn(B, T, F, generator=g)
    y = torch.randint(0, C, (B,), generator=g)
    ref.train()
    out_ref = ref(x)
    loss_ref = nn.functional.cross_entropy(out_ref, y)
    loss_ref.backward()
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision="bf16")
    m.load_state_dict(ref.state_dict())
    m = m.cuda().train()
    out = m(x.cuda())
    loss = nn.functional.cross_entropy(out, y.cuda())
    loss.backward()
    e_log = rel(out.detach().cpu().numpy(), out_ref.detach().numpy())
    got = torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).cpu().numpy()
    want = torch.cat([p.grad.reshape(-1) for p in ref.parameters()]).numpy()
    e_g = rel_l2(got, want)
    print(f"configs[4] (B{B}) bf16 tensor-core path: logits rel {e_log:.3e}, gradient flat rel-L2 {e_g:.3e}")
    path = os.environ.get("BIGRU_PARITY_REPORT_C4")
    if path:
        with open(path, "w") as f:
            json.dump({"shape": dict(B=B, T=T, F=F, H=H, L=L, C=C), "precision": "bf16", "logits_rel": e_log, "grad_flat_rel_l2": e_g,
                       "loss": float(loss.detach()), "loss_reference": float(loss_ref.detach())}, f, indent=1)
    assert e_log < tol["logits"], e_log
    assert e_g < tol["gflat"], e_g
    assert abs(float(loss.detach()) - float(loss_ref.detach())) < 3e-2


def test_training_trajectories_agree():
    """Ten fused optimisation steps: the tensor-core path follows the fp32 path's loss trajectory."""
    if "bf16" not in precisions():
        pytest.skip("tensor-core path not built")
    B, T, F, H, L, C = 64, 24, 32, 128, 2, 3
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, T, F, generator=g).cuda()
    t = torch.randint(0, C, (B,), generator=g).cuda()
    traj = {}
    for precision in ("fp32", "bf16"):
        torch.manual_seed(1)
        m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=precision).cuda()
        m.add_loss_fn(nn.CrossEntropyLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=3e-3))
        m.train()
        traj[precision] = [float(m.train_step(x, t)[0]) for _ in range(10)]
    a, b = np.array(traj["fp32"]), np.array(traj["bf16"])
    assert a[-1] < a[0] * 0.8                       # it learns
    assert np.abs(a - b).max() < 0.03 * a[0], (a, b)


def test_two_gpu_data_parallel_step_matches_single_gpu(tmp_path):
    """Batch data parallelism over NCCL: two ranks with half the batch each end up with the parameters of one
    rank stepping on the whole batch (one all-reduce of the flat gradient, loss normalised by the global batch)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import subprocess, sys, textwrap
    script = tmp_path / "dp.py"
    script.write_text(textwrap.dedent('''
        import os, sys, torch, torch.nn as nn, torch.distributed as dist
        sys.path.insert(0, os.environ["REPO"])
        import financial_market_data_analysis_b200 as pkg
        from financial_market_data_analysis_b200.parallel import shard_batch
        rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        g = torch.Generator().manual_seed(3)
        x = torch.randn(64, 12, 16, generator=g); t = torch.randint(0, 3, (64,), generator=g)
        def run(dp, prec, graph="1"):
            os.environ["BIGRU_B200_CUDA_GRAPH"] = graph
            torch.manual_seed(0)
            m = pkg.BiGRU(128, 16, 3, 2, 1, 0.0, False, True, precision=prec).cuda()
            m.add_loss_fn(nn.CrossEntropyLoss()); m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-2)); m.train()
            if dp:
                m.enable_data_parallel()
                xs, ts = shard_batch(x, rank, world), shard_batch(t, rank, world)
            else:
                xs, ts = x, t
            for _ in range(4):
                loss, _ = m.train_step(xs.cuda(), ts.cuda())
            return m.flat_parameters().clone(), float(loss)
        # fp32: the exact path; bf16x3: the tensor-core path, with and without the split backward whose upper-layer all-reduce
        # overlaps layer 0 (BIGRU_B200_DP_OVERLAP=1), captured in CUDA graphs and with plain launches
        for prec, overlap, graph, tol in (("fp32", "0", "1", 1e-5), ("bf16x3", "0", "1", 2e-3), ("bf16x3", "1", "1", 2e-3), ("bf16x3", "1", "0", 2e-3)):
            os.environ["BIGRU_B200_DP_OVERLAP"] = overlap
            pd, ld = run(True, prec, graph); ps, ls = run(False, prec, graph)
            err = float((pd - ps).norm() / ps.norm())
            if rank == 0: print("DPERR", prec, overlap, graph, err, ld, ls)
            assert err < tol and abs(ld - ls) < tol, (prec, overlap, err, ld, ls)
        dist.destroy_process_group()
    '''))
    env = dict(os.environ, REPO=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "DPERR" in out.stdout


def test_zero_copy_windows_match_collated_batches():
    """SURVEY.md 8(f) N1: forward / train step straight from the chunk equal collate-then-forward (same arithmetic,
    so the fp32 path is bit-exact on the logits)."""
    cols, targets, fields, query = fake_db.make_table(n_rows=200, with_nulls=False, n_plain=2, levels=2)
    cur = fake_db.FakeCursor(cols, targets)
    pkg = _pkg()
    cl = pkg.MySQLChunkLoader(cur, "stock_data_joined", query, 200, 12, norm_params_path=None)
    ids, norm = cl[0]
    F = len(fields)
    for precision in precisions():
        H = 32 if precision == "fp32" else 128
        if not supported(precision, 32, F, H):
            continue
        ds = pkg.MySQLBatchLoader(ids, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 12)
        torch.manual_seed(0)
        m = pkg.BiGRU(H, F, 4, 2, 50, 0.0, False, True, precision=precision).cuda()
        m.eval()
        x, y = ds.collate(5, 32)
        with torch.no_grad():
            want = m(x)
        got = m.forward_windows(ds, 5, 32)
        if precision == "fp32":
            assert torch.equal(got, want)
        else:
            assert rel(got.cpu().numpy(), want.cpu().numpy()) < 1e-6
        # training step: same parameters afterwards
        outs = []
        for mode in ("collated", "windows"):
            torch.manual_seed(0)
            mm = pkg.BiGRU(H, F, 4, 2, 1, 0.0, False, True, precision=precision).cuda()
            mm.add_loss_fn(nn.BCEWithLogitsLoss()); mm.add_optimizer(torch.optim.Adam(mm.parameters(), lr=1e-2)); mm.train()
            if mode == "collated":
                mm.train_step(x, y.squeeze(1))
            else:
                mm.train_step_windows(ds, 5, 32)
            outs.append(mm.flat_parameters().clone())
        assert rel_l2(outs[1].cpu().numpy(), outs[0].cpu().numpy()) < (1e-6 if precision == "fp32" else 1e-3)
    with pytest.raises(ValueError):
        m.forward_windows(ds, 170, 32)


def test_chunk_statistics_on_gpu_match_sql_path(golden_dir, tmp_path):
    """SURVEY.md 8(f) N3: per-chunk MIN/MAX from the reduction kernel + host guard / order-book rules equal what the
    unmodified reference computed through SQL aggregates (tests/golden/loader.npz)."""
    z = np.load(os.path.join(golden_dir, "loader.npz"))
    cols, targets, fields, query = fake_db.make_table(n_rows=250)
    import financial_market_data_analysis_b200.sql_pytorch_dataloader as L
    L.bid_levels, L.ask_levels = 2, 2
    table = torch.tensor(np.stack([cols[f] for f in fields], 1), dtype=torch.float32).cuda()      # NaN = NULL
    cl = L.MySQLChunkLoader.from_table(table, fields, 100, 30, norm_params_path=str(tmp_path / "norm_params"))
    assert len(cl) == int(z["n_chunks"])
    for i in range(len(cl)):
        ids, (mn, mx) = cl[i]
        assert np.array_equal(np.array(ids), z[f"chunk{i}_ids"])
        assert np.array_equal(mn.numpy(), z[f"chunk{i}_min"]) and np.array_equal(mx.numpy(), z[f"chunk{i}_max"])


# ---- SURVEY.md 8(f) N4: SQL window-function features on the GPU --------------------------------------------------------
def _market_columns(n, seed=5):
    rng = np.random.default_rng(seed)
    close = 2900 + np.cumsum(rng.normal(0, 2.0, n))
    cols = [close, close + rng.uniform(0.1, 3.0, n), close - rng.uniform(0.1, 3.0, n),
            rng.integers(100, 50000, n).astype(np.float64), rng.normal(0, 300, n)]
    return [np.float32(c) for c in cols]


@pytest.mark.gpu
def test_window_features_other_periods_match_oracle():
    """periods other than the reference's config.py take the generic (run-time period) code path"""
    from oracle import features_oracle as fo
    from financial_market_data_analysis_b200.features import window_features
    for kw in (dict(volume_MA_periods=[3, 10], price_MA_periods=[7, 31], delta_MA_periods=[5], bollinger_bands_period=10,
                    bollinger_bands_std=1.5, stochastic_oscillator=False),
               dict(volume_MA_periods=[], price_MA_periods=[300], delta_MA_periods=[], bollinger_bands_period=False,
                    bollinger_bands_std=2, stochastic_oscillator=True)):
        cols = _market_columns(3000, seed=9)
        ref_f, ref_t = fo.window_features(*[c.astype(np.float64) for c in cols], **kw)
        got_f, got_t = window_features(*[torch.from_numpy(c).cuda() for c in cols], **kw)
        g = got_f.cpu().numpy()
        assert g.shape == ref_f.shape and np.array_equal(np.isnan(g), np.isnan(ref_f))
        np.testing.assert_allclose(np.nan_to_num(g), np.nan_to_num(ref_f), rtol=2e-6, atol=5e-4)
        assert np.array_equal(got_t.cpu().numpy(), ref_t)


@pytest.mark.gpu
def test_window_features_match_reference_sql(golden_dir):
    """SURVEY.md 8(f) N4 against the reference's own SQL (tests/golden/features.npz: create_database.py's views executed
    unmodified through sqlite3): the kernel's features, NULL positions and target labels."""
    from financial_market_data_analysis_b200.features import window_features
    z = np.load(os.path.join(golden_dir, "features.npz"))
    cols = [torch.from_numpy(z[k].astype(np.float32)).cuda() for k in ("close", "high", "low", "volume", "delta")]
    got_f, got_t = window_features(*cols, volume_MA_periods=[int(v) for v in z["volume_MA_periods"]],
                                   price_MA_periods=[int(v) for v in z["price_MA_periods"]], delta_MA_periods=[int(v) for v in z["delta_MA_periods"]],
                                   bollinger_bands_period=int(z["bollinger_bands_period"]), bollinger_bands_std=float(z["bollinger_bands_std"]),
                                   stochastic_oscillator=True)
    g = got_f.cpu().numpy()
    assert np.array_equal(np.isnan(g), np.isnan(z["features"]))
    np.testing.assert_allclose(np.nan_to_num(g), np.nan_to_num(z["features"]), rtol=2e-6, atol=5e-4)
    assert np.array_equal(got_t.cpu().numpy(), z["targets"])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 16, 500, 20000])
def test_window_features_match_oracle(n):
    from oracle import features_oracle as fo
    from financial_market_data_analysis_b200.features import window_features, feature_names
    cols = _market_columns(n)
    if n == 500:
        cols[0][100:140] = cols[0][100]                                       # flat stretch: stochastic max == min -> NULL
    kw = dict(volume_MA_periods=[6, 20], price_MA_periods=[20], delta_MA_periods=[12], bollinger_bands_period=20,
              bollinger_bands_std=2, stochastic_oscillator=True)
    ref_f, ref_t = fo.window_features(*[c.astype(np.float64) for c in cols], **kw)
    got_f, got_t = window_features(*[torch.from_numpy(c).cuda() for c in cols], **kw)
    assert got_f.shape == (n, len(feature_names(**kw))) and got_t.shape == (n, 4)
    g = got_f.cpu().numpy()
    assert np.array_equal(np.isnan(g), np.isnan(ref_f))                        # SQL NULLs in the same places
    # double arithmetic rounded once to fp32: differences of large prices keep an absolute error of one fp32 ulp of the price
    np.testing.assert_allclose(np.nan_to_num(g), np.nan_to_num(ref_f), rtol=2e-6, atol=5e-4)
    assert np.array_equal(got_t.cpu().numpy(), ref_t)                          # labels are exact


@pytest.mark.gpu
def test_window_features_properties_large():
    from financial_market_data_analysis_b200.features import window_features
    n = 2_000_000
    g = torch.Generator(device="cuda").manual_seed(3)
    close = 3000 + torch.cumsum(torch.randn(n, device="cuda", generator=g), 0)
    spread = torch.rand(n, device="cuda", generator=g) + 0.5
    f, t = window_features(close, close + spread, close - spread, torch.full((n,), 7.0, device="cuda"), torch.zeros(n, device="cuda"))
    assert torch.all(f[:, 2] == 7) and torch.all(f[:, 3] == 7) and torch.all(f[:, 5] == 0)      # averages of constants
    assert torch.all((f[:, 0] + f[:, 1]) >= -1e-2)                              # upper + lower distance = 4 * std >= 0
    s = f[15:, 6]
    assert torch.all((s >= 0) & (s <= 1) | torch.isnan(s))                      # stochastic oscillator in [0, 1]
    assert torch.allclose(f[1:, 8], close[1:] - close[:-1], atol=1e-3)          # price change telescopes
    assert t[-8:, 0].sum() == 0 and t[-15:, 1].sum() == 0 and float((t[:, 0] * t[:, 2]).sum()) == 0   # up and down exclude each other


@pytest.mark.gpu
def test_window_features_errors():
    from financial_market_data_analysis_b200.features import window_features
    x = torch.ones(8)
    with pytest.raises(RuntimeError):
        window_features(x, x, x, x, x)                                           # CPU tensors: no fallback
    xc = x.cuda()
    with pytest.raises(ValueError):
        window_features(xc, xc, xc, None, xc)                                    # volume MA without the column
    with pytest.raises(ValueError):
        window_features(xc, xc, xc, xc, xc, volume_MA_periods=list(range(1, 10)))   # more than 8 periods


# ---- SURVEY.md 8(f) N5: the live predictor's forward in one launch -----------------------------------------------------
@pytest.mark.gpu
def test_live_predictor_known_answers(golden_dir):
    """predict.py's model block on the shipped checkpoint: KAT logits (<= 1e-5), sigmoid, labels; raw windows + norm params."""
    from financial_market_data_analysis_b200.predict import LivePredictor
    z = np.load(os.path.join(golden_dir, "kat.npz"))
    state = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("p:")}
    lp = LivePredictor(state, None)
    for i in (1, 2, 3):
        logits, probs = lp.forward_windows(z[f"x{i}"])
        assert np.abs(logits.cpu().numpy() - z[f"y{i}"]).max() < 1e-5
        assert np.abs(probs.cpu().numpy() - 1 / (1 + np.exp(-z[f"y{i}"]))).max() < 1e-5
        same = lp.model(torch.from_numpy(z[f"x{i}"]).cuda())                 # the step-by-step path of the same model
        assert np.abs(same.detach().cpu().numpy() - logits.cpu().numpy()).max() < 1e-5
    # raw rows + pickled-style norm params (predict.py:110-122, :170): same as normalising first
    mn, mx = z["norm_min"].astype(np.float32), z["norm_max"].astype(np.float32)
    lpn = LivePredictor(state, (mn, mx), prob_threshold=0.5)
    rng = np.random.default_rng(0)
    raw = (mn + rng.uniform(0, 1, (5, mn.size)) * (mx - mn)).astype(np.float32)
    out = lpn.predict(raw, "2020-03-02 10:05:00")
    want_logits, _ = lp.forward_windows(((raw - mn) / (mx - mn))[None])
    want = 1 / (1 + np.exp(-want_logits.cpu().numpy()[0]))
    assert np.abs(out["probabilities"].numpy() - want).max() < 1e-5
    assert list(out["pred_indices"]) == list(np.where(want > 0.5)[0])
    assert out["pred_labels"] == [lpn.y_fields[i] for i in out["pred_indices"]] and out["timestamp"] == "2020-03-02 10:05:00"


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(3, 7, 12, 16, 2, 3, True), (2, 9, 5, 33, 1, 2, False), (1, 4, 64, 128, 2, 4, True)])
def test_infer_window_matches_c_oracle(cfg):
    B, T, F, H, L, C, bidir = cfg
    D = 2 if bidir else 1
    torch.manual_seed(5)
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, bidir, precision="fp32").cuda().eval()
    x = torch.randn(B, T, F, generator=torch.Generator().manual_seed(2))
    flat = m.flat_parameters().cpu().numpy()
    ref_logits, _, _ = oracle_c.forward(flat, x.numpy(), H, L, C, D, None, keep=True)
    from financial_market_data_analysis_b200 import _lib
    lib = _lib.load()
    logits = torch.empty(B, C, device="cuda"); probs = torch.empty(B, C, device="cuda")
    xc = x.cuda()
    _lib.check(lib.bigru_infer_window(_lib.ptr(m.flat_parameters()), _lib.ptr(xc), None, None, B, T, F, H, L, C, int(bidir), _lib.ptr(logits),
                                      _lib.ptr(probs), torch.cuda.current_stream().cuda_stream), "bigru_infer_window")
    scale = max(np.abs(ref_logits).max(), 1e-3)
    assert np.abs(logits.cpu().numpy() - ref_logits).max() / scale < 1e-5
    with pytest.raises(ValueError):                                          # D*H above one CTA: belongs to bigru_forward
        _lib.check(lib.bigru_infer_window(_lib.ptr(m.flat_parameters()), _lib.ptr(xc), None, None, B, T, F, 1024, L, C, 1, _lib.ptr(logits),
                                          _lib.ptr(probs), torch.cuda.current_stream().cuda_stream), "bigru_infer_window")


def test_cuda_graph_step_matches_plain_launches():
    """SURVEY.md 8(f) N5: the train step replayed from a captured CUDA graph (static buffers, device-resident Adam step
    counter) follows the same parameter trajectory as plain C-ABI launches."""
    B, T, F, H, L, C = 64, 12, 16, 128, 2, 3
    g = torch.Generator().manual_seed(5)
    xs = [torch.randn(B, T, F, generator=g).cuda() for _ in range(5)]
    ts = [torch.randint(0, C, (B,), generator=g).cuda() for _ in range(5)]
    for precision in precisions():
        out = {}
        for graph in (False, True):
            torch.manual_seed(9)
            m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=precision).cuda()
            m.use_cuda_graph = graph
            m.add_loss_fn(nn.CrossEntropyLoss())
            m.add_optimizer(torch.optim.Adam(m.parameters(), lr=2e-3))
            m.train()
            losses = [float(m.train_step(x, t)[0]) for x, t in zip(xs, ts)]
            if graph:
                assert m.use_cuda_graph and len(m._graphs) == 1, "the step was not captured"
                assert int(m._adam["dstep"].item()) == 5 and m._adam["step"] == 5
            out[graph] = (np.array(losses), m.flat_parameters().cpu().numpy())
        print(f"graph[{precision}] losses plain {out[False][0]} graph {out[True][0]} param rel-L2 {rel_l2(out[True][1], out[False][1]):.2e}")
        # not bit-exact: split-K partial sums land in a run-dependent order, and the bf16 path rounds activations after them
        # (measured: fp32 4e-8, bf16x3 2e-7, bf16 1.4e-3 relative on the parameters after five steps)
        ltol, ptol = (1e-3, 1e-2) if precision == "bf16" else (1e-5, 1e-5)
        assert np.abs(out[True][0] - out[False][0]).max() < ltol, precision
        assert rel_l2(out[True][1], out[False][1]) < ptol, precision


@pytest.mark.parametrize("F", [64, 24])
def test_zero_copy_windows_against_loader_and_model_oracles(F):
    """SURVEY.md 8(f) N1 against the ORACLES (not against the repo's own collation): windows of a chunk through
    ``forward_windows`` / ``train_step_windows`` equal loader_oracle.normalise + collate (sql_pytorch_dataloader.py:239-245)
    followed by the reference model (biGRU_model.py:63-138, :198-210).  B = 128 windows: the tensor-core paths then never
    materialise x[B,T,F] (the chunk is normalised / cast once and addressed as windows by TMA); F = 64 takes the fused
    layer-0 projection of the bf16 scan, F = 24 the projection GEMM."""
    pkg = _pkg()
    B, T, H, L, C = 128, 12, 128, 2, 4
    g = torch.Generator().manual_seed(21)
    n_rows = B + T - 1 + 9
    x_raw = torch.rand(n_rows, F, generator=g) * 50 + 3
    y = (torch.rand(n_rows, C, generator=g) < 0.3).float()
    xmin, xmax = x_raw.min(0, keepdim=True).values - 1, x_raw.max(0, keepdim=True).values + 2
    start = 4
    xb, yb = lo.collate(lo.normalise(x_raw.numpy(), xmin.numpy()[0], xmax.numpy()[0]), y.numpy(), list(range(start, start + B)), T)
    torch.manual_seed(0)
    ref = bo.OracleBiGRU(H, F, C, L, 1.0, 0.0, False, True)
    sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
    ropt = torch.optim.Adam(ref.parameters(), lr=1e-2)
    ref.train()
    want_logits = ref(torch.from_numpy(xb)).detach().numpy()
    bo.train_step(ref, ropt, nn.BCEWithLogitsLoss(), torch.from_numpy(xb), torch.from_numpy(yb[:, 0]))
    want_upd = np.concatenate([(v - sd0[k]).numpy().ravel() for k, v in ref.state_dict().items()])
    for precision in precisions():
        if not supported(precision, B, F, H):
            continue
        tol = TOL[precision]
        ds = pkg.MySQLBatchLoader.from_tensors(x_raw.cuda(), y.cuda(), (xmin, xmax), window=T)
        m = pkg.BiGRU(H, F, C, L, 1.0, 0.0, False, True, precision=precision)
        m.load_state_dict(sd0)
        m = m.cuda()
        m.add_loss_fn(nn.BCEWithLogitsLoss()); m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-2)); m.train()
        got = m.forward_windows(ds, start, B)
        assert rel(got.cpu().numpy(), want_logits) < tol["logits"], (precision, rel(got.cpu().numpy(), want_logits))
        m.train_step_windows(ds, start, B)
        got_upd = np.concatenate([(v.cpu() - sd0[k]).numpy().ravel() for k, v in m.state_dict().items()])
        assert rel_l2(got_upd, want_upd) < tol["update"], (precision, rel_l2(got_upd, want_upd))


def _bigru_uniform(seed, stream, idx):
    """common.cuh bigru_uniform restated: splitmix64 finaliser over (seed, stream, element index) -> [0, 1)."""
    M = np.uint64(0xFFFFFFFFFFFFFFFF)
    idx = np.asarray(idx, np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * (idx + np.uint64(1)) + (np.uint64(stream) << np.uint64(40)) * np.uint64(0xD1B54A32D192ED03)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(40)).astype(np.float64) * (1.0 / 16777216.0)


@pytest.mark.parametrize("spatial", [False, True])
def test_dropout_mask_injection_parity(spatial):
    """A6 by mask injection: the kernels' dropout masks are a pure function of (seed, element index), so the test rebuilds
    them on the host, applies the SAME masks inside the reference computation (input dropout biGRU_model.py:87-94 -
    elementwise or per (b, f) channel over T - and nn.GRU's inter-layer dropout :55) and compares logits and dx."""
    p = 0.3
    for precision in precisions():
        B, T, F, H, L, C = (8, 6, 10, 16, 2, 3) if precision == "fp32" else (32, 6, 16, 128, 2, 3)
        torch.manual_seed(12)
        m = _pkg().BiGRU(H, F, C, L, 50, p, spatial, True, precision=precision).cuda()
        m.train()
        g = torch.Generator().manual_seed(3)
        x = torch.randn(B, T, F, generator=g)
        dl = torch.randn(B, C, generator=g)
        xg = x.cuda().requires_grad_(True)
        y = m(xg)
        y.backward(dl.cuda())
        seed = m._last_seed
        bi, ti, fi = np.meshgrid(np.arange(B), np.arange(T), np.arange(F), indexing="ij")
        key0 = bi * F + fi if spatial else (bi * T + ti) * F + fi
        mask0 = torch.from_numpy((_bigru_uniform(seed, 0, key0) >= p).astype(np.float32) / (1 - p))
        bi, ti, ci = np.meshgrid(np.arange(B), np.arange(T), np.arange(2 * H), indexing="ij")
        mask1 = torch.from_numpy((_bigru_uniform(seed, 1, (bi * T + ti) * (2 * H) + ci) >= p).astype(np.float32) / (1 - p))
        sd = {k: v.detach().cpu().double() for k, v in m.state_dict().items()}
        layers = []
        for l in range(L):
            gl = nn.GRU(F if l == 0 else 2 * H, H, num_layers=1, batch_first=True, bidirectional=True).double()
            gl.load_state_dict({k.replace(f"_l{l}", "_l0").replace("gru.", ""): v for k, v in sd.items() if f"_l{l}" in k})
            layers.append(gl)
        xr = x.double().requires_grad_(True)
        out0, h0n = layers[0](xr * mask0.double())
        out1, h1n = layers[1](out0 * mask1.double())
        last = h1n.sum(0)
        s = out1[..., :H] + out1[..., H:]
        cat = torch.cat([last, s.max(dim=1).values, s.sum(dim=1) / T], dim=1)
        want = cat @ sd["linear.weight"].t() + sd["linear.bias"]
        want.backward(dl.double())
        tol = TOL[precision]
        assert rel(y.detach().cpu().numpy(), want.detach().numpy()) < tol["logits"], (precision, spatial)
        assert rel_l2(xg.grad.cpu().numpy(), xr.grad.numpy()) < tol["grads"] * 5, (precision, spatial)
        assert ((xg.grad.cpu() == 0) == (mask0 == 0)).all()                # dx is zero exactly where the input was dropped
