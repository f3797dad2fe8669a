"""Initial hidden state (biGRU_model.py:63 `hidden`) and its gradient on the bf16 tensor-core path (precision="bf16"):
hidden 128 / 256 (tc_scan.cuh) and 512 (tc_scan_w.cuh), against the C oracle, the reference's autograd and torch.nn.GRU.
Run on the B200 box:  python -m pytest tests/test_bf16_initial_state.py -m gpu -q"""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch
import torch.nn as nn

import golden_cases
import oracle_c
from oracle import bigru_oracle as bo
from test_gpu_parity import TOL, loss_from, make_model, params_of, precisions, rel, rel_l2

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PREC = "bf16"
TB = TOL[PREC]


def _pkg():
    import financial_market_data_analysis_b200 as pkg
    return pkg


@pytest.fixture(autouse=True)
def _needs_bf16():
    if PREC not in precisions():
        pytest.skip("tensor-core path not built")


def _per_tensor_errors(got, want):
    return {k: rel_l2(g, want[k]) for k, g in got.items() if np.abs(g - want[k]).max() >= 1e-7}


SWEEP = [  # B, T, F, H, L, C, bidir
    (32, 9, 64, 128, 2, 3, True),      # H 128 (1-CTA clusters), F = 64: layer-0 projection fused into the forward scan
    (19, 6, 13, 40, 3, 3, True),       # odd batch (zero-padded rows), hidden 40 -> 128, n_features % 8 != 0, three layers
    (40, 5, 108, 128, 1, 4, False),    # the reference's feature count, unidirectional
    (16, 5, 64, 256, 1, 2, False),     # H 256 (2-CTA clusters), fused projection, unidirectional
    (48, 7, 108, 256, 3, 4, True),
    (32, 1, 16, 256, 1, 2, True),      # single time step: the d(h0) product is the only one
    (64, 2, 24, 256, 2, 2, True),
    (32, 300, 8, 256, 1, 2, True),     # many steps: barrier phases of the extra backward product far beyond the ring depths
    (64, 6, 24, 512, 2, 3, True),      # H 512 (8-CTA clusters, tc_scan_w.cuh), two batch tiles
    (32, 1, 16, 512, 1, 2, False),
    (32, 2, 64, 512, 1, 2, True),
    (40, 4, 108, 300, 2, 3, True),     # hidden 300 -> 512, batch 40 -> 64
]


@pytest.mark.parametrize("cfg", SWEEP)
def test_sweep_against_c_oracle(cfg):
    """Logits, h_n, every parameter gradient, dx and dh0 against the C oracle."""
    B, T, F, H, L, C, bidir = cfg
    D = 2 if bidir else 1
    torch.manual_seed(3)
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, bidir, precision=PREC).cuda()
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, T, F, generator=g)
    h0 = torch.randn(L * D, B, H, generator=g) * 0.5
    dl = torch.randn(B, C, generator=g)
    flat = m.flat_parameters().cpu().numpy()
    ref_logits, ref_hn, stash = oracle_c.forward(flat, x.numpy(), H, L, C, D, h0.numpy(), keep=True)
    ref_g, ref_dx, ref_dh0 = oracle_c.backward(flat, x.numpy(), stash, dl.numpy(), H, L, C, D)
    xg = x.cuda().requires_grad_(True)
    hg = h0.cuda().requires_grad_(True)
    y = m(xg, hg)
    y.backward(dl.cuda())
    scale = max(np.abs(ref_logits).max(), 1e-3)
    assert np.abs(y.detach().cpu().numpy() - ref_logits).max() / scale < TB["logits"], cfg
    assert rel(m._last_hidden.cpu().numpy(), ref_hn) < TB["logits"] * 10, cfg
    got = {o: p.grad.reshape(-1).cpu().numpy() for p, (o, _, _) in zip(m._ordered_params(), m._views)}     # C-ABI order
    want = {o: ref_g[o:o + n] for (o, n, _) in m._views}
    errs = _per_tensor_errors(got, want)
    assert all(v < TB["grads"] for v in errs.values()), (cfg, errs)
    gflat = np.concatenate([got[o] for (o, _, _) in m._views])
    assert rel_l2(gflat, ref_g) < TB["gflat"], (cfg, rel_l2(gflat, ref_g))
    assert rel_l2(xg.grad.cpu().numpy(), ref_dx) < TB["grads"], cfg
    assert rel_l2(hg.grad.cpu().numpy(), ref_dh0) < TB["grads"], (cfg, rel_l2(hg.grad.cpu().numpy(), ref_dh0))


def test_golden_h0_autograd_and_fused_step(golden_dir):
    """small_bi_h0_mlsm (the unmodified reference's autograd, with `hidden`) on the bf16 path: logits, loss, gradients, dx, dh0
    through autograd, then one fused train_step against the reference's step."""
    z = golden_cases.load(golden_dir, "small_bi_h0_mlsm")
    B, T, F, H, L, C, bidir = [int(v) for v in z["meta"]]
    d = dict(B=B, T=T, F=F, H=H, L=L, C=C, bidir=bool(bidir))
    m = make_model(d, params_of(z), PREC)
    m.train()
    x = torch.from_numpy(z["x"]).cuda().requires_grad_(True)
    h0 = torch.from_numpy(z["h0"]).cuda().requires_grad_(True)
    loss_fn, tgt = loss_from(z)
    pred = m(x, h0)
    assert rel(pred.detach().cpu().numpy(), z["logits"]) < TB["logits"]
    loss = loss_fn.cuda()(pred, tgt.cuda())
    loss.backward()
    assert abs(loss.item() - float(z["loss"])) < 10 * TB["logits"] * max(1.0, abs(float(z["loss"])))
    errs = _per_tensor_errors({k: p.grad.cpu().numpy() for k, p in m.named_parameters()},
                              {k: z["g:" + k] for k, _ in m.named_parameters()})
    assert all(v < TB["grads"] for v in errs.values()), errs
    got = np.concatenate([p.grad.cpu().numpy().ravel() for _, p in m.named_parameters()])
    ref = np.concatenate([z["g:" + k].ravel() for k, _ in m.named_parameters()])
    assert rel_l2(got, ref) < TB["gflat"], rel_l2(got, ref)
    assert rel_l2(x.grad.cpu().numpy(), z["dx"]) < TB["grads"]
    assert rel_l2(h0.grad.cpu().numpy(), z["dh0"]) < TB["grads"], rel_l2(h0.grad.cpu().numpy(), z["dh0"])

    m = make_model(d, params_of(z), PREC)
    loss_fn, tgt = loss_from(z)
    m.add_loss_fn(loss_fn)
    m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
    m.train()
    loss, logits = m.train_step(torch.from_numpy(z["x"]).cuda(), tgt.cuda(), torch.from_numpy(z["h0"]).cuda())
    assert abs(float(loss) - float(z["loss"])) < 10 * TB["logits"] * max(1.0, abs(float(z["loss"])))
    assert rel(logits.cpu().numpy(), z["logits"]) < TB["logits"]
    gn = float(torch.sqrt(m._adam["scal"][1]))
    assert abs(gn - float(z["grad_norm"])) < TB["grads"] * float(z["grad_norm"])
    upd_got, upd_ref = [], []
    for k, v in m.state_dict().items():
        if "q:" + k not in z:
            continue
        assert np.abs(v.cpu().numpy() - z["q:" + k]).max() < TB["step"], k
        upd_got.append((v.cpu().numpy() - z["p:" + k]).ravel())
        upd_ref.append((z["q:" + k] - z["p:" + k]).ravel())
    assert rel_l2(np.concatenate(upd_got), np.concatenate(upd_ref)) < TB["update"]


@pytest.mark.parametrize("H, F", [(256, 64), (256, 24), (512, 24)])
def test_zero_initial_state_equals_none(H, F):
    """hidden = zeros takes the initial-state code (W_hh h0 GEMM, step-0 read, the extra backward product, the dW_hh term) and must
    give what hidden = None gives: logits and h_n bit for bit, gradients up to the order of the backward's atomic sums."""
    B, T, L, C = 64, 7, 2, 3
    torch.manual_seed(6)
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=PREC).cuda().train()
    g = torch.Generator().manual_seed(8)
    x = torch.randn(B, T, F, generator=g).cuda()
    dl = torch.randn(B, C, generator=g).cuda()
    outs = []
    for h0 in (None, torch.zeros(2 * L, B, H, device="cuda", requires_grad=True)):
        m.zero_grad()
        xg = x.clone().requires_grad_(True)
        y = m(xg, h0)
        hn = m._last_hidden.clone()
        y.backward(dl)
        grads = torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).cpu().numpy()
        outs.append((y.detach().cpu(), hn.cpu(), grads, xg.grad.cpu().numpy()))
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1])
    assert rel_l2(outs[1][2], outs[0][2]) < 1e-5, rel_l2(outs[1][2], outs[0][2])
    assert rel_l2(outs[1][3], outs[0][3]) < 1e-5


@pytest.mark.parametrize("H", [256, 512])
def test_split_backward_matches_one_call(H):
    """bigru_backward_layers(L-1..1) then (0..0) - the data-parallel split - gives the dh0 and gradient vector of one
    bigru_backward call."""
    pkg = _pkg()
    lib = pkg._lib.load()
    ptr = pkg._lib.ptr
    B, T, F, L, C = 64, 6, 24, 2, 3
    torch.manual_seed(7)
    m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision=PREC).cuda()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, T, F, generator=g).cuda()
    h0 = (torch.randn(2 * L, B, H, generator=g) * 0.5).cuda()
    dl = torch.randn(B, C, generator=g).cuda()
    plan = m._plan_for(x)
    pflat = m.flat_parameters()
    stash = plan.acquire_stash()
    logits = torch.empty(B, C, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    args = (0.0, 0, 0, 0)
    pkg._lib.check(lib.bigru_forward(plan.handle, ptr(pflat), ptr(x), ptr(h0), *args, ptr(stash), ptr(plan.scratch),
                                     ptr(logits), None, s), "bigru_forward")
    g1, dh1 = torch.empty_like(pflat), torch.empty_like(h0)
    pkg._lib.check(lib.bigru_backward(plan.handle, ptr(pflat), ptr(x), ptr(h0), *args, ptr(stash), ptr(plan.scratch), ptr(dl),
                                      ptr(g1), None, ptr(dh1), s), "bigru_backward")
    g2, dh2 = torch.empty_like(pflat), torch.full_like(h0, float("nan"))
    for lo_hi in ((L - 1, 1), (0, 0)):
        pkg._lib.check(lib.bigru_backward_layers(plan.handle, ptr(pflat), ptr(x), ptr(h0), *args, ptr(stash), ptr(plan.scratch),
                                                 ptr(dl), ptr(g2), None, ptr(dh2), lo_hi[0], lo_hi[1], s), "bigru_backward_layers")
    torch.cuda.synchronize()
    plan.release_stash(stash)
    assert bool(torch.isfinite(dh2).all())
    assert rel_l2(dh2.cpu().numpy(), dh1.cpu().numpy()) < 1e-5
    assert rel_l2(g2.cpu().numpy(), g1.cpu().numpy()) < 1e-5
    assert float(dh1.abs().max()) > 0


def test_fused_step_with_hidden_matches_generic_step():
    """Three train_step(x, y, hidden) calls (C-ABI calls only) against autograd + torch.optim.Adam on the same kernels."""
    B, T, F, H, L, C = 32, 8, 16, 128, 2, 4
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, F, generator=g).cuda()
    y = torch.randint(0, C, (B,), generator=g).cuda()
    h0 = (torch.randn(2 * L, B, H, generator=g) * 0.5).cuda()
    outs, p0 = [], None
    for fused in (True, False):
        torch.manual_seed(5)
        m = _pkg().BiGRU(H, F, C, L, 1, 0.0, False, True, precision=PREC).cuda()       # clip=1 so that clipping is active
        p0 = m.flat_parameters().clone()
        m.add_loss_fn(nn.CrossEntropyLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
        m.train()
        for _ in range(3):
            if fused:
                m.train_step(x, y, h0)
            else:
                m.optimizer.zero_grad()
                nn.functional.cross_entropy(m(x, h0), y).backward()
                nn.utils.clip_grad_norm_(m.parameters(), m.clip)
                m.optimizer.step()
        outs.append(m.flat_parameters().clone().cpu().numpy())
    assert np.abs(outs[0] - outs[1]).max() < TB["step"], np.abs(outs[0] - outs[1]).max()
    p0 = p0.cpu().numpy()
    assert rel_l2(outs[0] - p0, outs[1] - p0) < TB["update"]


def test_long_sequence_config_with_hidden():
    """BASELINE configs[4] at full length (T1024, F128, H512, L2, bidirectional), batch 64, with an initial hidden state, on the
    8-CTA-cluster kernels: logits, the flat gradient and dh0 against torch.nn.GRU (OracleBiGRU(x, hidden)) at the bf16
    path's tolerances."""
    B, T, F, H, L, C = 64, 1024, 128, 512, 2, 3
    torch.manual_seed(0)
    ref = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
    g = torch.Generator().manual_seed(99)
    x = torch.randn(B, T, F, generator=g)
    y = torch.randint(0, C, (B,), generator=g)
    h0 = torch.randn(2 * L, B, H, generator=g) * 0.5
    ref.train()
    hr = h0.clone().requires_grad_(True)
    out_ref = ref(x, hr)
    loss_ref = nn.functional.cross_entropy(out_ref, y)
    loss_ref.backward()
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=PREC)
    m.load_state_dict(ref.state_dict())
    m = m.cuda().train()
    hg = h0.cuda().requires_grad_(True)
    out = m(x.cuda(), hg)
    loss = nn.functional.cross_entropy(out, y.cuda())
    loss.backward()
    e_log = rel(out.detach().cpu().numpy(), out_ref.detach().numpy())
    got = torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).cpu().numpy()
    want = torch.cat([p.grad.reshape(-1) for p in ref.parameters()]).numpy()
    e_g = rel_l2(got, want)
    e_h = rel_l2(hg.grad.cpu().numpy(), hr.grad.numpy())
    print(f"configs[4] (B{B}) with hidden, bf16 tensor-core path: logits rel {e_log:.3e}, gradient flat rel-L2 {e_g:.3e}, "
          f"dh0 rel-L2 {e_h:.3e}")
    path = os.environ.get("BIGRU_PARITY_REPORT_C4_H0")
    if path:
        with open(path, "w") as f:
            json.dump({"shape": dict(B=B, T=T, F=F, H=H, L=L, C=C), "precision": PREC, "initial_state": "randn * 0.5",
                       "reference": "oracle/bigru_oracle.OracleBiGRU(x, hidden) (torch.nn.GRU CPU fp32)",
                       "logits_rel": e_log, "grad_flat_rel_l2": e_g, "dh0_rel_l2": e_h,
                       "loss": float(loss.detach()), "loss_reference": float(loss_ref.detach())}, f, indent=1)
    assert e_log < TB["logits"], e_log
    assert e_g < TB["gflat"], e_g
    assert e_h < TB["grads"], e_h
    assert abs(float(loss.detach()) - float(loss_ref.detach())) < 3e-2


def test_single_form_wide_backward_with_hidden(tmp_path):
    """BIGRU_W_BWD=single (the single-tile hidden-512 backward scan; the setting is read once per process) with an initial
    state, against the C oracle."""
    script = tmp_path / "single.py"
    script.write_text(textwrap.dedent('''
        import os, sys
        import numpy as np, torch
        sys.path.insert(0, os.environ["REPO"]); sys.path.insert(0, os.path.join(os.environ["REPO"], "tests"))
        import financial_market_data_analysis_b200 as pkg
        import oracle_c
        from test_gpu_parity import TOL, rel, rel_l2
        tol = TOL["bf16"]
        B, T, F, H, L, C, D = 32, 5, 24, 512, 2, 3, 2
        torch.manual_seed(3)
        m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision="bf16").cuda()
        g = torch.Generator().manual_seed(12)
        x = torch.randn(B, T, F, generator=g); h0 = torch.randn(L * D, B, H, generator=g) * 0.5; dl = torch.randn(B, C, generator=g)
        flat = m.flat_parameters().cpu().numpy()
        ref_logits, ref_hn, stash = oracle_c.forward(flat, x.numpy(), H, L, C, D, h0.numpy(), keep=True)
        ref_g, ref_dx, ref_dh0 = oracle_c.backward(flat, x.numpy(), stash, dl.numpy(), H, L, C, D)
        xg = x.cuda().requires_grad_(True); hg = h0.cuda().requires_grad_(True)
        y = m(xg, hg)
        y.backward(dl.cuda())
        got = torch.cat([p.grad.reshape(-1) for p in m._ordered_params()]).cpu().numpy()
        errs = dict(logits=rel(y.detach().cpu().numpy(), ref_logits), grads=rel_l2(got, ref_g),
                    dx=rel_l2(xg.grad.cpu().numpy(), ref_dx), dh0=rel_l2(hg.grad.cpu().numpy(), ref_dh0))
        print("SINGLE", errs)
        assert errs["logits"] < tol["logits"] and errs["grads"] < tol["gflat"], errs
        assert errs["dx"] < tol["grads"] and errs["dh0"] < tol["grads"], errs
    '''))
    env = dict(os.environ, REPO=ROOT, BIGRU_W_BWD="single")
    out = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "SINGLE" in out.stdout


@pytest.mark.parametrize("H", [256, 512])
def test_forward_with_hidden_is_repeatable(H):
    """Two forwards with the same initial state on identical inputs give byte-identical logits (no atomics in the forward)."""
    B, T, F, L, C = 64, 9, 64, 2, 3
    torch.manual_seed(2)
    m = _pkg().BiGRU(H, F, C, L, 50, 0.0, False, True, precision=PREC).cuda().eval()
    g = torch.Generator().manual_seed(13)
    x = torch.randn(B, T, F, generator=g).cuda()
    h0 = (torch.randn(2 * L, B, H, generator=g) * 0.5).cuda()
    with torch.no_grad():
        a = m(x, h0).clone()
        hn_a = m._last_hidden.clone()
        b = m(x, h0).clone()
        hn_b = m._last_hidden.clone()
    assert torch.equal(a, b)
    assert torch.equal(hn_a, hn_b)
