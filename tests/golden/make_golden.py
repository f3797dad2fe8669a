"""Generates tests/golden/*.npz by running the UNMODIFIED reference (a checkout of the original project).

  python tests/golden/make_golden.py REFERENCE_DIR

The fixtures are committed, so the tests never need the reference.  Nothing here is imported by the product.

  kat.npz          shipped model_params.pt (H=8,F=108,C=4,L=1) + two fixed inputs -> logits
  model_<case>.npz seed-fixed synthetic cases through reference BiGRU: inputs, state_dict,
                   logits, loss, every gradient, (dx, dh0), params after clip+Adam
                   (model_c0 in the compact form that tests/golden_cases.py reads)
  loader.npz       reference MySQLChunkLoader / MySQLBatchLoader / TrainValTestSplit driven by
                   tests/fake_db.FakeCursor: chunk ranges, norm params, delivered batches
"""
import os
import pickle
import sys
import warnings

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, REF)
import fake_db  # noqa: E402
import golden_cases  # noqa: E402

fake_db.install_reference_stubs(bid_levels=2, ask_levels=2)
from biGRU_model import BiGRU  # noqa: E402  (reference, unmodified)
import sql_pytorch_dataloader as ref_loader  # noqa: E402  (reference, unmodified)

torch.set_num_threads(4)


def sd_np(sd, prefix):
    return {prefix + k: v.detach().cpu().numpy().copy() for k, v in sd.items()}


def gen_kat():
    sd = torch.load(os.path.join(REF, "model_params.pt"), map_location="cpu")
    m = BiGRU(8, 108, 4, 1, 50, 0.2, False, True)
    m.load_state_dict(sd)
    m.eval()
    x1 = torch.full((1, 5, 108), 0.5)
    x2 = (torch.arange(540).view(1, 5, 108) % 17).float() / 17
    g = torch.Generator().manual_seed(5)
    x3 = torch.rand(6, 5, 108, generator=g)
    with torch.no_grad():
        out = {"x1": x1.numpy(), "y1": m(x1).numpy(), "x2": x2.numpy(), "y2": m(x2).numpy(),
               "x3": x3.numpy(), "y3": m(x3).numpy()}
    out.update(sd_np(sd, "p:"))
    with open(os.path.join(REF, "norm_params"), "rb") as f:
        npar = pickle.load(f)
    out["norm_min"] = np.array([float(v["MIN"]) for v in npar.values()], np.float32)
    out["norm_max"] = np.array([float(v["MAX"]) for v in npar.values()], np.float32)
    np.savez_compressed(os.path.join(HERE, "kat.npz"), **out)
    print("kat", out["y1"], out["y2"])


def compact(out, seed):
    """Keeps model_c0 under 1 MB (its float32 arrays do not compress): the inputs are left out - tests/golden_cases.py
    rebuilds them from the two seeds and checks them against inputs_sha256 - and the parameters after the step are stored
    as their difference from the initial ones (an exact round trip, asserted here)."""
    names = [k[2:] for k in out if k.startswith("p:")]
    out["input_seeds"] = np.array([0, seed], np.int64)
    out["inputs_sha256"] = np.array(golden_cases.inputs_sha256(out["x"], [out["p:" + k] for k in names]))
    for k in names:
        p, q = out.pop("p:" + k), out.pop("q:" + k)
        dq = (q.astype(np.float64) - p).astype(np.float32)
        assert np.array_equal(p + dq, q), k
        out["dq:" + k] = dq
    del out["x"]


def gen_model(name, B, T, F, H, L, C, bidir, loss, with_h0=False, seed=1234, rebuilt_inputs=False):
    torch.manual_seed(0)
    m = BiGRU(H, F, C, L, 50, 0.0, False, bidir)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, F, generator=g)
    D = 2 if bidir else 1
    out = {}
    if loss == "ce":
        target = torch.randint(0, C, (B,), generator=g)
        loss_fn = nn.CrossEntropyLoss()
    else:
        target = (torch.rand(B, C, generator=g) < 0.25).float()
        if loss == "bce":
            w = torch.rand(C, generator=g) + 0.5
            pw = torch.rand(C, generator=g) * 3 + 0.5
            loss_fn = nn.BCEWithLogitsLoss(weight=w, pos_weight=pw)
            out["loss_weight"], out["loss_pos_weight"] = w.numpy(), pw.numpy()
        else:
            loss_fn = nn.MultiLabelSoftMarginLoss()
    h0 = None
    if with_h0:
        h0 = (torch.randn(L * D, B, H, generator=g) * 0.5).requires_grad_(True)
        out["h0"] = h0.detach().numpy()
    x.requires_grad_(True)
    m.train()                      # dropout p=0: identical to eval, exercises the training path
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    out.update(sd_np(m.state_dict(), "p:"))
    opt.zero_grad()
    pred = m.forward(x, h0)
    lv = loss_fn(pred, target)
    lv.backward()
    out.update({"x": x.detach().numpy(), "target": target.numpy(), "logits": pred.detach().numpy(),
                "loss": np.array(lv.item(), np.float64), "dx": x.grad.numpy()})
    if with_h0:
        out["dh0"] = h0.grad.numpy()
    for k, p in m.named_parameters():
        out["g:" + k] = p.grad.detach().numpy().copy()
    norm = nn.utils.clip_grad_norm_(m.parameters(), m.clip)
    out["grad_norm"] = np.array(float(norm), np.float64)
    opt.step()
    out.update(sd_np(m.state_dict(), "q:"))          # params after one clip+Adam step
    out["meta"] = np.array([B, T, F, H, L, C, int(bidir)], np.int64)
    out["loss_kind"] = np.array(loss)
    if rebuilt_inputs:
        compact(out, seed)
    np.savez_compressed(os.path.join(HERE, f"model_{name}.npz"), **out)
    print(name, "loss", lv.item(), "norm", float(norm))


def gen_loader():
    warnings.simplefilter("ignore")
    cols, targets, fields, query = fake_db.make_table(n_rows=250)
    cur = fake_db.FakeCursor(cols, targets)
    cwd = os.getcwd()
    os.chdir("/tmp")               # the reference pickles ./norm_params as a side effect
    try:
        cl = ref_loader.MySQLChunkLoader(cur, "stock_data_joined", query, chunk_size=100, window=30)
    finally:
        os.chdir(cwd)
    out = {"n_chunks": np.array(len(cl))}
    for i in range(len(cl)):
        idx, (mn, mx) = cl[i]
        out[f"chunk{i}_ids"] = np.array(idx, np.int64)
        out[f"chunk{i}_min"] = mn.numpy()
        out[f"chunk{i}_max"] = mx.numpy()
    split = ref_loader.TrainValTestSplit(cl, 0.1, 0.1)
    tr, va, te = split.get_sets()
    out["split_train"] = np.array([len(i) for i, _ in tr], np.int64)
    out["split_val"] = np.array([len(i) for i, _ in va], np.int64)
    out["split_test"] = np.array([len(i) for i, _ in te], np.int64)
    for bs in (2, 8):
        idx, norm = cl[1]
        ds = ref_loader.MySQLBatchLoader(idx, norm, cur, "stock_data_joined", query, "t0, t1, t2, t3", 30)
        dl = torch.utils.data.DataLoader(ds, batch_size=bs)
        xs, ys = [], []
        for xb, yb in dl:
            xs.append(xb.numpy())
            ys.append(yb.numpy())
        out[f"bs{bs}_x"] = np.concatenate(xs)
        out[f"bs{bs}_y"] = np.concatenate(ys)
        out[f"bs{bs}_nbatches"] = np.array(len(xs))
        out[f"bs{bs}_xnorm"] = ds.x.numpy()
    out["fields"] = np.array(fields)
    np.savez_compressed(os.path.join(HERE, "loader.npz"), **out)
    print("loader chunks", len(cl), "bs2 windows", out["bs2_x"].shape, "bs8", out["bs8_x"].shape)


if __name__ == "__main__":
    gen_kat()
    gen_model("c0", 32, 64, 32, 128, 1, 3, True, "ce", rebuilt_inputs=True)    # BASELINE config 0
    gen_model("small_l2", 4, 7, 5, 8, 2, 3, True, "ce")
    gen_model("small_uni_bce", 3, 6, 4, 8, 2, 4, False, "bce", with_h0=True)
    gen_model("small_bi_h0_mlsm", 5, 9, 12, 16, 2, 4, True, "mlsm", with_h0=True)
    gen_model("ragged", 3, 1, 7, 24, 1, 3, True, "ce")                 # T=1 edge, odd sizes
    gen_loader()
