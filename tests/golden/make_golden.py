"""Generates tests/golden/*.npz by EXECUTING THE REAL REFERENCE in the authoring container.

    python tests/golden/make_golden.py          (needs /root/reference; not run on the GPU box)

* buyer_tower_*.npz : inputs, parameters and outputs of the unmodified
  /root/reference/src/models/buyer_tower.py::BuyerTower (torch CPU, fp32) on seeded inputs, plus the
  same module in fp64 for the noise floor.
* infonce_*.npz     : inputs, loss and autograd gradients of the unmodified /root/reference/src/training/losses.py
  ::InfoNCELoss (torch CPU, fp32, plus the loss in fp64).
* vector_db_*.npz   : outputs of the unmodified /root/reference/src/inference/vector_db.py
  ::VectorDatabase.  Its `import faiss` is satisfied by oracle/faiss_shim (faiss-cpu is not
  installable here), so these pin the WRAPPER logic (normalisation, k clamp, id mapping, row-0-only
  quirk) — not faiss itself, whose boundary stays unpinned (see oracle/flat_ip_oracle.py).
"""
import io
import contextlib
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
OUT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "oracle" / "faiss_shim"))
sys.path.insert(0, "/root/reference")

from src.models.buyer_tower import BuyerTower  # noqa: E402  (the reference)
from src.inference.vector_db import VectorDatabase  # noqa: E402  (the reference, over the shim)
from src.training.losses import InfoNCELoss  # noqa: E402  (the reference)
from conftest import infonce_inputs  # noqa: E402

EVENT_W = np.array([1.0, 5.0, 10.0], dtype=np.float32)


def event_weights(rng, shape):
    return EVENT_W[rng.choice(3, size=shape, p=[0.75, 0.18, 0.07])]


def buyer_case(name, B, S, D, H, seed, scale=1.0, special=None):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, S, D)).astype(np.float32)
    w = event_weights(rng, (B, S))
    if special == "ragged":           # zero-padded tails with zero weights (trainer.py:144-151)
        for b in range(B):
            L = 1 + (b * 7) % S
            x[b, L:] = 0
            w[b, L:] = 0
    if special == "zero_weight_row":  # all-zero weights -> exactly-zero output in weighted_avg
        w[0] = 0
    if special == "nonzero_row_zero_weight":   # attention does NOT mask: such rows still contribute
        w[:, ::2] = 0
    if special == "unit_rows":        # serving: history rows are L2-normalised catalog rows
        x /= np.linalg.norm(x, axis=2, keepdims=True)
    out = {"x": x, "w": w}
    xt, wt = torch.from_numpy(x), torch.from_numpy(w)
    m = BuyerTower(D, "weighted_avg").eval()
    with torch.no_grad():
        out["weighted_avg"] = m(xt, wt).numpy()
        out["weighted_avg_f64"] = m.double()(xt.double(), wt.double()).numpy()
    torch.manual_seed(seed)
    m = BuyerTower(D, "attention", H).eval()
    with torch.no_grad():
        for p in m.parameters():
            p.mul_(scale)
        sd = {k: v.numpy().copy() for k, v in m.state_dict().items()}
        out["attention"] = m(xt, wt).numpy()
        out["attention_seq0"] = m.encode_from_sequence(xt[0], wt[0]).numpy()
        out["attention_f64"] = m.double()(xt.double(), wt.double()).numpy()
    out.update({"W1": sd["attention.0.weight"], "b1": sd["attention.0.bias"],
                "W2": sd["attention.2.weight"], "b2": sd["attention.2.bias"]})
    np.savez_compressed(OUT / f"buyer_tower_{name}.npz", **out)
    print(name, {k: v.shape for k, v in out.items() if k in ("x", "weighted_avg", "attention")})


def vdb_case(name, N, D, nq, k, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((N, D)) * rng.uniform(0.1, 3.0, (N, 1))).astype(np.float32)   # un-normalised rows
    q = rng.standard_normal((nq, D)).astype(np.float32)
    pids = [f"p{i:05d}" for i in range(N)]
    db = VectorDatabase(embedding_dim=D)
    with contextlib.redirect_stdout(io.StringIO()):
        db.build_index(x, pids)
    batch = db.retrieve_batch(q, k)
    single = db.retrieve(q[0], k)
    multi_as_single = db.retrieve(q[:3], k)      # reference quirk: only query 0 is returned (vector_db.py:164)
    kk = len(batch[0])
    out = {
        "x": x, "q": q, "k": np.int64(k),
        "batch_ids": np.array([[int(p[1:]) for p, _ in row] for row in batch], dtype=np.int64).reshape(nq, kk),
        "batch_scores": np.array([[s for _, s in row] for row in batch], dtype=np.float32).reshape(nq, kk),
        "single_ids": np.array([int(p[1:]) for p, _ in single], dtype=np.int64),
        "single_scores": np.array([s for _, s in single], dtype=np.float32),
        "multi_as_single_ids": np.array([int(p[1:]) for p, _ in multi_as_single], dtype=np.int64),
    }
    np.savez_compressed(OUT / f"vector_db_{name}.npz", **out)
    print(name, out["batch_ids"].shape)


def infonce_case(name, B, M, D, seed, temperature=0.07, unit=True, store_buyer_pos=True):
    """The real InfoNCELoss (losses.py:8-79) and its autograd gradients on seeded inputs.  store_buyer_pos=False
    stores the seed in place of buyer and pos (tests/conftest.py:golden regenerates them) for a case that would
    otherwise exceed 1 MB."""
    b, p, n = infonce_inputs(B, M, D, seed, unit)
    crit = InfoNCELoss(temperature)
    tb, tp, tn = (torch.from_numpy(a).requires_grad_(True) for a in (b, p, n))
    loss = crit(tb, tp, tn)
    loss.backward()
    with torch.no_grad():
        loss64 = crit(tb.double(), tp.double(), tn.double())
    inputs = dict(buyer=b, pos=p) if store_buyer_pos else dict(input_seed=np.int64(seed), input_unit=np.bool_(unit))
    np.savez_compressed(OUT / f"infonce_{name}.npz", **inputs, neg=n, temperature=np.float64(temperature),
                        loss=np.float32(loss.item()), loss_f64=np.float64(loss64.item()), d_buyer=tb.grad.numpy(),
                        d_pos=tp.grad.numpy(), d_neg=tn.grad.numpy())
    print(f"infonce_{name}: loss {loss.item():.6f}")


if __name__ == "__main__":
    infonce_case("b16_m4_d384", 16, 4, 384, 21)                 # trainer defaults: 4 sampled negatives (losses.py:36-79)
    infonce_case("b64_m4_d384", 64, 4, 384, 22, store_buyer_pos=False)
    infonce_case("b5_m0_d384", 5, 0, 384, 23)                   # no sampled negatives: in-batch only
    infonce_case("b9_m3_d100_raw", 9, 3, 100, 24, temperature=0.5, unit=False)   # unnormalised, D % 32 != 0
    infonce_case("b1_m2_d64", 1, 2, 64, 25)                     # batch of one: the in-batch block is all masked
    buyer_case("ref_test_shape", 2, 5, 384, 128, 1)             # tests/test_buyer_tower.py shapes
    buyer_case("b8_s50_d384", 8, 50, 384, 128, 2)               # C2 shape per buyer
    buyer_case("ragged", 6, 33, 384, 128, 3, special="ragged")
    buyer_case("zero_weight_row", 3, 9, 384, 128, 4, special="zero_weight_row")
    buyer_case("nomask", 4, 12, 384, 128, 5, special="nonzero_row_zero_weight")
    buyer_case("scaled20", 4, 20, 384, 128, 6, scale=20.0)     # stresses the softmax range
    buyer_case("unit_rows_s100", 2, 100, 384, 128, 7, special="unit_rows")
    buyer_case("d100_h24", 5, 11, 100, 24, 8)                   # D % 128 != 0, small H
    buyer_case("d30_odd", 3, 4, 30, 7, 9)                       # D % 4 != 0 -> generic kernels
    buyer_case("s1", 4, 1, 384, 128, 10)
    vdb_case("n500_d32_k10", 500, 32, 5, 10, 11)
    vdb_case("n7_k10_clamp", 7, 16, 4, 10, 12)                  # k > ntotal -> k clamps (vector_db.py:159)
    vdb_case("n2000_d96_k100", 2000, 96, 3, 100, 13)
