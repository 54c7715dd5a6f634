"""Attention pooling at C2: the fused kernel vs its logits-only mode (MMA side alone) vs plain weighted pooling."""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import two_tower_model_v2_b200 as pkg  # noqa: E402
from two_tower_model_v2_b200 import ops  # noqa: E402


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def main():
    import os
    B, S, D = int(os.environ.get('TT_DIAG_B', 4096)), 50, 384
    g = torch.Generator(device="cuda").manual_seed(99)
    x = torch.randn((B, S, D), device="cuda", generator=g)
    w = torch.tensor([1.0, 5.0, 10.0], device="cuda")[torch.randint(0, 3, (B, S), device="cuda", generator=g)]
    torch.manual_seed(0)
    m = pkg.BuyerTower(D, "attention").cuda()
    W1, b1, W2, b2 = m._mlp_params(x.device)
    import os
    if os.environ.get("TT_DIAG_LOGITS_ONLY"):
        with torch.no_grad():
            print(json.dumps({"logits_only_us": timeit(lambda: ops.attention_logits(x.view(B * S, D), W1, b1, W2, b2))}))
        return
    with torch.no_grad():
        out = {"fused_us": timeit(lambda: m(x, w)),
               "logits_only_us": timeit(lambda: ops.attention_logits(x.view(B * S, D), W1, b1, W2, b2)),
               "weighted_pool_us": timeit(lambda: ops.pool_weighted(x, w))}
        lg = ops.attention_logits(x.view(B * S, D), W1, b1, W2, b2).view(B, S)
        out["pool_attention_given_logits_us"] = timeit(lambda: ops.pool_attention(x, lg, w))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
