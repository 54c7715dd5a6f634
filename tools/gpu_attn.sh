#!/bin/bash
mkdir -p gpurun_out
python -c "import __graft_entry__ as g; g.build()" > gpurun_out/build.log 2>&1
python - <<'PY'
import sys, torch
sys.path.insert(0, ".")
import two_tower_model_v2_b200 as pkg
from two_tower_model_v2_b200 import ops
torch.manual_seed(0)
for (R, D, H) in [(1000, 384, 128), (4096 * 50, 384, 128), (777, 100, 24), (300, 64, 256)]:
    x = torch.randn(R, D, device="cuda"); x = x / x.norm(dim=1, keepdim=True)
    l1 = torch.nn.Linear(D, H).cuda(); l2 = torch.nn.Linear(H, 1).cuda()
    W1, b1, W2, b2 = l1.weight.detach(), l1.bias.detach(), l2.weight.detach().reshape(-1).contiguous(), l2.bias.detach()
    got = ops.attention_logits(x, W1, b1, W2, b2)
    torch.cuda.synchronize()
    ref64 = (torch.relu(x.double() @ W1.double().t() + b1.double()) @ W2.double() + b2.double())
    ref32 = (torch.relu(x @ W1.t() + b1) @ W2 + b2)
    print(f"R={R} D={D} H={H}: |tc-fp64| max {float((got.double()-ref64).abs().max()):.3e}  |torch32-fp64| max {float((ref32.double()-ref64).abs().max()):.3e}  |logit| max {float(ref64.abs().max()):.3f}", flush=True)
PY
timeout 600 python -m pytest tests/test_gpu_pool.py -q -x 2>&1 | tail -4
timeout 300 python tools/pool_only.py 2>&1 | tail -1 | cut -c1-600
