import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowcompare_b200 import configs, engine, spec
torch.set_grad_enabled(False)
cfg = configs.get_config("dgcnn_attn", n_flow_layers=12)
fsd, esd = spec.random_state_dicts(cfg, seed=0)
e = engine.FlowCompareB200((fsd, esd), cfg, device="cuda:0", precision=os.environ.get("FC_PRECISION", "fp16x3"))
b = spec.synthetic_batch(cfg, 16, seed=3)
args = (b["extract_0"].cuda(), b["extract_1"].cuda(), None); eps = b["eps"].cuda()
ref = e.inner_loop(args, eps=eps)[1].clone()
nd = 0
for i in range(10):
    out = e.inner_loop(args, eps=eps)[1]
    d = (out - ref).abs().max().item()
    nd += int(d != 0)
print("runs differing from the first:", nd, "of 10")
