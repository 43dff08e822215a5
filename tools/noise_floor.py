import os, torch, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gdr_net_b200 import synth
from oracle import fixtures, gdrn_oracle as O
torch.set_num_threads(8)
sd = fixtures.calibrated_state_dict(0)
batch = synth.make_batch(4, seed=1)
res = {}
for dt in (torch.float32, torch.float64):
    leaf = O.leaf_state_dict(sd, dtype=dt)
    b = {k: (v.to(dt) if isinstance(v, torch.Tensor) and v.dtype.is_floating_point else v) for k, v in batch.items()}
    o = O.gdrn_forward(leaf, b, train=True, do_loss=True)
    sum(o["losses"].values()).backward()
    res[dt] = (o, leaf)
o32, l32 = res[torch.float32]; o64, l64 = res[torch.float64]
def rel(a,b): return float((a.double()-b.double()).norm()/b.double().norm())
print("head", rel(o32["head"], o64["head"]), "rot", rel(o32["rot"], o64["rot"]), "trans", rel(o32["trans"], o64["trans"]))
for k in o32["losses"]: print(k, float(o32["losses"][k]), float(o64["losses"][k]))
names = [k for k in l32 if l32[k].requires_grad]
for k in names[::-1][:12] + names[:6]:
    print(f"{k:44s} {rel(l32[k].grad, l64[k].grad):.2e}")
