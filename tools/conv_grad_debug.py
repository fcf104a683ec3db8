import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import test_gpu_cfd as T
from baler_b200 import engine
g = np.load(os.path.join(ROOT, "tests", "golden", "conv_train.npz"))
m = T._conv_model()
tr, sp = T._conv_trainer(m)
x = torch.from_numpy(g["blocks"]).cuda()
tr.step(x[:300].contiguous(), engine.make_hyper(lr=1e-3), phase=1)
grads = tr.grads_view().cpu().numpy().astype(np.float64)
named = T._named_flat(m, sp, grads[:-1])
scale = max(float(np.abs(np.asarray(v)).max()) for v in named.values())
for k, a in named.items():
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    if k in T.CONV_BIG:
        ref = g["g0/%s#sample" % k]; a = a[::101]
    else:
        ref = g["g0/%s" % k].reshape(-1)
    print("%-28s n=%6d max|ref| %.3e  max|err| %.3e %s" % (k, a.size, np.abs(ref).max(), np.abs(a - ref).max(), "DEAD" if k in T.CONV_DEAD else ""))
