import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from baler_b200 import synth
from baler_b200.modules import models
nb = 600000
torch.manual_seed(0)
cm = models.Conv_AE(5, 250).eval()
snaps = synth.cfd_snapshots((nb + 99) // 100)
snaps = (snaps - snaps.min()) / (snaps.max() - snaps.min())
blocks = torch.from_numpy(np.ascontiguousarray(snaps.reshape(-1, 1, 5, 5)[:nb])).cuda()
codec = cm.codec(5, 5)
x = blocks.reshape(-1, 25).contiguous()
z = codec.encode(x); y = codec.decode(z)
torch.cuda.synchronize()
for name, fn in (("enc", lambda: codec.encode(x)), ("enc", lambda: codec.encode(x)), ("dec", lambda: codec.decode(z)), ("dec", lambda: codec.decode(z)),
                 ("enc_nocheck", lambda: codec.encode(x, check_range=False)), ("model.enc", lambda: cm.encode(blocks))):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record()
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    print(name, "gpu %.2f ms, host enqueue %.2f ms" % (e0.elapsed_time(e1), (t1 - t0) * 1e3))
