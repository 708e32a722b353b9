import os, sys, ctypes as C, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch, epp_b200 as epp
from epp_b200 import capi
from tools import workload_setup as helpers, tracegen as tg
tg.build()
R = int(sys.argv[1])
w = tg.baseline_configs()["config3"].scaled(R=max(R, 64), name="config3")
trace = tg.Trace(w)
lib = capi.load()
buf = epp.PinnedBuffer(w.R * w.prompt_bytes)
tokens = buf.array.view(np.uint32).reshape(w.R, w.T)
trace.requests(0, w.R, out=tokens)
out = epp.PinnedBuffer(32 * w.R)
with helpers.make_engine(w) as eng:
    helpers.setup_engine(eng, w, trace)
    b = capi.Batch(); b.n_requests = R; b.uniform_len = w.prompt_bytes; b.data = buf.array.ctypes.data
    for it in range(6):
        assert lib.epp_schedule(eng._h, C.byref(b), out.array.ctypes.data_as(C.c_void_p), None, 0) == 0
    torch.cuda.synchronize()
