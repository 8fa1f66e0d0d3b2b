"""Where the 512-pair (literal cfg2) call spends its time: Python layers vs the C call vs GPU."""
import ctypes, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "pydrobert-pytorch_b200")):
    sys.path.insert(0, p)
import numpy as np, torch
import b200lev.functional as F
from b200lev import _abi, _ops
from bench import make_batch, NBEST
dev = torch.device("cuda", 0)
ref_np, hyp_np, cells = make_batch(64, seed=7)
ref = torch.from_numpy(np.repeat(ref_np, NBEST, axis=1)).to(dev)
hyp = torch.from_numpy(hyp_np).to(dev)
def wall(fn, n=2000):
    for _ in range(50): fn()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(n): fn()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e6
print("functional.prefix_error_rates        %.1f us" % wall(lambda: F.prefix_error_rates(ref, hyp, eos=0, warn=False)))
args = (ref, hyp, 0, True, False, 1.0, 1.0, 1.0, True, True, False, -100, True, 1)
print("_ops.string_matching_impl            %.1f us" % wall(lambda: _ops.string_matching_impl(*args)))
L = _abi.lib()
rt, ht = _ops._tok_struct(ref, False), _ops._tok_struct(hyp, False)
o = _ops._opts(0, True, 1.0, 1.0, 1.0, True, False, -100, True, 1)
nbytes = L.b200lev_workspace_bytes(ctypes.byref(rt), ctypes.byref(ht), 2, 0)
ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
out = torch.empty((hyp.shape[0] + 1, hyp.shape[1]), dtype=torch.float32, device=dev)
flags = torch.zeros(1, dtype=torch.int32, device=dev)
st = torch.cuda.current_stream().cuda_stream
def raw():
    L.b200lev_prefix(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o), out.data_ptr(), out.shape[1], 1,
                     ws.data_ptr(), nbytes, flags.data_ptr(), st)
print("raw b200lev_prefix (preallocated)    %.1f us" % wall(raw))
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
g = torch.cuda.CUDAGraph()
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    st2 = s.cuda_stream
    def raw2():
        L.b200lev_prefix(ctypes.byref(rt), ctypes.byref(ht), ctypes.byref(o), out.data_ptr(), out.shape[1], 1,
                         ws.data_ptr(), nbytes, flags.data_ptr(), st2)
    raw2(); torch.cuda.synchronize()
    with torch.cuda.graph(g, stream=s):
        raw2()
print("CUDA graph replay of the same call   %.1f us" % wall(lambda: g.replay()))
