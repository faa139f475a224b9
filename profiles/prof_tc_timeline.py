import ctypes as C, os, sys, numpy as np, torch
NB = int(os.environ.get("NB", "4096"))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.gpu_helpers import make_pair, synth_xy, dev
from lcn_pose_b200 import _lib as L
eng,cfg,p = make_pair(L=3, knn=3, path='bf16')
x,_ = synth_xy(NB)
xd = dev(x)
for _ in range(3): eng.forward(xd, bn_group=NB, training=True)
torch.cuda.synchronize()
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
flush = torch.empty(256<<20, dtype=torch.uint8, device='cuda')
for cold in (0,1):
    if cold: flush.zero_()
    torch.cuda.synchronize()
    L.check(eng.lib.lcn_layer_gemm(eng.h, eng.params.data_ptr(), eng.ws.data_ptr(), eng.ws.numel(), NB, NB, 2, 0, st))
    torch.cuda.synchronize()
    buf = (C.c_ulonglong*512)()
    eng.lib.lcn_debug_read_prof.argtypes=[C.c_void_p]
    assert eng.lib.lcn_debug_read_prof(buf)==0
    t = np.array(buf[:], dtype=np.int64)
    t0 = t[0]
    print('cold' if cold else 'warm', 'setup', t[1]-t0, 'first_chunk_done', t[2]-t0, 'last_chunk_staged', t[3]-t0, 'stores_read', t[4]-t0, 'epi_end', t[5]-t0, 'end', t[6]-t0)
    for it in range(34):
        b = 16+4*it
        if t[b]==0: break
        print(' it', it, 'empty_ok', t[b]-t0, 'issued', t[b+1]-t0, 'full_ok', t[b+2]-t0, 'mma_issued', t[b+3]-t0)
    for e in range(6):
        b = 200 + 8 * e
        if t[b] == 0: continue
        print(' chunk', e, 'done_ok', t[b]-t0, 'tmem_ld', t[b+1]-t0, 'staged', t[b+2]-t0, 'bar_B', t[b+3]-t0, 'stats', t[b+4]-t0, 'bar_C', t[b+5]-t0, 'part_out', t[b+6]-t0)
# kernel duration by CUDA events: back to back (warm L2) and with an L2 flush before every launch
def timed(flush_each, reps=20):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        if flush_each: flush.zero_()
        a.record()
        L.check(eng.lib.lcn_layer_gemm(eng.h, eng.params.data_ptr(), eng.ws.data_ptr(), eng.ws.numel(), NB, NB, 2, 0, st))
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    return ts[0], ts[len(ts) // 2]
print("events us (min, median): warm", timed(False), "flushed", timed(True))
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(50):
    L.check(eng.lib.lcn_layer_gemm(eng.h, eng.params.data_ptr(), eng.ws.data_ptr(), eng.ws.numel(), NB, NB, 2, 0, st))
b.record(); torch.cuda.synchronize()
print("50 back-to-back launches: us per launch", a.elapsed_time(b) * 1e3 / 50)
