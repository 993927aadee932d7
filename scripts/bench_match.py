"""Micro-benchmark of the match kernel alone: bench_match.py [pairs] [keypoints] [EVZ_OPT_MATCH_VARIANT values, default 0,5] [descriptor bytes: 128 | 32]."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evenvizion_b200 as evz
from evenvizion_b200 import synth
P = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
N = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
variants = [int(v) for v in sys.argv[3].split(",")] if len(sys.argv) > 3 else [0, 5]
eng = evz.GeometryEngine(0)
D = int(sys.argv[4]) if len(sys.argv) > 4 else 128
ch = synth.make_chain(P + 1, N, d=D, seed=0, device="cuda")
st = eng.ingest(ch["desc"], ch["coords"])
pq = torch.arange(1, P + 1, dtype=torch.int32, device="cuda"); pt = torch.arange(0, P, dtype=torch.int32, device="cuda")
out_off = st.row_off[:-1][pq.long()].contiguous()
idx = torch.empty((st.rows, 2), dtype=torch.int32, device="cuda"); d2 = torch.empty_like(idx)
import ctypes as C
p = lambda t: C.c_void_p(t.data_ptr())
for v in variants:
    eng.set_option(2, v)
    call = lambda: eng._check(eng.lib.evz_match_top2_d(eng.h, p(st.desc), D, p(st.ckey), st.rows, p(st.row_off), p(st.n_kp), p(pq), p(pt), p(out_off), P, p(idx), p(d2), eng._stream()))
    for _ in range(3): call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(5): call()
    e1.record(); e1.synchronize()
    ms = e0.elapsed_time(e1) / 5
    line = f"variant {v}: {ms:.3f} ms  {2.0*N*N*D*P/ms/1e9:.1f} TOP/s (whole call)"
    if v == 0:            # V-space kernel: duration of the main kernel alone (EVZ_OPT_TIME_MATCH)
        eng.set_option(4, 1)
        for _ in range(5): call()
        torch.cuda.synchronize()
        km = sum(eng.match_kernel_ms(k) for k in range(5)) / 5
        eng.set_option(4, 0)
        line += f"; kernel {km:.3f} ms  {2.0*N*N*D*P/km/1e9:.1f} TOP/s"
    print(line, flush=True)
