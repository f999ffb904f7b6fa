"""Timeline of the persistent tcgen05 GEMM on conv-like shapes (many tiles, few k-blocks), which make_tc_plan runs on the
persistent kernel at bn = 32.  Prints, for CTA 0's first 12 tiles, nanoseconds (relative to the first stamp) of: TMA
issued, operands landed, accumulator committed, epilogue start, epilogue end; then the average time of the GEMM planned
at each tile width."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from rlrep_b200 import _lib  # noqa: E402

lib = _lib.load()
dev = "cuda"
for (M, N, K) in [(430336, 288, 32), (430336, 32, 288)]:
    A = torch.randn(M, K, device=dev)
    B = torch.randn(N, K, device=dev)
    Cm = torch.empty(M, N, device=dev)
    dbg = torch.zeros(80, dtype=torch.int64, device=dev)
    _lib.check(lib.rlrep_gemm_set_debug_buffer(dbg.data_ptr()))
    _lib.gemm(A, B, Cm, bn=32, split_k=1)
    torch.cuda.synchronize()
    _lib.check(lib.rlrep_gemm_set_debug_buffer(None))
    t = dbg.cpu().reshape(5, 16)
    t0 = int(t[t > 0].min()) if (t > 0).any() else 0
    print(f"M={M} N={N} K={K}")
    for i in range(12):
        print("  tile %2d: " % i + "  ".join(f"{(int(t[r, i]) - t0) if t[r, i] > 0 else -1:7d}" for r in range(5)))
    for bn in (32, 64, 128, 256):
        ms, bno, so = _lib.gemm_bench(A, B, Cm, bn=bn, split_k=1, iters=20)
        print(f"  bn={bno} split={so}: {ms * 1e3:.1f} us")
