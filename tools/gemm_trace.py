"""Per-phase timeline of the tcgen05 GEMM (debug hook avsep_test_gemm_trace): mean/max ns per phase over CTAs."""
import ctypes as C, math, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "av-separation-transformer_b200"))
from avsep_b200.engine import Engine, EngineConfig

eng = Engine(EngineConfig(65, 64, 4, 1, 1, 2, "bf16"), 0)
for (M, N, K, ln, act, tag) in [(16128, 256, 768, 1, 0, "K=768 LN (conv1d_2-sized, plain rows)"), (16128, 256, 768, 0, 0, "K=768 std"), (16128, 768, 256, 0, 0, "qkv"), (12800, 768, 256, 0, 0, "qkv visual"), (16128, 256, 256, 0, 0, "cross_q"), (16128, 1024, 256, 0, 1, "ffn1 relu"), (16128, 1024, 256, 0, 2, "ffn1 gelu"), (16128, 256, 1024, 1, 0, "ffn2 LN"), (16128, 256, 256, 1, 0, "LN full"), (16128, 256, 256, 2, 0, "LN no-resid-load"),
                                (16128, 256, 256, 3, 0, "LN no-x'-store"), (16128, 256, 256, 4, 0, "LN no-bf16-store"),
                                (16128, 256, 256, 5, 0, "LN no resid, no x' store"), (16128, 256, 256, 6, 0, "LN cast only (no stats)")]:
    A = torch.randn(M, K, device="cuda").bfloat16()
    W = (torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device="cuda")
    x = torch.randn(M, N, device="cuda")
    g = torch.randn(N, device="cuda"); b = torch.randn(N, device="cuda")
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    trace = torch.zeros(148 * 64, device="cuda", dtype=torch.int64)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for it in range(3):
        trace.zero_()
        torch.cuda.synchronize()
        rc = eng.lib.avsep_test_gemm_trace(eng.h, A.data_ptr(), W.data_ptr(), bias.data_ptr(), x.data_ptr(), g.data_ptr(),
                                           b.data_ptr(), out.data_ptr(), M, N, K, ln, act, trace.data_ptr(), s)
        assert rc == 0, eng.lib.avsep_last_error(eng.h)
        torch.cuda.synchronize()
    t = trace.cpu().numpy().reshape(148, 64).astype(np.int64)
    t = t[t[:, 0] > 0]
    t0 = t[:, 0].min()
    print(f"== {tag}: M={M} N={N} K={K} ctas={len(t)}; all times us since first CTA entry")
    print(f"   setup done mean {(t[:,1]-t0).mean()/1e3:.2f}; CTA done mean {(t[:,7]-t0).mean()/1e3:.2f} max {(t[:,7]-t0).max()/1e3:.2f}")
    if (t[:, 2] > 0).any():
        r = (t[:, 2:7] - t0) / 1e3
        print("   tile-1 epilogue of warp 2: entered %.2f  bias-barrier %.2f  first-chunk-in-regs %.2f  values-done %.2f  stores-issued %.2f"
              % tuple(r.mean(axis=0)))
    for lt in range(6):
        cols = t[:, 8 + 4 * lt: 12 + 4 * lt]
        ok = cols[:, 3] > 0
        if not ok.any():
            break
        r = (cols[ok] - t0) / 1e3
        print(f"   tile {lt} (n={ok.sum():3d}): operands {r[:,0].mean():6.2f}  mma_issued {r[:,1].mean():6.2f}  acc_ready {r[:,2].mean():6.2f}  epi_done {r[:,3].mean():6.2f} (max {r[:,3].max():6.2f})")
