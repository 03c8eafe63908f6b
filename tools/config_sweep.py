"""Throughput of the other BASELINE.json configs (parity for these is covered by tests/golden):
C1 demo default (B=8), C3 long-form (10 s @ 16 kHz: T=1251, N=500), C4 scaled model (d=512, 6+6 layers, S=3) and the
per-GPU batch sweep B=1..1024 of the default model.  Device-resident inputs, CUDA-graph replay, CUDA events.
    python tools/config_sweep.py [--precision bf16|tf32] > profiles/...json
"""
import argparse, json, os, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "av-separation-transformer_b200"))
from avsep_b200 import AVSeparationTransformer
from avsep_b200.synth import synthetic_batch

ap = argparse.ArgumentParser(); ap.add_argument("--precision", default="bf16"); ap.add_argument("--profile", action="store_true"); ap.add_argument("--small", action="store_true"); args = ap.parse_args()

def run(model_kw, B, T, N, seconds, label, iters=30):
    torch.manual_seed(0)
    m = AVSeparationTransformer(**model_kw, precision=args.precision).cuda()
    mixed, frames = synthetic_batch(B, model_kw.get("freq_bins", 257), T, N, 32, 32, seed=1, device="cuda")
    m.prepack("cuda")
    for _ in range(4):
        m(mixed, frames)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        m(mixed, frames)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    out = dict(config=label, B=B, T=T, N=N, ms_per_forward=round(ms, 4), utt_s_per_s=round(B * seconds / (ms * 1e-3), 1),
               launches=m.engine.launch_count(), precision=args.precision)
    print(json.dumps(out), flush=True)
    if args.profile:
        m.engine.set_profile(True); m.engine.profile_report(reset=True)
        for _ in range(5):
            m(mixed, frames)
        prof = m.engine.profile_report(reset=True); m.engine.set_profile(False)
        tot = sum(v[1] for v in prof.values())
        print("   " + "  ".join(f"{k}:{v[1]/5:.3f}ms({100*v[1]/tot:.0f}%)" for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])), flush=True)
    m.engine.close()
    return out

default = dict(freq_bins=257, d_model=256, nhead=4, num_encoder_layers=2, num_fusion_layers=2, num_speakers=2)
scaled = dict(freq_bins=257, d_model=512, nhead=8, num_encoder_layers=6, num_fusion_layers=6, num_speakers=3)
res = []
if args.small:
    for B in (8, 16, 32, 64, 96, 128):
        run(default, B, 63, 50, 1.0, f"B={B}")
    sys.exit(0)
if args.profile:
    run(default, 32, 1251, 500, 10.0, "C3 long-form B=32", iters=5)
    run(scaled, 256, 63, 50, 1.0, "C4 scaled B=256", iters=5)
    run(default, 8, 63, 50, 1.0, "C1 B=8", iters=5)
    sys.exit(0)
res.append(run(default, 8, 63, 50, 1.0, "C1 demo default B=8"))
res.append(run(default, 256, 63, 50, 1.0, "C2 B=256"))
res.append(run(default, 8, 1251, 500, 10.0, "C3 long-form 10 s @ 16 kHz, B=8"))
res.append(run(default, 32, 1251, 500, 10.0, "C3 long-form B=32", iters=10))
res.append(run(scaled, 32, 63, 50, 1.0, "C4 scaled d=512 6+6 S=3, B=32"))
res.append(run(scaled, 256, 63, 50, 1.0, "C4 scaled B=256", iters=10))
for B in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024):
    res.append(run(default, B, 63, 50, 1.0, f"C5 sweep B={B}", iters=20 if B <= 256 else 8))
