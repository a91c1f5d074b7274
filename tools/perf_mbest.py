"""Quick device-resident throughput probe (not the contract bench): python tools/perf_mbest.py [B] [modes]

modes: comma-separated, run in the order given (repeat them to alternate): hier, direct, norider, f32, or default
(Periods() without a fold mode, which ranks plain M-best with the fp32 nomination sweep)."""
import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from pyperiod_b200 import Periods, _lib, synth

B = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
modes = sys.argv[2].split(",") if len(sys.argv) > 2 else ["hier", "direct"]
stream = synth.synth_stream(B)
dev = torch.from_numpy(stream).cuda()
win = torch.as_strided(dev, (B, 4096), (512, 1))
TRUNC = os.environ.get("PP_TRUNC", "0") == "1"      # PP_TRUNC=1: Periods(True, False), the truncated fold
prof = torch.zeros(8, dtype=torch.int64, device="cuda")
_lib.set_profile_buffer(prof)
for mode in modes:
    fold = {"direct": _lib.FOLD_DIRECT, "norider": _lib.FOLD_HIERARCHICAL_NO_RIDERS, "f32": _lib.FOLD_NOMINATE_F32,
            "hier": _lib.FOLD_HIERARCHICAL, "default": None}[mode]
    P = Periods(True, False, fold_mode=fold) if TRUNC else Periods(fold_mode=fold)
    for name, fn in (("m_best", P.m_best), ("m_best_gamma", P.m_best_gamma)):
        fn(win, num=10, max_length=1024)
        fn(win, num=10, max_length=1024)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            r = fn(win, num=10, max_length=1024)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        pr = prof.cpu().numpy().astype(float); prof.zero_()
        print("   cycles/window: sweep %.0f  project %.0f  update %.0f  step2+out %.0f (factor norms %.0f, norms+decision %.0f, thread-0 block %.0f)" % (tuple(pr[:4] / pr[4]) + tuple(pr[5:8] / pr[4])))
        print(f"{mode:7s} {name:13s} B={B} {ms:9.2f} ms  {B / ms * 1e3:10.0f} win/s  sweeps/win={float(r.sweeps.float().mean()):.3f}", flush=True)
