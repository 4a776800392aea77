"""Measured block-scaled FP4 tensor peak of this GPU (tcgen05.mma kind::mxf4, A operand in tensor memory, on every
SM for >= 2 s) with the clocks and power seen meanwhile, beside the int8 figure bench.py reports against.  Writes
one JSON line; king_ts_kernel's share of peak is its rate over ts_n160."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import plink_ng_b200 as p
from bench import ClockSampler

out = {}
with p.GpuContext(0) as ctx:
    for name, n, secs in (("ts_n160", 160, 2.5), ("ts_n80", 80, 1.0)):
        s = ClockSampler(0)
        s.start()
        tops, t = ctx.mxf4_peak(n, secs)
        out[name] = {"tops": tops, "seconds": t, "clocks": s.stop()}
    s = ClockSampler(0)
    s.start()
    tops, t = ctx.int8_peak(160, 1, 2.5)
    out["int8_ts_n160"] = {"tops": tops, "seconds": t, "clocks": s.stop()}
out["note"] = "all SMs, two issuer warps per SM, rounds of 32 back-to-back UMMAs (M=128, K=64 for mxf4, K=32 for int8) per commit"
print(json.dumps(out))
