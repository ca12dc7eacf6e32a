import os, cProfile, pstats, sys, time, io
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
n = int(sys.argv[1]) if len(sys.argv) > 1 else 512
frames = synthetic.movie_frames(n)
mask = synthetic.random_mask((768, 1024), seed=1)
for name, kw in (("uint8", dict(output="uint8", mask=mask, ct2pi=256)), ("float64", dict(output="float64"))):
    for rep in range(3):
        t0 = time.perf_counter()
        out = ghs.sequence_holograms(frames, 50, precision="fp32", batch=32, **kw)
        torch.cuda.synchronize()
        print(name, "call", rep, "%.3f s" % (time.perf_counter() - t0), flush=True)
    pr = cProfile.Profile()
    pr.enable()
    out = ghs.sequence_holograms(frames, 50, precision="fp32", batch=32, **kw)
    torch.cuda.synchronize()
    pr.disable()
    s = io.StringIO()
    pstats.Stats(pr, stream=s).sort_stats("tottime").print_stats(14)
    print(s.getvalue()[:3500])
    del out
