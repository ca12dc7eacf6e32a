import os, sys, time, argparse, contextlib, io
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from spatial_light_modulator_module_b200 import algorithms, display_holograms, host_logic as hl, synthetic
from spatial_light_modulator_module_b200.engine import get_engine
shape=(1024,1024)
ns = argparse.Namespace(incomming_intensity="uniform", tolerance=0, max_loops=100, gif=False, print_info=False, plot_error=False, initial_guess="random", random_seed=42, white_attention=1, learning_rate=0.005, unsettle=0, precision="fp32", device=0)
t = synthetic.noise_target(shape, seed=1); mask = synthetic.random_mask(shape)
def T(): torch.cuda.synchronize(); return time.perf_counter()
with contextlib.redirect_stdout(io.StringIO()):
    algorithms.gradient_descent(t, ns); ns.learning_rate=0.005
for rep in range(3):
    eng = get_engine(shape, "fp32", 1, 0)
    a=T(); u = eng.python_random_uniform(42, shape); b=T()
    x0 = eng.random_phasor_guess(u, 1.0); c=T()
    during, after = hl.learning_rate_schedule(0.005, 0, 100)
    res, x = eng.gd(t, x0, during, 100); d=T()
    h = eng.to_host(res.hologram)[0]; e=T()
    ex = eng.to_host(res.expected)[0]; f=T()
    g = display_holograms.hologram_to_grey(h, mask, 256); gg=T()
    print(f"MT19937 stream on device {1e3*(b-a):.2f}  phasor {1e3*(c-b):.2f}  gd {1e3*(d-c):.2f}  holo D2H {1e3*(e-d):.2f}  exp D2H {1e3*(f-e):.2f}  grey(upload+quant+D2H) {1e3*(gg-f):.2f}  total {1e3*(gg-a):.2f}")
