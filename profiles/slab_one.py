"""One 16384^2 plane through the slab path on ONE GPU (world = 1), a few iterations of GS and GD: the command the ncu
captures of the slab kernels are taken from (profiles/r2_ncu_slab.md)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from spatial_light_modulator_module_b200 import host_logic as hl
from spatial_light_modulator_module_b200.slab import SlabEngine
n = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
eng = SlabEngine(n, 1, 0, "fp32")
t = eng._mem_upload((np.random.default_rng(100).random((n, n)) * 255).astype(np.uint8))
h, _, errs = eng.gs(t, 3, want_expected=False, on_device=True)
u = eng._mem_upload(np.random.default_rng(200).random((n, n)))
x0 = eng._mem_empty((n, n), eng.complex_dtype)
eng._check(eng._lib.slm_random_phasor(eng._ctx, eng._mem_ptr(u), eng._mem_ptr(x0), n * n, 1.0))
h, _, errs_gd = eng.gd(t, x0, hl.learning_rate_schedule(0.005, 0, 3)[0], 3, want_expected=False, on_device=True)
print("GS", errs, "GD", errs_gd)
eng.close()
