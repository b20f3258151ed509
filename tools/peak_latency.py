"""Developer tool: the arithmetic-only micro-kernel (te_idm_peak_form) at w warps per SM -> updates per clock per SM and
the implied latency of one dependent IDM update (w = 4: one warp per scheduler), for both forms of the update."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from traffic_env_b200.vec_env import idm_arithmetic_peak
for w in (4, 8, 12, 16, 20, 24, 28, 32):
    r = idm_arithmetic_peak(iters=4000, form=0, warps_per_sm=w)
    per_clk_sm = r / 148 / 1.965e9
    # w/4 warps per scheduler, each issuing one update of 32 cars per L cycles: r = 148 * w * 32 / L * clk
    L = 148 * w * 32 * 1.965e9 / r
    print("general checked form, warps/SM %2d  %.3e updates/s  %.3f updates/clk/SM  cycles per warp-update %.0f" % (w, r, per_clk_sm, L))
for w in (4, 8, 12, 16, 20, 24, 32, 0):
    r = idm_arithmetic_peak(iters=4000, form=5, warps_per_sm=w)
    print("tame form (step kernels on a tame handle), warps/SM %2d  %.3e updates/s" % (w or 64, r))
print("general checked form, 64 warps/SM: %.3e" % idm_arithmetic_peak(iters=4000, form=0, warps_per_sm=0))
