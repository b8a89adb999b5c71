"""Launch the dominant kernels of the resnet_cifar10 B=256 cycle in isolation (for `ncu --set full`):
3x3 256->256 conv at 32x32 (G B3 / conv2) and the D-side 128->128 conv at 32x32 with B=512 — forward, input gradient,
filter gradient — each in the variants the library has: operand pre-rounded to TF32 by its producer (how the training
step runs them) or rounded in shared memory; per-tap boxes (default), halo boxes.
Every variant is launched ONCE after a warm-up pass that ncu skips (cudaProfilerStart): 2 shapes x 2 operand modes x
(2 forward + 2 input-gradient variants + 1 filter gradient) = 20 captured launches."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from compare_gan_b200 import _lib, kernels as K, tape

K.init(0)
K.set_math_mode(1)
lib = K.lib()
rng = np.random.RandomState(0)
for it, (b, h, cin, cout) in enumerate([(256, 32, 256, 256), (512, 32, 128, 128)] * 2):
  if it == 2:
    torch.cuda.synchronize()
    torch.cuda.profiler.start()          # the first pass over both shapes is the warm-up
  xr = K.relu(K.from_numpy(rng.randn(b, h, h, cin).astype(np.float32)), round_tf32=True)      # TF32-representable values
  w = K.from_numpy((rng.randn(3, 3, cin, cout) * 0.02).astype(np.float32), req=True)
  bias = K.zeros(cout)
  d = K.conv_desc(b, h, h, cin, cout, 3, 3, 1, False, "SAME")
  g = K.relu(K.from_numpy(rng.randn(b, h, h, cout).astype(np.float32)), round_tf32=True)
  for pre in (True, False):
    xr.tf32 = g.tf32 = pre
    for halo in (0, 2):
      lib.set_option(_lib.OPT_TC_HALO, halo)
      with tape.no_record():
        K.conv2d(xr, w, bias)
        K.conv2d_dgrad(d, g, w)
    lib.set_option(_lib.OPT_TC_HALO, 1)
    with tape.no_record():
      K.conv2d_wgrad(d, xr, g)
  torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("done")
