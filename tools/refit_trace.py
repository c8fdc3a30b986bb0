import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import b7_oracle as o
from bot7_b200 import _lib as L, models
N, d = 4096, 6
X = o.sobol_points(d, N); y = o.hartmann6(X); y = (y - y.mean()) / y.std()
h = np.zeros((1, d + 3)); h[0, :d] = np.log(0.4); h[0, d + 1] = 0.5 * np.log(1e-2)
f = models.GPFactors(X, y, h, flags=L.FIT_LOGML_ONLY)
for _ in range(3): f.refit(h + 0.01, L.FIT_LOGML_ONLY)
f.free()
