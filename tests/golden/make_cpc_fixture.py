"""Converts the reference's real-world test raster (py-dcdf/tests/testdata.txt: one 360x720 float32
CPC-precip day, read by py-dcdf/tests/test_dcdf.py:344-355) into tests/golden/cpc_day_360x720.npz.
Usage: python tests/golden/make_cpc_fixture.py <py-dcdf checkout>/tests/testdata.txt"""
import os
import sys

import numpy as np
vals = np.loadtxt(sys.argv[1], dtype=np.float32)
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpc_day_360x720.npz"), day=vals.reshape(360, 720))
print(vals.shape, np.isnan(vals).mean())
