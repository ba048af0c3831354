#!/usr/bin/env python
"""FFT Toeplitz timing probe (development tool): python tools/fft_probe.py [L ...]"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmomap2_b200 as cm  # noqa: E402
from cosmomap2_b200 import synthetic, _device as dv  # noqa: E402
from kbench import timeit  # noqa: E402


def main():
    nt, ndet = 100000000, 64
    ns = nt // ndet
    d = dv.to_dev_f64(np.random.default_rng(2).standard_normal(nt))
    out = {}
    for L in [int(a) for a in sys.argv[1:]] or [256, 4096]:
        N = cm.BlockLO(ns, synthetic.toeplitz_bands(ndet, L), offdiag=True)
        t = timeit(lambda: N._apply(d), reps=5, warm=2)
        out["toeplitz%d_fft_ms" % L] = t
    print(json.dumps(out))


if __name__ == "__main__":
    main()
