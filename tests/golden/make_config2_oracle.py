"""Record the CPU oracle's config-2 results that test_config2_oracle_parity_large compares the CUDA path
against (run: python tests/golden/make_config2_oracle.py).

bench.cpu_pipeline at N = 32768 is a dense LAPACK Cholesky of a 8.6 GB matrix: minutes of CPU time and
~35 GB of host memory on every GPU test run.  Its output (logpdf, posterior mean and variance at the
512 test points of bench.make_inputs) is stored instead, so the comparison runs on any host.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import bench  # noqa: E402

SIZES = (16384, 32768)
NS = 512


def main():
    out = {}
    for n in SIZES:
        x, y, xs = bench.make_inputs(n, NS)
        lp, mean, var, _ = bench.cpu_pipeline(x, y, xs, bench.SIGMA2)
        out[str(n)] = {"n": n, "ns": NS, "sigma2": bench.SIGMA2, "logpdf": float(lp),
                       "mean": [float(v) for v in mean], "var": [float(v) for v in var]}
        print(n, lp, flush=True)
    path = os.path.join(HERE, "config2_oracle.json")
    with open(path, "w") as fh:
        json.dump(out, fh)
    print("wrote", path)


if __name__ == "__main__":
    main()
