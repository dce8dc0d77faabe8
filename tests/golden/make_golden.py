#!/usr/bin/env python
"""Collects the reference's own golden DATA (no code) into tests/golden/ from a checkout of Pioran.jl:
    python tests/golden/make_golden.py PATH_TO_PIORAN_JL

What is collected (all are outputs or inputs of the reference itself, MIT licence):
  * test/data/simu_log.txt, test/data/simu.txt                      — inputs of test/test_likelihood.jl
  * examples/ultranest/inference/<run>/<run>_subset_time_series.txt  — the exact series a shipped run used
  * examples/ultranest/inference/<run>/chains/weighted_post.txt      — (θ, logL) pairs produced by the reference
    (Julia Pioran.logpdf called by ultranest, examples/ultranest/{single_pl,double_pl,single_pl_periodicity}.jl)
  * examples/ultranest/inference/simu_single/info/results.json       — maximum_likelihood {logl, point}
Chains are stored as float64 .npy inside compressed .npz files (text → binary is exact: 18 significant digits):
simu_single and simu_double in chains.npz, simu_periodic_rednoise in simu_periodic_rednoise_chains.npz, so that no
golden file exceeds 1 MB.
"""
import json, os, shutil, sys
import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
OWN_FILE = ("simu_periodic_rednoise",)   # runs written to <stem>_chains.npz instead of chains.npz

def main(ref):
    for f in ("simu_log.txt", "simu.txt"):
        shutil.copyfile(f"{ref}/test/data/{f}", f"{OUT}/{f}")
    runs = {
        "simu_single": "simu_single",
        "simu_double": "simu_double",
        "simu_periodic_rednoise_123_factor": "simu_periodic_rednoise",
    }
    chains = {}
    for run, stem in runs.items():
        base = f"{ref}/examples/ultranest/inference/{run}"
        shutil.copyfile(f"{base}/{stem}_subset_time_series.txt", f"{OUT}/{stem}_subset_time_series.txt")
        with open(f"{base}/chains/weighted_post.txt") as fh:
            header = fh.readline().split()
        arr = np.loadtxt(f"{base}/chains/weighted_post.txt", skiprows=1)
        print(run, arr.shape, header)
        if stem in OWN_FILE:
            np.savez_compressed(f"{OUT}/{stem}_chains.npz", **{stem: arr, stem + "_columns": np.array(header)})
        else:
            chains[stem] = arr
            chains[stem + "_columns"] = np.array(header)
    np.savez_compressed(f"{OUT}/chains.npz", **chains)
    with open(f"{ref}/examples/ultranest/inference/simu_single/info/results.json") as fh:
        res = json.load(fh)
    with open(f"{OUT}/simu_single_maximum_likelihood.json", "w") as fh:
        json.dump(res["maximum_likelihood"], fh, indent=1)

if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
