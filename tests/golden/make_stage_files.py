#!/usr/bin/env python
"""Regenerates tests/golden/stage_files.npz: the files the UNMODIFIED reference binary writes when a user runs the whole stage on a
tools/simgen.py read set — `hifiasm -o X -t<cores> -f0 --write-paf --write-ec reads.fa` (oracle/_ref/hifiasm) — kept as the size and
blake2b-128 digest of each file (goldenlib.stage_file_digests; the files themselves are tens of megabytes).  The sets are the ones
__graft_entry__.smoke() and tests/test_gpu_scale.py run the device's stage on.
Only runs where oracle/_ref/hifiasm is built."""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tools"))
import goldenlib  # noqa: E402
import simgen  # noqa: E402

HIFIASM = os.path.join(ROOT, "oracle", "_ref", "hifiasm")
# name: (genome Mb, coverage, seed, N rate)
SETS = {"smoke": (0.5, 30, 5, 0.0002), "scale": (4, 30, 77, 0.0002)}


def main():
    if not os.path.exists(HIFIASM):
        sys.exit("build oracle/_ref first: make -C oracle ref")
    arrs = {"sets": np.array(",".join(SETS))}
    for name, (mb, cov, seed, n_rate) in SETS.items():
        with tempfile.TemporaryDirectory() as td:
            fa = os.path.join(td, "reads.fa")
            simgen.make(mb, cov, seed=seed, n_rate=n_rate, fasta=fa)
            p = subprocess.run([HIFIASM, "-o", os.path.join(td, "ref"), "-t%d" % len(os.sched_getaffinity(0)), "-f0", "--write-paf", "--write-ec", fa],
                               capture_output=True, text=True)
            assert p.returncode == 0, p.stderr[-2000:]
            d = goldenlib.stage_file_digests(os.path.join(td, "ref"))
        arrs[name + "_params"] = np.array([mb, cov, seed, n_rate], np.float64)
        arrs[name + "_suffix"] = np.array(list(d))
        arrs[name + "_size"] = np.array([v[0] for v in d.values()], np.uint64)
        arrs[name + "_dg"] = np.array([v[1] for v in d.values()])
        print(name, d)
    np.savez_compressed(goldenlib.STAGE_FILES, **arrs)
    print("->", goldenlib.STAGE_FILES, os.path.getsize(goldenlib.STAGE_FILES), "bytes")


if __name__ == "__main__":
    main()
