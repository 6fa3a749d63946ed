"""Parity at benchmark shape, on the GPU: the whole stage (stage.run_stage: FASTA -> filter table -> 3 EC rounds -> final pass -> files) against
the files of the UNMODIFIED reference binary (-f0 --write-paf --write-ec) on the same seeded read set of SURVEY.md §8(d)'s shape:
diploid genome with 0.1 % SNPs, 5 % of it in 50-copy 5 kb repeat families (both orientations), 30x reads of 15 kb with 0.2 % errors, N bases.
.ovlp.paf / .ec.fa / .ovlp.source.bin / .ovlp.reverse.bin are compared by size and digest, .ec.bin up to the pad bytes the reference leaves undefined.
The reference's digests for the default set (4 Mb genome = 8000 reads, seed 77) are stored in tests/golden/stage_files.npz; HB_SCALE_MB /
HB_SCALE_SEED pick another set, which needs the reference binary built in oracle/_ref/ (profiles/ holds the log of a 20 Mb run)."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__)); ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools")); sys.path.insert(0, HERE)

import goldenlib  # noqa: E402

pytestmark = [pytest.mark.gpu]


def _cmp_files(td, a, b):
    """the files of prefix `a` that differ from those of prefix `b` (both under td)"""
    return goldenlib.diff_digests(goldenlib.stage_file_digests(os.path.join(td, a)), goldenlib.stage_file_digests(os.path.join(td, b)))


@pytest.fixture(scope="module")
def ref_run(tmp_path_factory):
    """the seeded read set and the digests of the reference binary's files for it: stored for the default set, else one run of oracle/_ref/hifiasm"""
    import simgen
    mb = float(os.environ.get("HB_SCALE_MB", "4")); seed = int(os.environ.get("HB_SCALE_SEED", "77")); td = str(tmp_path_factory.mktemp("scale"))
    fa = os.path.join(td, "reads.fa")
    rs = simgen.make(mb, 30, seed=seed, n_rate=0.0002, fasta=fa)
    want = goldenlib.stored_stage_digests(mb, 30, seed, 0.0002)
    if want is None:
        ref = os.path.join(ROOT, "oracle", "_ref", "hifiasm")
        if not os.path.exists(ref):
            pytest.skip("no stored digests for a %g Mb genome with seed %d, and oracle/_ref/hifiasm is not built (make -C oracle ref)" % (mb, seed))
        thr = len(os.sched_getaffinity(0))
        p = subprocess.run([ref, "-o", os.path.join(td, "ref"), "-t%d" % thr, "-f0", "--write-paf", "--write-ec", fa], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr[-2000:]
        want = goldenlib.stage_file_digests(os.path.join(td, "ref"))
    return mb, td, fa, rs, want


# default: the batches the anchor budget gives at this size (two), on two lanes.  Then many small batches on two lanes (each lane's host thread takes
# batches in turn on its own stream; what they add to the lists is added in batch order) and on one lane: the files must not depend on either.
@pytest.mark.parametrize("budget,lanes", [(None, None), ("6000000", "2"), ("6000000", "1")])
def test_whole_stage_files_equal_reference_binary_at_scale(ref_run, monkeypatch, budget, lanes):
    from hifiasm_b200 import stage
    mb, td, fa, rs, want = ref_run
    if budget:
        monkeypatch.setenv("HB_ANCHOR_BUDGET", budget)
    if lanes:
        monkeypatch.setenv("HB_LANES", lanes)
    if lanes == "1":
        monkeypatch.setenv("HB_NO_SKETCH_REUSE", "1")        # (this variant also sketches the query reads again instead of reading the index build's sketch)
    out = "gpu_%s_%s" % (budget, lanes)
    info = stage.run_stage(fa, os.path.join(td, out))
    assert info["reads"] == rs.n and info["bases"] == rs.bases
    diff = goldenlib.diff_digests(want, goldenlib.stage_file_digests(os.path.join(td, out)))
    print("scale parity (budget %s, lanes %s): %g Mb genome, %d reads, %d bases, corrected per round %s, overlaps %d + %d: %s" % (budget, lanes, mb, rs.n, rs.bases, info["corrected_bases"], info["overlaps_src"], info["overlaps_rev"], "identical" if not diff else diff))
    assert not diff, diff
