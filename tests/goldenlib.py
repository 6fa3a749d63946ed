"""Helpers shared by the CPU and GPU suites: load a golden data set
(tests/golden/*.npz, made by make_golden.py from the unmodified reference)."""
import hashlib
import io
import os
import tempfile

import numpy as np

from hifiasm_b200 import binio

GOLDEN = os.environ.get("HB_GOLDEN_DIR", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))  # the override: tools/fuzz_vs_reference.py
CH = np.dtype([("x_pos_s", "<u4"), ("x_pos_e", "<u4"), ("y_id", "<u4"), ("y_pos_s", "<u4"), ("y_pos_e", "<u4"),
               ("y_pos_strand", "<u4"), ("shared_seed", "<i4"), ("first_hit", "<u4"), ("n_fc", "<u4")])


def dg(b: bytes) -> int:
    return int.from_bytes(hashlib.blake2b(b, digest_size=8).digest(), "little")


def _load_bin(arr, loader):
    with tempfile.NamedTemporaryFile(suffix=".bin", delete=False) as f:
        f.write(arr.tobytes())
        p = f.name
    try:
        return loader(p)
    finally:
        os.unlink(p)


class Golden:
    def __init__(self, name):
        self.name = name
        self.z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.raw = _load_bin(self.z["raw_ec"], binio.load_ec_bin)
        self.pre = _load_bin(self.z["pre_ec"], binio.load_ec_bin)
        self.pre_src = _load_bin(self.z["pre_ovlp_source"], binio.load_ovlp_bin)
        self.pre_rev = _load_bin(self.z["pre_ovlp_reverse"], binio.load_ovlp_bin)
        self.fin_src = _load_bin(self.z["fin_ovlp_source"], binio.load_ovlp_bin)
        self.fin_rev = _load_bin(self.z["fin_ovlp_reverse"], binio.load_ovlp_bin)

    def params(self, mode):
        return dict(s.split("=") for s in self.z[mode + "_params"])

    def digest(self, mode, stage):
        return self.z["%s_dg_%s" % (mode, stage)]

    def count(self, mode, stage):
        return self.z["%s_n_%s" % (mode, stage)]


STAGE_FILES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stage_files.npz")


def stage_file_digests(prefix):
    """{file suffix: (size, blake2b-128 hex)} of the files a whole stage writes under `prefix` (-o prefix --write-paf --write-ec).
    .ec.bin is taken by what it holds (lengths, reads with the pad bytes the reference leaves undefined masked, names, coverage peaks), its size by
    the number of reads."""
    out = {}
    for suf in ("ovlp.paf", "ec.fa", "ovlp.source.bin", "ovlp.reverse.bin"):
        b = open(prefix + "." + suf, "rb").read()
        out[suf] = (len(b), hashlib.blake2b(b, digest_size=16).hexdigest())
    rs = binio.load_ec_bin(prefix + ".ec.bin")
    h = hashlib.blake2b(digest_size=16)
    for part in (rs.length.astype("<u8").tobytes(), binio.canonical_packed(rs).tobytes(), rs.name_blob, np.array([rs.hom_cov, rs.het_cov], "<i4").tobytes()):
        h.update(part)
    out["ec.bin"] = (rs.n, h.hexdigest())
    return out


def diff_digests(want, got):
    """the files whose digests differ, with both (size, digest) pairs"""
    return ["%s (%s vs %s)" % (k, want[k], got.get(k)) for k in sorted(want) if want[k] != got.get(k)]


def stored_stage_digests(genome_mb, cov, seed, n_rate):
    """stage_file_digests of the unmodified reference binary's files for the tools/simgen.py read set of these parameters
    (tests/golden/stage_files.npz, made by tests/golden/make_stage_files.py); None when that set is not stored"""
    z = np.load(STAGE_FILES)
    for name in str(z["sets"]).split(","):
        if tuple(z[name + "_params"]) == (float(genome_mb), float(cov), float(seed), float(n_rate)):
            return {str(s): (int(n), str(d)) for s, n, d in zip(z[name + "_suffix"], z[name + "_size"], z[name + "_dg"])}
    return None


def chain_digest(ch, fc_pool):
    """digest of chain records + fake cigars, the way make_golden.read_stages does.
    ch: structured array with fields of CH plus fc_off/fc_n"""
    h = hashlib.blake2b(digest_size=8)
    for c in ch:
        r = np.zeros(1, dtype=CH)
        for f in ("x_pos_s", "x_pos_e", "y_id", "y_pos_s", "y_pos_e", "y_pos_strand", "shared_seed"):
            r[f] = c[f]
        r["first_hit"] = c["non_homopolymer_errors"]
        r["n_fc"] = c["fc_n"]
        h.update(r.tobytes())
        h.update(np.ascontiguousarray(fc_pool[int(c["fc_off"]):int(c["fc_off"]) + int(c["fc_n"])]).tobytes())
    return int.from_bytes(h.digest(), "little")
