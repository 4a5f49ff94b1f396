"""The .pgen restatement (oracle/pgen.py) against the reference's own fixture pair: example/example.pgen must decode to
exactly the genotypes of example/example.bed (both ship with the reference and hold the same 1000 x 500 calls), and a
synthetic file written record type by record type (tests/helpers.write_pgen) must round-trip."""
import collections

import numpy as np

import helpers
from oracle import pgen, plink


def test_example_pgen_equals_example_bed(golden_dir):
    d = golden_dir
    pg = pgen.Pgen(d + "/example.pgen")
    bim = plink.read_bim(d + "/example.bim")
    keys, _ = plink.read_fam(d + "/example.fam")
    G = plink.decode_bed(plink.read_bed_rows(d + "/example.bed", len(keys), bim.offset), len(keys))
    assert (pg.m, pg.n) == (1000, 500) and int(pg.fpos[-1]) == len(pg.d)
    for v in range(pg.m):
        g = pg.read(v).astype(float)
        g[g == 3] = -3.0
        assert np.array_equal(g, G[v]), v
    pv = pgen.read_pvar(d + "/example.pvar")
    ks, _ = pgen.read_psam(d + "/example.psam")
    assert ks == keys
    assert [(r[2], r[3], r[4]) for r in pv] == list(zip(bim.ids, bim.allele0, bim.allele1))   # ALLELE0 = REF, ALLELE1 = ALT


def synthetic_calls(N=700, M=160, seed=1):
    rng = np.random.default_rng(seed)
    g = np.zeros((M, N), dtype=np.uint8)
    for v in range(M):
        kind = v % 8
        if kind == 0:
            pass                                              # all hom-ref
        elif kind == 1:
            g[v] = rng.binomial(2, 0.15, N)                   # common (hom-alt below n / 16: a 1-bit record)
        elif kind == 2:
            g[v] = rng.binomial(2, 0.01, N)                   # rare
        elif kind == 3:
            g[v] = 2 - rng.binomial(2, 0.01, N)               # almost fixed for ALT
        elif kind == 4:
            g[v] = np.where(rng.random(N) < 0.95, 3, rng.binomial(2, 0.4, N))   # mostly missing
        elif kind == 5:
            g[v] = g[v - 4].copy(); g[v, rng.integers(0, N, 5)] = 1              # in LD with a common one
        elif kind == 6:
            t = g[v - 5].copy(); t[rng.integers(0, N, 4)] = 3
            g[v] = np.array([2, 1, 0, 3], dtype=np.uint8)[t]                      # inverted LD
        elif v % 16 == 7:
            g[v] = rng.integers(0, 4, N)                      # nothing compresses
        else:
            g[v] = g[v - 2].copy(); g[v, rng.integers(0, N, 6)] = 2              # LD with the latest non-LD record
    return g


def test_pgen_round_trip_all_record_types(tmp_path):
    g = synthetic_calls()
    for storage in (1, 6):
        prefix = str(tmp_path / ("syn%d" % storage))
        types = helpers.write_pgen(prefix, g, storage=storage)
        assert set(types) >= {0, 1, 2, 3, 4, 5, 6, 7}, collections.Counter(types)
        pg = pgen.Pgen(prefix + ".pgen")
        for v in list(range(g.shape[0])) + [150, 7, 6, 5, 13, 14]:       # sequential, then random access into LD records
            assert np.array_equal(pg.read(v), g[v]), (storage, v, types[v])


# ------------------------------------------------------------------------------------ pinned on the reference's own pgenlib
# What pgenlib returned is stored as digests (tests/golden/ref/, helpers.ref_golden): the bytes of each file it validated
# and of the calls it read from it.
def test_oracle_equals_pgenlib_on_the_reference_fixture(golden_dir):
    """oracle/pgen.py vs the reference's vendored pgenlib, called as the reference calls it (ReadHardcalls, allele 1)."""
    path = golden_dir + "/example.pgen"

    def pgenlib():
        from oracle import pgenlib_ref as ref
        ref.validate(path)
        return {"pgen": helpers.sha256(np.fromfile(path, dtype=np.uint8)),
                "calls": helpers.sha256(ref.read_hardcalls(path, 500, 0, 1000))}
    want = helpers.ref_golden("pgenlib_example", pgenlib)
    assert np.array_equal(helpers.sha256(np.fromfile(path, dtype=np.uint8)), want["pgen"])
    pg = pgen.Pgen(path)
    got = np.stack([pg.read(v).astype(float) for v in range(1000)])
    got[got == 3] = -3.0
    assert np.array_equal(helpers.sha256(got), want["calls"])


def test_synthetic_files_pass_pgenlib_validation_and_read_back(tmp_path):
    """The test writer (helpers.write_pgen) is itself checked by the reference library: PgrValidate accepts the files
    (record types, difflist group byte counts, trailing bits) and ReadHardcalls returns the calls that were written - with
    all samples and with a sample subset (pgenlib's proper-subset readers skip difflist groups by their byte counts) - and
    oracle/pgen.py agrees.  Covers difflists of > 32 groups and 1 / 2 / 3-byte sample ids, which the fixture does not."""
    from test_host_cpu import big_pgen_calls
    cases = ((700, 160, 5), (33333, 40, 6), (70001, 20, 2))
    files = {}
    for N, M, storage in cases:
        g = synthetic_calls() if N == 700 else big_pgen_calls(N, M)
        pfx = str(tmp_path / ("s%d" % N))
        types = helpers.write_pgen(pfx, g, storage=storage)
        assert set(types) >= set(range(8))
        sub = np.sort(np.random.default_rng(N).choice(g.shape[1], g.shape[1] // 3, replace=False))
        files[N] = (g, pfx + ".pgen", sub)

    def pgenlib():
        from oracle import pgenlib_ref as ref
        out = {}
        for N, (g, path, sub) in files.items():
            ref.validate(path)
            out["pgen%d" % N] = helpers.sha256(np.fromfile(path, dtype=np.uint8))
            out["calls%d" % N] = helpers.sha256(ref.read_hardcalls(path, g.shape[1], 0, g.shape[0]))
            out["subset%d" % N] = helpers.sha256(ref.read_hardcalls(path, g.shape[1], 0, g.shape[0], subset=sub))
        return out
    ref = helpers.ref_golden("pgenlib_synthetic", pgenlib)
    for N, (g, path, sub) in files.items():
        assert np.array_equal(helpers.sha256(np.fromfile(path, dtype=np.uint8)), ref["pgen%d" % N]), N
        want = g.astype(float)
        want[want == 3] = -3.0
        assert np.array_equal(helpers.sha256(want), ref["calls%d" % N]), N
        assert np.array_equal(helpers.sha256(want[:, sub]), ref["subset%d" % N]), N
        pg = pgen.Pgen(path)
        for v in (list(range(g.shape[0])) + [g.shape[0] - 1, 3, 1]):
            assert np.array_equal(pg.read(v), g[v]), (N, v)
