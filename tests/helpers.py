"""Shared builders for the parity tests: synthetic PLINK filesets + oracle-side preparation."""
import os

import numpy as np

from oracle import plink, prep, step1
from regenie_b200 import synth


def write_fileset(d, g, Y, cov, na, n_chr=3, drop_pheno=(), drop_cov=()):
    """Write <d>/syn.{bed,bim,fam}, pheno.txt, covar.txt.  g: [M, N] codes (3 = missing)."""
    M, N = g.shape
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "syn.bed"), "wb") as fh:
        fh.write(b"\x6c\x1b\x01")
        fh.write(synth.pack_bed(g).tobytes())
    per = int(np.ceil(M / n_chr))
    with open(os.path.join(d, "syn.bim"), "w") as fh:
        for i in range(M):
            fh.write("%d rs%d 0 %d A G\n" % (i // per + 1, i, 1000 + i))
    with open(os.path.join(d, "syn.fam"), "w") as fh:
        for s in range(N):
            fh.write("F%d I%d 0 0 %d -9\n" % (s, s, 1 + s % 2))
    with open(os.path.join(d, "pheno.txt"), "w") as fh:
        fh.write("FID IID " + " ".join("Y%d" % (p + 1) for p in range(Y.shape[1])) + "\n")
        for s in range(N):
            if s in drop_pheno:
                continue
            fh.write("F%d I%d " % (s, s) + " ".join(
                "NA" if na[s, p] else repr(float(Y[s, p])) for p in range(Y.shape[1])) + "\n")
    with open(os.path.join(d, "covar.txt"), "w") as fh:
        fh.write("FID IID " + " ".join("V%d" % (c + 1) for c in range(cov.shape[1])) + "\n")
        for s in range(N):
            if s in drop_cov:
                continue
            fh.write("F%d I%d " % (s, s) + " ".join(repr(float(v)) for v in cov[s]) + "\n")
    return os.path.join(d, "syn")


class Problem:
    """Everything both sides need for a QT Step-1 run on a PLINK fileset."""

    def __init__(self, prefix, pheno, covar, bsize, K=5, loocv=False, remove=None, rint=False):
        self.bim = plink.read_bim(prefix + ".bim")
        keys_file, _ = plink.read_fam(prefix + ".fam")
        self.n_file = len(keys_file)
        remove = set(remove or ())
        self.keep = np.array([k not in remove for k in keys_file])
        self.sample_idx = np.nonzero(self.keep)[0].astype(np.int32)
        self.keys = [k for k in keys_file if k not in remove]
        self.prep = prep.prepare(self.keys, pheno, covar, rint=rint)
        self.blocks = prep.set_blocks(self.bim.chrom, bsize)
        self.bsize = bsize
        self.loocv = loocv
        self.K = K
        self.fold_sizes = (np.array([len(self.keys)]) if loocv
                           else prep.set_folds(self.prep.in_analysis, K))
        self.packed = plink.read_bed_rows(prefix + ".bed", self.n_file, self.bim.offset)
        self.M = len(self.bim.ids)
        self.h0 = prep.set_ridge_params(5)
        self.lam = self.M * (1 - self.h0) / self.h0

    def oracle_block(self, b):
        c, s, bs = self.blocks[b]
        g = plink.decode_bed(self.packed[s:s + bs], self.n_file, keep=self.keep)
        gi, mu = plink.mean_impute_block(g, self.prep.in_analysis)
        return gi, mu

    def oracle_l0(self, b):
        gi, mu = self.oracle_block(b)
        pr = self.prep
        Gt, sd = step1.residualize_genotypes(gi, pr.X, pr.in_analysis, pr.n_analyzed, pr.ncov)
        if self.loocv:
            W = step1.level0_loocv(Gt, pr.Y, pr.mask, self.lam, pr.neff)
        else:
            W = step1.level0_kfold(Gt, pr.Y, pr.mask, self.fold_sizes, self.lam, pr.neff)
        return W, mu, sd, Gt

    def gpu_step1(self, device=0):
        from regenie_b200 import capi
        pr = self.prep
        return capi.Step1(pr.X, pr.Y, pr.mask, pr.in_analysis, self.fold_sizes, self.lam, pr.neff,
                          pr.n_analyzed, self.bsize, len(self.blocks), loocv=self.loocv, device=device)

    def gpu_l0_block(self, st, b):
        c, s, bs = self.blocks[b]
        idx = None if self.keep.all() else self.sample_idx
        st.l0_block_bed(self.packed[s:s + bs], bs, b, sample_idx=idx)


def synthetic_problem(tmp, N=1000, M=300, P=3, C=3, bsize=128, K=5, miss=0.02, seed=7, na_frac=0.03,
                      drop=True, loocv=False):
    g = synth.genotypes(N, M, seed=seed, miss=miss)
    Y, cov, na = synth.phenotypes(g, P, C, seed=seed, na_frac=na_frac)
    drop_p = {5, 77, N - 3} if drop else ()
    drop_c = {11, 500 % N} if drop else ()
    prefix = write_fileset(str(tmp), g, Y, cov, na, drop_pheno=drop_p, drop_cov=drop_c)
    return Problem(prefix, str(tmp) + "/pheno.txt", str(tmp) + "/covar.txt", bsize, K=K, loocv=loocv)


def oracle_step2_rows(prefix, pheno, covar, pred_list, bsize, remove=None, htp=None):
    """Full QT Step 2 on the CPU oracle, reading the .loco files like the reference does.

    Returns {phenotype name: [row strings]} in the native split-by-phenotype format, or (htp = cohort name) as HTP rows.
    """
    from oracle import step2
    bim = plink.read_bim(prefix + ".bim")
    keys_file, _ = plink.read_fam(prefix + ".fam")
    remove = set(remove or ())
    keep = np.array([k not in remove for k in keys_file])
    keys = [k for k in keys_file if k not in remove]
    sidx = {k: i for i, k in enumerate(keys)}
    n = len(keys)
    pr = prep.prepare(keys, pheno, covar, step=2)
    files = dict(l.split() for l in open(pred_list) if l.strip())
    locos = [step2.read_loco(files[nm]) for nm in pr.pheno_names]
    extra = np.stack([step2.blup_mask(ids, rows[1], sidx, n) for ids, rows in locos], axis=1)
    # blup_read masks, then prep_run's second setMasks + basis + residualise (src/Pheno.cpp:1060-1175)
    names, Yraw, in_ph = prep.read_table(pheno, sidx, n)
    pr = prepare_step2_with_mask(keys, pheno, covar, extra)
    strict = len(pr.pheno_names) == 1
    packed = plink.read_bed_rows(prefix + ".bed", len(keys_file), bim.offset)
    out = {nm: [] for nm in pr.pheno_names}
    cur = None
    for i in range(len(bim.ids)):
        c = int(bim.chrom[i])
        if c != cur:
            cur = c
            blups = np.stack([step2.blup_chr(ids, rows[c], sidx, n, pr.in_analysis, pr.mask[:, ph])
                              for ph, (ids, rows) in enumerate(locos)], axis=1)
            res, p_sd, scf = step2.compute_res(pr.Y, blups, pr.mask, pr.neff, pr.ncov, pr.scale_Y)
            YtX = res.T @ pr.X
        graw = plink.decode_bed(packed[i:i + 1], len(keys_file), keep=keep)[0]
        vs = step2.variant_stats(graw, pr.in_analysis, pr.mask)
        if vs["ignored"]:
            continue
        sc = step2.score_qt(vs["g"], pr.X, res, pr.mask, pr.in_analysis, pr.n_analyzed, pr.ncov, scf, YtX, strict)
        if sc is None:
            continue
        for ph, nm in enumerate(pr.pheno_names):
            if vs["ignored_trait"][ph]:
                continue
            if htp is not None:
                gc = step2.genocounts(graw, np.nonzero(pr.mask[:, ph])[0])
                out[nm].append(step2.htp_row(bim.ids[i], c, int(bim.pos[i]), bim.allele0[i], bim.allele1[i], nm, htp,
                                             step2.htp_model(), sc["beta"][ph], sc["se"][ph], sc["chisq"][ph], sc["logp"][ph],
                                             vs["af"][ph], vs["mac"][ph], gc, score=sc["score"][ph], skat_var=sc["skat_var"][ph]))
                continue
            out[nm].append(step2.sumstats_row(c, int(bim.pos[i]), bim.ids[i], bim.allele0[i], bim.allele1[i],
                                              vs["af"][ph], vs["ns"][ph], sc["beta"][ph], sc["se"][ph],
                                              sc["chisq"][ph], sc["logp"][ph]))
    return out


def prepare_step2_with_mask(keys, pheno, covar, extra_mask):
    """prep.prepare(step=2) with the LOCO-availability mask applied where blup_read applies it."""
    n = len(keys)
    sidx = {k: i for i, k in enumerate(keys)}
    names, Y, in_ph = prep.read_table(pheno, sidx, n)
    P = len(names)
    strict = P == 1
    miss = Y == prep.MISSING
    mask = np.ones((n, P), dtype=bool) & ~miss
    if strict:
        anym = miss.any(axis=1); mask[anym] = False; all_miss = anym
    else:
        all_miss = miss.all(axis=1)
    in_ph = in_ph & ~all_miss
    mask &= in_ph[:, None]
    X = np.ones((n, 1)); in_cov = np.ones(n, dtype=bool)
    if covar:
        cn, Cv, in_cov = prep.read_table(covar, sidx, n, lambda nm: nm not in names)
        in_cov = in_cov & ~(Cv == prep.MISSING).any(axis=1)
        X = np.hstack([X, Cv])
    in_an = in_ph & in_cov
    # first setMasks + impute (read_pheno_and_cov)
    in_an = in_an & (mask.all(axis=1) if strict else mask.any(axis=1))
    mask = mask & in_an[:, None]
    Y = Y * in_an[:, None]; X = X * in_an[:, None]
    for j in range(P):
        y = Y[:, j]; ok = y != prep.MISSING
        y[~ok] = y[ok].sum() / (in_an & ok).sum()
    Y = Y * mask
    # blup_read + second setMasks (prep_run)
    mask = mask & extra_mask
    in_an = in_an & (mask.all(axis=1) if strict else mask.any(axis=1))
    mask = mask & in_an[:, None]
    Y = Y * in_an[:, None]; X = X * in_an[:, None]
    neff = mask.sum(axis=0).astype(float)
    Xb, ncov = prep.get_basis(X)
    beta = Y.T @ Xb
    Y = Y - (Xb @ beta.T) * mask
    scale_Y = np.linalg.norm(Y, axis=0) / np.sqrt(neff - ncov)
    Y = Y / scale_Y[None, :]
    return prep.Prepared(list(keys), names, Y, None, mask, Xb, in_an, neff, scale_Y, ncov, int(in_an.sum()))


# ---------------------------------------------------------------------------------------- .pgen writer
from regenie_b200.synth import write_pgen, gather_pgen_records  # noqa: E402,F401  (synthetic-data generator; checked by pgenlib in tests)


def gather_pgen(pg, variants):
    """What host/pgen.cpp PgenFile::gather hands to rg_pgen_decode, from an oracle.pgen.Pgen: the record bytes of the
    variants (and of the bases of LD-compressed ones) at 16-byte aligned offsets + the index tables."""
    recs = {}

    def rec(v):
        if v not in recs:
            recs[v] = pg.d[int(pg.fpos[v]):int(pg.fpos[v + 1])]
        return recs[v]
    return gather_pgen_records(rec, lambda v: int(pg.vrtype[v]) & 7, variants)


def write_pvar_psam(prefix, chroms, ids, pos, ref, alt, keys, sex=None):
    with open(prefix + ".pvar", "w") as fh:
        fh.write("##fileformat=test\n#CHROM\tPOS\tID\tREF\tALT\n")
        for c, p, i, r, a in zip(chroms, pos, ids, ref, alt):
            fh.write("%s\t%d\t%s\t%s\t%s\n" % (c, p, i, r, a))
    with open(prefix + ".psam", "w") as fh:
        fh.write("#FID\tIID\tSEX\n")
        for j, k in enumerate(keys):
            f, i = k.split("_", 1)
            fh.write("%s\t%s\t%s\n" % (f, i, "NA" if sex is None else sex[j]))


# ---------------------------------------------------------------------------------------- BGEN re-compression (tests only)
def recompress_bgen(src, dst, mode):
    """Rewrite a zlib-compressed BGEN v1.2 file with compression flag `mode` (0 = none, 2 = zstd via libzstd)."""
    import ctypes
    import struct
    import zlib
    d = open(src, "rb").read()
    (offset,) = struct.unpack_from("<I", d, 0)
    lh, m, n = struct.unpack_from("<III", d, 4)
    (flags,) = struct.unpack_from("<I", d, 4 + lh - 4)
    assert flags & 3 == 1
    out = bytearray(d[:offset + 4])
    struct.pack_into("<I", out, 4 + lh - 4, (flags & ~3) | mode)
    zs = None
    if mode == 2:
        zs = ctypes.CDLL("libzstd.so.1")
        zs.ZSTD_compress.restype = ctypes.c_size_t
        zs.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int]
        zs.ZSTD_compressBound.restype = ctypes.c_size_t
        zs.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    p = offset + 4
    for _ in range(m):
        p0 = p
        for _k in range(3):
            (l,) = struct.unpack_from("<H", d, p); p += 2 + l
        p += 4
        (k,) = struct.unpack_from("<H", d, p); p += 2
        for _a in range(k):
            (l,) = struct.unpack_from("<I", d, p); p += 4 + l
        out += d[p0:p]
        c, dl = struct.unpack_from("<II", d, p); p += 8
        raw = zlib.decompress(d[p:p + c - 4]); p += c - 4
        if mode == 0:
            out += struct.pack("<I", len(raw)) + raw
        else:
            cap = zs.ZSTD_compressBound(len(raw))
            buf = ctypes.create_string_buffer(cap)
            got = zs.ZSTD_compress(buf, cap, raw, len(raw), 3)
            out += struct.pack("<II", got + 4, len(raw)) + buf.raw[:got]
    open(dst, "wb").write(bytes(out))


# ---------------------------------------------------------------------------------------- --test dominant / recessive (tests only)
def recode_bed(src_prefix, dst_prefix, test, ref_first=False):
    """Copy a PLINK 1 fileset with every genotype recoded the way the reference recodes it before a dominant
    (2 -> 1) or recessive (1 -> 0, 2 -> 1) test (src/Geno.cpp:2509-2516), counting the effect allele (.bim column 5, or
    column 6 with --ref-first).  An additive run on the copy must give the test columns of `--test <test>` on the
    original."""
    import shutil
    import numpy as np
    raw = np.fromfile(src_prefix + ".bed", dtype=np.uint8)
    two, none = (3, 0) if ref_first else (0, 3)                  # PLINK codes of 2 / 0 copies of the effect allele
    m = [0, 1, 2, 3]
    if test == "dominant":
        m[two] = 2
    else:
        m[two] = 2
        m[2] = none
    lut = np.zeros(256, dtype=np.uint8)
    for b in range(256):
        o = 0
        for k in range(4):
            o |= m[(b >> (2 * k)) & 3] << (2 * k)
        lut[b] = o
    out = raw.copy()
    out[3:] = lut[raw[3:]]
    out.tofile(dst_prefix + ".bed")
    shutil.copy(src_prefix + ".bim", dst_prefix + ".bim")
    shutil.copy(src_prefix + ".fam", dst_prefix + ".fam")


def check_recoded_test(run, read, tmp_path, golden_dir, extra=()):
    """`--test dominant|recessive` == additive test on the recoded fileset for BETA/SE/CHISQ/LOG10P, with A1FREQ and N of
    the additive coding of the original; shared by the CPU (mock ABI) and the GPU driver tests."""
    d = golden_dir
    base = ["--step", "2", "--phenoFile", d + "/phenotype.txt", "--covarFile", d + "/covariates.txt", "--bsize", "100",
            "--ignore-pred", "--minMAC", "1"] + list(extra)
    ref_first = "--ref-first" in extra
    orig = d + "/example_3chr"
    run(base + ["--bed", orig, "--out", str(tmp_path / "add")])
    add = {l.split()[2]: l.split() for l in read(str(tmp_path / "add") + "_Y1.regenie").splitlines()[1:]}
    for test, name in (("dominant", "DOM"), ("recessive", "REC")):
        rec = str(tmp_path / ("rec_" + test))
        recode_bed(orig, rec, test, ref_first)
        run(base + ["--bed", orig, "--test", test, "--out", str(tmp_path / test)])
        run(base + ["--bed", rec, "--out", str(tmp_path / (test + "_ref"))])
        got = [l.split() for l in read(str(tmp_path / test) + "_Y1.regenie").splitlines()[1:]]
        want = {l.split()[2]: l.split() for l in read(str(tmp_path / (test + "_ref")) + "_Y1.regenie").splitlines()[1:]}
        assert len(got) > 300 and [t[2] for t in got] == [k for k in add if k in want]
        for t in got:
            assert t[7] == name and t[:7] == add[t[2]][:7], t             # CHROM..ALLELE1, A1FREQ, N of the additive coding
            assert t[8:] == want[t[2]][8:], (t, want[t[2]])               # BETA SE CHISQ LOG10P EXTRA of the recoded genotypes


def check_na_invariance(run, read, tmp_path, golden_dir, bt):
    """The reference's test/check_na.sh: a single-trait run must not change when the samples whose phenotype is NA are
    deleted from the phenotype and covariate files instead (Step 1 on example.bed, Step 2 on example_3chr.bed)."""
    d = golden_dir
    rows = open(d + "/phenotype_bin_wNA.txt").read().splitlines()
    kept = [l for l in rows if "NA" not in l.split()]
    assert len(kept) < len(rows)
    (tmp_path / "noNA.txt").write_text("\n".join(kept) + "\n")
    ids = {tuple(l.split()[:2]) for l in kept[1:]}
    cov = open(d + "/covariates.txt").read().splitlines()
    (tmp_path / "noNA_covs.txt").write_text("\n".join([cov[0]] + [l for l in cov[1:] if tuple(l.split()[:2]) in ids]) + "\n")
    mode = ["--bt"] if bt else []
    outs = []
    for tag, ph, cv in (("wna", d + "/phenotype_bin_wNA.txt", d + "/covariates.txt"), ("nona", tmp_path / "noNA.txt", tmp_path / "noNA_covs.txt")):
        fit, res = str(tmp_path / ("fit_" + tag)), str(tmp_path / ("test_" + tag))
        run(["--step", "1", "--bed", d + "/example", "--covarFile", cv, "--phenoFile", ph, "--phenoCol", "Y1", "--bsize", "100",
             "--lowmem", "--lowmem-prefix", str(tmp_path / "tmp_rg"), "--out", fit] + mode)
        run(["--step", "2", "--bed", d + "/example_3chr", "--covarFile", cv, "--phenoFile", ph, "--phenoCol", "Y1", "--bsize", "200",
             "--pThresh", "0.01", "--pred", fit + "_pred.list", "--out", res] + mode + (["--firth", "--approx"] if bt else []))
        outs.append((read(fit + "_1.loco"), read(res + "_Y1.regenie")))
    assert len(outs[0][1].splitlines()) > 10
    assert outs[0] == outs[1]


def check_htp(run, read, tmp_path, golden_dir, extra=()):
    """--htp COHORT for quantitative traits (src/Step2_Models.cpp:2400-2426, :2542-2646): same variants and the same AAF as
    the native file, per-trait genotype counts checked against the .bed and the phenotype masks, Info column keys, and
    --no-split is ignored (src/Regenie.cpp:1068-1071).  Shared by the CPU (mock ABI) and GPU driver tests."""
    import numpy as np
    from oracle import plink, prep
    d = golden_dir
    base = ["--step", "2", "--bed", d + "/example_3chr", "--phenoFile", d + "/phenotype.txt", "--covarFile", d + "/covariates.txt",
            "--bsize", "100", "--ignore-pred"] + list(extra)
    run(base + ["--out", str(tmp_path / "native")])
    run(base + ["--htp", "MYCOHORT", "--no-split", "--out", str(tmp_path / "htp")])
    bim = plink.read_bim(d + "/example_3chr.bim")
    keys, _ = plink.read_fam(d + "/example_3chr.fam")
    rf = "--ref-first" in extra
    G = plink.decode_bed(plink.read_bed_rows(d + "/example_3chr.bed", len(keys), bim.offset), len(keys), ref_first=rf)
    pr = prep.prepare(keys, d + "/phenotype.txt", d + "/covariates.txt", step=2)
    idx = {v: k for k, v in enumerate(bim.ids)}
    for ph, nm in enumerate(("Y1", "Y2")):
        nat = [l.split() for l in read(str(tmp_path / "native") + "_%s.regenie" % nm).splitlines()[1:]]
        rows = read(str(tmp_path / "htp") + "_%s.regenie" % nm).splitlines()
        assert rows[0].split("\t") == ["Name", "Chr", "Pos", "Ref", "Alt", "Trait", "Cohort", "Model", "Effect", "LCI_Effect",
                                       "UCI_Effect", "Pval", "AAF", "Num_Cases", "Cases_Ref", "Cases_Het", "Cases_Alt",
                                       "Num_Controls", "Controls_Ref", "Controls_Het", "Controls_Alt", "Info"]
        assert len(rows) - 1 == len(nat) > 400
        m = pr.mask[:, ph].astype(bool)
        for l, n in zip(rows[1:], nat):
            t = l.split("\t")
            assert len(t) == 22
            assert [t[1], t[2], t[0], t[3], t[4]] == n[:5] and t[5:8] == [nm, "MYCOHORT", "ADD-LR"]
            assert t[12] == n[5] and t[13] == n[6]                                   # AAF = A1FREQ, Num_Cases = N
            g = G[idx[t[0]]][m]
            assert [int(x) for x in t[14:17]] == [int((g == 0).sum()), int((g == 1).sum()), int((g == 2).sum())], l
            assert t[17:21] == ["NA"] * 4
            assert [k.split("=")[0] for k in t[21].split(";")] == ["REGENIE_SE", "MAC", "SCORE", "SKATV", "LOG10P"]
            assert float(t[8]) == float(n[8])                                         # Effect = BETA


def check_htp_bt(run, read, tmp_path, golden_dir, extra=(), numbers=True):
    """--htp COHORT for binary traits on hard calls (print_sum_stats_htp, src/Step2_Models.cpp:2542-2646; update_genocounts,
    src/Geno.cpp:2986-3018): same variants and AAF as the native file, genotype counts of the cases and of the controls of
    each trait checked against the .bed and the phenotype file, model string, Info keys; with `numbers` (the real library -
    the mock's statistics are not regenie's) Effect / CI / Pval / REGENIE_BETA / REGENIE_SE / LOG10P against the native
    file of the same options and SCORE^2 / SKATV = the score-test chi-square where no correction was applied."""
    import math
    import numpy as np
    from oracle import plink, prep
    d = golden_dir
    firth = "--firth" in extra
    base = ["--step", "2", "--bed", d + "/example_3chr", "--phenoFile", d + "/phenotype_bin.txt", "--covarFile", d + "/covariates.txt",
            "--bsize", "100", "--ignore-pred", "--bt"] + list(extra)
    run(base + ["--out", str(tmp_path / "native")])
    run(base + ["--htp", "MYCOHORT", "--af-cc", "--out", str(tmp_path / "htp")])      # --af-cc has no HTP columns: ignored
    bim = plink.read_bim(d + "/example_3chr.bim")
    keys, _ = plink.read_fam(d + "/example_3chr.fam")
    G = plink.decode_bed(plink.read_bed_rows(d + "/example_3chr.bed", len(keys), bim.offset), len(keys), ref_first="--ref-first" in extra)
    pr = prep.prepare(keys, d + "/phenotype_bin.txt", d + "/covariates.txt", step=2, bt=True)
    idx = {v: k for k, v in enumerate(bim.ids)}
    model = "ADD" + ("-FIRTH" if firth else "-SPA" if "--spa" in extra else "-LOG")
    zc = 1.959963984540054
    n_rows = 0
    for ph, nm in enumerate(("Y1", "Y2")):
        nat = [l.split() for l in read(str(tmp_path / "native") + "_%s.regenie" % nm).splitlines()[1:]]
        rows = read(str(tmp_path / "htp") + "_%s.regenie" % nm).splitlines()
        assert rows[0].split("\t")[13:21] == ["Num_Cases", "Cases_Ref", "Cases_Het", "Cases_Alt", "Num_Controls", "Controls_Ref",
                                              "Controls_Het", "Controls_Alt"]
        assert len(rows) - 1 == len(nat) > 300
        m = pr.mask[:, ph].astype(bool)
        y = pr.Y_raw[:, ph]
        for l, n in zip(rows[1:], nat):
            t = l.split("\t")
            assert len(t) == 22
            assert [t[1], t[2], t[0], t[3], t[4]] == n[:5] and t[5:8] == [nm, "MYCOHORT", model], l
            assert t[12] == n[5]                                                       # AAF = A1FREQ
            for cols, sel in ((t[13:17], m & (y == 1)), (t[17:21], m & (y == 0))):
                g = G[idx[t[0]]][sel]
                want = [int((g == 0).sum()), int((g == 1).sum()), int((g == 2).sum())]
                assert [int(x) for x in cols] == [sum(want)] + want, l
            info = dict(kv.split("=") for kv in t[21].split(";"))
            failed = n[-1] == "TEST_FAIL"
            keys_want = [] if failed else ["REGENIE_BETA", "REGENIE_SE"] + ([] if firth else ["SE"])
            assert list(info) == keys_want + ["MAC", "SCORE", "SKATV", "LOG10P"], l
            n_rows += 1
            if not numbers or failed:
                continue
            # every number below went through a 6-significant-digit print on both sides: tolerances are a few 1e-5
            beta, se, chisq, lp = (float(x) for x in n[-5:-1])
            assert abs(float(info["REGENIE_BETA"]) - beta) <= 2e-5 * abs(beta) + 1e-12, l
            assert abs(float(info["REGENIE_SE"]) - se) <= 2e-5 * se, l
            assert abs(float(info["LOG10P"]) - lp) <= 2e-5 * lp + 1e-12, l
            if lp > 0:
                assert abs(math.log10(float(t[11])) + lp) < 2e-5 * (1.0 + lp), l       # Pval
            if firth:                                                                  # odds ratio scale
                assert abs(math.log(float(t[8])) - beta) <= 3e-5 * (1.0 + abs(beta)), l
                assert abs(math.log(float(t[9])) - (beta - zc * se)) <= 3e-5 * (1.0 + abs(beta) + zc * se), l
            else:                                                                      # allelic odds ratio from the counts
                c = [int(x) for x in t[14:17]] + [int(x) for x in t[18:21]]
                eff = (2 * c[3] + c[4] + .5) * (2 * c[2] + c[1] + .5) / (2 * c[5] + c[4] + .5) / (2 * c[0] + c[1] + .5)
                assert abs(float(t[8]) - eff) <= 1e-5 * eff, l
                assert abs(float(info["SE"]) - abs(math.log(eff)) / math.sqrt(chisq)) <= 5e-5 * abs(float(info["SE"])) + 1e-12, l
            score, skv = float(info["SCORE"]), float(info["SKATV"])
            z_thr = 1.6448536269514722 if firth else float("inf")                      # --pThresh 0.1: |z| above it is corrected
            if skv > 0 and abs(score) / math.sqrt(skv) <= 0.99 * z_thr:                # no correction: SKATV = denum, SCORE^2 / SKATV = CHISQ
                assert abs(score * score / skv - chisq) <= 1e-4 * chisq + 1e-9, l
                assert (score > 0) == (beta > 0) or beta == 0, l                       # sign: the minor-allele flip is undone like in BETA
    assert n_rows > 600


def check_no_split(run, read, tmp_path, golden_dir, extra=(), bt=False):
    """--no-split (src/Step2_Models.cpp:2364-2383, 2441-2493): one file for all traits whose per-trait columns are those of
    the split files, with N_RR / N_RA / N_AA of all analysed samples (src/Geno.cpp:2480-2486) checked against the .bed."""
    import numpy as np
    from oracle import plink
    d = golden_dir
    pheno = d + ("/phenotype_bin.txt" if bt else "/phenotype.txt")
    base = ["--step", "2", "--bed", d + "/example_3chr", "--phenoFile", pheno, "--covarFile", d + "/covariates.txt", "--bsize", "100",
            "--ignore-pred"] + (["--bt", "--firth", "--approx", "--pThresh", "0.1"] if bt else []) + list(extra)
    run(base + ["--out", str(tmp_path / "split")])
    run(base + ["--no-split", "--out", str(tmp_path / "all")])
    assert read(str(tmp_path / "all") + ".regenie.Ydict").splitlines() == ["Y1 Y1", "Y2 Y2"]
    rows = read(str(tmp_path / "all") + ".regenie").splitlines()
    assert rows[0] == ("CHROM GENPOS ID ALLELE0 ALLELE1 A1FREQ N N_RR N_RA N_AA TEST BETA.Y1 SE.Y1 CHISQ.Y1 LOG10P.Y1 "
                       "BETA.Y2 SE.Y2 CHISQ.Y2 LOG10P.Y2 EXTRA")
    split = [{l.split()[2]: l.split() for l in read(str(tmp_path / "split") + "_%s.regenie" % nm).splitlines()[1:]} for nm in ("Y1", "Y2")]
    bim = plink.read_bim(d + "/example_3chr.bim")
    keys, _ = plink.read_fam(d + "/example_3chr.fam")
    G = plink.decode_bed(plink.read_bed_rows(d + "/example_3chr.bed", len(keys), bim.offset), len(keys), ref_first="--ref-first" in extra)
    idx = {v: k for k, v in enumerate(bim.ids)}
    assert len(rows) > 400
    for l in rows[1:]:
        t = l.split()
        assert len(t) == 20 and t[19] == "NA"
        g = G[idx[t[2]]]
        ok = g != -3
        assert [int(x) for x in t[6:10]] == [int(ok.sum()), int((g[ok] == 0).sum()), int((g[ok] == 1).sum()), int((g[ok] == 2).sum())], t
        for k in range(2):
            s = split[k].get(t[2])
            cols = t[11 + 4 * k: 15 + 4 * k]
            if s is None:
                assert cols == ["NA"] * 4
            else:
                assert t[:6] == s[:6] and t[10] == s[7] and cols == s[8:12], (t, s)
    assert {t.split()[2] for t in rows[1:]} == set(split[0]) | set(split[1])


# ---------------------------------------------------------------------------------------- minimal BGEN v1.2 writer (tests only)
def write_bgen(path, probs, missing, chroms, positions, ids, alleles=("A", "G"), sample_ids=None, level=6):
    """Layout 2, zlib, 8-bit, unphased, biallelic, diploid - the subset rgb200 and the reference's fast parser read.
    probs: u8 [M, N, 2] (P(first-allele homozygote), P(het)) with p0 + p1 <= 255; missing: bool [M, N]."""
    import struct
    import zlib
    import numpy as np
    M, N, _ = probs.shape
    if sample_ids is None:
        sample_ids = ["s%d_s%d" % (i, i) for i in range(N)]
    sblock = b"".join(struct.pack("<H", len(s)) + s.encode() for s in sample_ids)
    sblock = struct.pack("<II", 8 + len(sblock), N) + sblock
    header = struct.pack("<I", 20) + struct.pack("<II", M, N) + b"bgen" + struct.pack("<I", 1 | (2 << 2) | (1 << 31))
    out = [struct.pack("<I", len(header) + len(sblock)), header, sblock]
    for v in range(M):
        vid = ids[v].encode()
        c = str(chroms[v]).encode()
        rec = struct.pack("<H", len(vid)) + vid + struct.pack("<H", len(vid)) + vid + struct.pack("<H", len(c)) + c
        rec += struct.pack("<IH", int(positions[v]), 2)
        for a in alleles:
            rec += struct.pack("<I", len(a)) + a.encode()
        ploidy = np.where(missing[v], 0x82, 0x02).astype(np.uint8)
        pr = np.where(missing[v][:, None], 0, probs[v]).astype(np.uint8)
        raw = struct.pack("<IHBB", N, 2, 2, 2) + ploidy.tobytes() + bytes([0, 8]) + pr.tobytes()
        z = zlib.compress(raw, level)
        rec += struct.pack("<II", len(z) + 4, len(raw)) + z
        out.append(rec)
    with open(path, "wb") as fh:
        fh.write(b"".join(out))


def synthetic_dosage_probs(M, N, seed=0, miss_rate=0.01):
    """Imputed-looking probability pairs: most calls certain, the rest spread, 1 % missing."""
    import numpy as np
    rng = np.random.default_rng(seed)
    maf = rng.uniform(0.02, 0.5, M)
    g = rng.binomial(2, maf[:, None], (M, N))
    p = np.zeros((M, N, 2), dtype=np.uint8)
    p[..., 0] = np.where(g == 2, 255, 0)
    p[..., 1] = np.where(g == 1, 255, 0)
    unsure = rng.random((M, N)) < rng.uniform(0.0, 0.6, M)[:, None]
    a = rng.integers(0, 256, (M, N))
    b = (rng.random((M, N)) * (255 - a)).astype(np.int64)
    p[..., 0] = np.where(unsure, a, p[..., 0])
    p[..., 1] = np.where(unsure, b, p[..., 1])
    return p, rng.random((M, N)) < miss_rate


def check_recoded_test_bgen(run, read, tmp_path, golden_dir, bt=False):
    """--test dominant|recessive on dosages (src/Geno.cpp:2084-2100: P(het) + P(hom) / P(hom)): the test columns equal an
    additive run on a .bgen whose probability pairs were recoded the same way; A1FREQ / INFO / N stay additive."""
    import numpy as np
    d = golden_dir
    keys = ["_".join(l.split()[:2]) for l in open(d + "/example.fam")]
    M, N = 120, len(keys)
    probs, miss = synthetic_dosage_probs(M, N, seed=11)
    chroms, pos, ids = [1] * 60 + [3] * 60, range(1, M + 1), ["v%d" % v for v in range(M)]
    f = str(tmp_path / "orig.bgen")
    write_bgen(f, probs, miss, chroms, pos, ids, sample_ids=keys)
    pheno = d + ("/phenotype_bin.txt" if bt else "/phenotype.txt")
    base = ["--step", "2", "--phenoFile", pheno, "--covarFile", d + "/covariates.txt", "--bsize", "50", "--ignore-pred", "--minMAC", "0"] + \
        (["--bt"] if bt else [])
    run(base + ["--bgen", f, "--out", str(tmp_path / "add")])
    add = {l.split()[2]: l.split() for l in read(str(tmp_path / "add") + "_Y1.regenie").splitlines()[1:]}
    for test, name in (("dominant", "DOM"), ("recessive", "REC")):
        rp = np.zeros_like(probs)
        hom, het = probs[..., 0].astype(np.int64), probs[..., 1].astype(np.int64)
        rp[..., 1] = np.minimum(255, hom + het) if test == "dominant" else hom
        g = str(tmp_path / (test + ".bgen"))
        write_bgen(g, rp, miss, chroms, pos, ids, sample_ids=keys)
        run(base + ["--bgen", f, "--test", test, "--out", str(tmp_path / test)])
        run(base + ["--bgen", g, "--out", str(tmp_path / (test + "_ref"))])
        got = [l.split() for l in read(str(tmp_path / test) + "_Y1.regenie").splitlines()[1:]]
        want = {l.split()[2]: l.split() for l in read(str(tmp_path / (test + "_ref")) + "_Y1.regenie").splitlines()[1:]}
        assert len(got) > 100 and [t[2] for t in got] == [k for k in add if k in want]
        for t in got:
            assert t[8] == name and t[:8] == add[t[2]][:8], t             # ..., A1FREQ, INFO, N of the additive coding
            assert t[9:] == want[t[2]][9:], (t, want[t[2]])


def check_af_cc(run, read, tmp_path, golden_dir, extra=()):
    """--af-cc (src/Geno.cpp:3069-3075, :3120-3127; print_sum_stats_single src/Step2_Models.cpp:2509-2521): allele frequency
    and sample count among cases and controls, checked against the .bed and the phenotype file; all other columns must
    be those of the run without the option."""
    import numpy as np
    from oracle import plink
    d = golden_dir
    base = ["--step", "2", "--bed", d + "/example_3chr", "--phenoFile", d + "/phenotype_bin_wNA.txt", "--covarFile", d + "/covariates.txt",
            "--bsize", "100", "--ignore-pred", "--bt"] + list(extra)
    run(base + ["--out", str(tmp_path / "plain")])
    log = run(base + ["--af-cc", "--out", str(tmp_path / "cc")])
    assert "disabling option --af-cc" not in log
    bim = plink.read_bim(d + "/example_3chr.bim")
    keys, _ = plink.read_fam(d + "/example_3chr.fam")
    G = plink.decode_bed(plink.read_bed_rows(d + "/example_3chr.bed", len(keys), bim.offset), len(keys), ref_first="--ref-first" in extra)
    idx = {v: k for k, v in enumerate(bim.ids)}
    ph = {"_".join(l.split()[:2]): l.split()[2:] for l in open(d + "/phenotype_bin_wNA.txt").read().splitlines()[1:]}
    for j, nm in enumerate(("Y1", "Y2")):
        y = np.array([np.nan if ph[k][j] == "NA" else float(ph[k][j]) for k in keys])
        plain = read(str(tmp_path / "plain") + "_%s.regenie" % nm).splitlines()
        cc = read(str(tmp_path / "cc") + "_%s.regenie" % nm).splitlines()
        assert cc[0] == "CHROM GENPOS ID ALLELE0 ALLELE1 A1FREQ A1FREQ_CASES A1FREQ_CONTROLS N N_CASES N_CONTROLS TEST BETA SE CHISQ LOG10P EXTRA"
        assert len(cc) == len(plain) > 300
        for a, b in zip(plain[1:], cc[1:]):
            t, u = a.split(), b.split()
            assert u[:6] == t[:6] and u[8] == t[6] and u[11:] == t[7:], (a, b)
            g = G[idx[t[2]]]
            ok = (g != -3) & ~np.isnan(y)
            ca, co = ok & (y == 1), ok & (y == 0)
            want = ["%g" % (g[ca].sum() / (2.0 * ca.sum())), "%g" % (g[co].sum() / (2.0 * co.sum())), str(int(ca.sum())), str(int(co.sum()))]
            assert [u[6], u[7], u[9], u[10]] == want, (b, want)


def check_htp_chrx(run, read, tmp_path):
    """--htp on chromosome X, hard calls: on the non-PAR part a male with g >= 1 counts as alt and any other male call as ref,
    females and the PAR variants count as on the autosomes (update_genocounts, src/Geno.cpp:2986-3018; in_non_par :2802-2814)."""
    g = synth.genotypes(240, 120, seed=31, miss=0.03)
    Y, cov, na = synth.phenotypes(g, 2, 2, seed=31)
    prefix = write_fileset(str(tmp_path), g, Y, cov, na, n_chr=1)
    M, N = g.shape
    pos = [1000 + i if i % 2 == 0 else 5_000_000 + i for i in range(M)]               # even: PAR1, odd: non-PAR (default bounds)
    with open(prefix + ".bim", "w") as fh:
        for i in range(M):
            fh.write("23 rs%d 0 %d A G\n" % (i, pos[i]))
    run(["--step", "2", "--bed", prefix, "--phenoFile", str(tmp_path) + "/pheno.txt", "--covarFile", str(tmp_path) + "/covar.txt",
         "--bsize", "50", "--ignore-pred", "--minMAC", "1", "--htp", "CX", "--out", str(tmp_path / "x")])
    keys, _ = plink.read_fam(prefix + ".fam")
    pr = prep.prepare(keys, str(tmp_path) + "/pheno.txt", str(tmp_path) + "/covar.txt", step=2)
    male = np.array([(s % 2) == 0 for s in range(N)])                                  # write_fileset: sex = 1 + s % 2
    n_np = 0
    for ph, nm in enumerate(("Y1", "Y2")):
        rows = read(str(tmp_path / "x") + "_%s.regenie" % nm).splitlines()[1:]
        assert len(rows) > 80
        m = pr.mask[:, ph].astype(bool)
        for l in rows:
            t = l.split("\t")
            i = int(t[0][2:])
            gi = g[i].astype(int)                                                      # codes: 0 / 1 / 2 copies, 3 = missing
            ok = m & (gi != 3)
            if i % 2 == 1:
                alt = int((ok & ~male & (gi == 2)).sum() + (ok & male & (gi >= 1)).sum())
                het = int((ok & ~male & (gi == 1)).sum())
                n_np += 1
            else:
                alt, het = int((ok & (gi == 2)).sum()), int((ok & (gi == 1)).sum())
            assert [int(x) for x in t[13:17]] == [int(ok.sum()), int(ok.sum()) - het - alt, het, alt], l
    assert n_np > 40


def check_htp_bgen_chrx(run, read, tmp_path, golden_dir):
    """--htp on chromosome X dosages: the male rule of update_genocounts on the non-PAR part (dosage >= 1 -> alt, else ref)."""
    from oracle import bgen as obgen, prep
    d = golden_dir
    fam = [l.split() for l in open(d + "/example.fam")]
    keys = ["_".join(t[:2]) for t in fam]
    M, N = 60, len(keys)
    probs, miss = synthetic_dosage_probs(M, N, seed=29)
    f = str(tmp_path / "x.bgen")
    pos = [1000 + i if i % 2 == 0 else 5_000_000 + i for i in range(M)]
    write_bgen(f, probs, miss, [23] * M, pos, ["v%d" % v for v in range(M)], sample_ids=keys)
    male = np.array([(k % 3) == 0 for k in range(N)])
    with open(str(tmp_path / "x.sample"), "w") as fh:
        fh.write("ID_1 ID_2 missing sex\n0 0 0 D\n")
        for k, t in enumerate(fam):
            fh.write("%s %s 0 %d\n" % (t[0], t[1], 1 if male[k] else 2))
    run(["--step", "2", "--bgen", f, "--sample", str(tmp_path / "x.sample"), "--phenoFile", d + "/phenotype.txt", "--covarFile",
         d + "/covariates.txt", "--bsize", "25", "--ignore-pred", "--minMAC", "1", "--htp", "CX", "--out", str(tmp_path / "x")])
    pr = prep.prepare(keys, d + "/phenotype.txt", d + "/covariates.txt", step=2)
    n_np = 0
    for ph, nm in enumerate(("Y1", "Y2")):
        rows = read(str(tmp_path / "x") + "_%s.regenie" % nm).splitlines()[1:]
        assert len(rows) > 40
        m = pr.mask[:, ph].astype(bool)
        for l in rows:
            t = l.split("\t")
            v = int(t[0][1:])
            g, _ = obgen.dosage(probs[v, :, 0], probs[v, :, 1], miss[v])
            ok = m & ~miss[v]
            if v % 2 == 1:
                alt = int((ok & ~male & (g >= 1.5)).sum() + (ok & male & (g >= 1)).sum())
                het = int((ok & ~male & (g >= 0.5) & (g < 1.5)).sum())
                n_np += 1
            else:
                alt, het = int((ok & (g >= 1.5)).sum()), int((ok & (g >= 0.5) & (g < 1.5)).sum())
            assert [int(x) for x in t[13:17]] == [int(ok.sum()), int(ok.sum()) - het - alt, het, alt], l
    assert n_np > 20


def check_htp_bgen(run, read, tmp_path, golden_dir, bt=False):
    """--htp on dosages: the thresholded genotype counts of each trait's samples (cases / controls for a binary trait) against
    oracle.step2.genocounts on the float dosages (update_genocounts, src/Geno.cpp:2986-3018), INFO= in the Info column, same
    variants as the native file.  The driver forms the counts on the host from the inflated bytes (BgenFile::trait_counts)."""
    from oracle import bgen as obgen, prep, step2
    d = golden_dir
    keys = ["_".join(l.split()[:2]) for l in open(d + "/example.fam")]
    M, N = 90, len(keys)
    probs, miss = synthetic_dosage_probs(M, N, seed=23)
    f = str(tmp_path / "syn.bgen")
    write_bgen(f, probs, miss, [1] * 50 + [2] * 40, range(1, M + 1), ["v%d" % v for v in range(M)], sample_ids=keys)
    pheno = d + ("/phenotype_bin.txt" if bt else "/phenotype.txt")
    base = ["--step", "2", "--bgen", f, "--phenoFile", pheno, "--covarFile", d + "/covariates.txt", "--bsize", "40",
            "--ignore-pred", "--minMAC", "1"] + (["--bt"] if bt else [])
    run(base + ["--out", str(tmp_path / "native")])
    run(base + ["--htp", "C1", "--gpu-inflate", "--out", str(tmp_path / "htp")])       # --gpu-inflate falls back to the host here
    pr = prep.prepare(keys, pheno, d + "/covariates.txt", step=2, bt=bt)
    n_rows = 0
    for ph, nm in enumerate(("Y1", "Y2")):
        nat = [l.split() for l in read(str(tmp_path / "native") + "_%s.regenie" % nm).splitlines()[1:]]
        rows = read(str(tmp_path / "htp") + "_%s.regenie" % nm).splitlines()[1:]
        assert len(rows) == len(nat) > 60
        m = pr.mask[:, ph].astype(bool)
        if bt:
            cases, controls = np.nonzero(m & (pr.Y_raw[:, ph] == 1))[0], np.nonzero(m & (pr.Y_raw[:, ph] == 0))[0]
        else:
            cases, controls = np.nonzero(m)[0], None
        for l, n in zip(rows, nat):
            t = l.split("\t")
            assert len(t) == 22 and t[0] == n[2] and t[7] == ("ADD-LOG" if bt else "ADD-LR")
            v = int(t[0][1:])
            g, _ = obgen.dosage(probs[v, :, 0], probs[v, :, 1], miss[v])
            want = step2.genocounts(g, cases, controls)
            assert [int(x) for x in t[14:17]] == want[:3] and int(t[13]) == sum(want[:3]), l
            if bt:
                assert [int(x) for x in t[18:21]] == want[3:] and int(t[17]) == sum(want[3:]), l
            else:
                assert t[17:21] == ["NA"] * 4
            info = dict(kv.split("=") for kv in t[21].split(";"))
            assert list(info) == (["REGENIE_BETA", "REGENIE_SE", "SE"] if bt else ["REGENIE_SE"]) + ["INFO", "MAC", "SCORE", "SKATV", "LOG10P"], l
            assert abs(float(info["INFO"]) - float(n[6])) <= 2e-6 * max(1.0, abs(float(n[6]))), l     # the trait's INFO column
            n_rows += 1
    assert n_rows > 120


def check_no_split_bgen(run, read, tmp_path, golden_dir):
    """--no-split on dosages: INFO over all analysed samples and the threshold genotype counts (dosage < 0.5 / >= 1.5,
    src/Geno.cpp:2048-2050) come from the inflated bytes; per-trait columns are those of the split files."""
    import numpy as np
    from oracle import bgen as obgen
    d = golden_dir
    keys = ["_".join(l.split()[:2]) for l in open(d + "/example.fam")]
    M, N = 90, len(keys)
    probs, miss = synthetic_dosage_probs(M, N, seed=21)
    f = str(tmp_path / "syn.bgen")
    write_bgen(f, probs, miss, [1] * 50 + [2] * 40, range(1, M + 1), ["v%d" % v for v in range(M)], sample_ids=keys)
    base = ["--step", "2", "--bgen", f, "--phenoFile", d + "/phenotype.txt", "--covarFile", d + "/covariates.txt", "--bsize", "40",
            "--ignore-pred", "--minMAC", "1"]
    run(base + ["--out", str(tmp_path / "split")])
    run(base + ["--no-split", "--gpu-inflate", "--out", str(tmp_path / "all")])
    rows = read(str(tmp_path / "all") + ".regenie").splitlines()
    assert rows[0].split()[:12] == "CHROM GENPOS ID ALLELE0 ALLELE1 A1FREQ INFO N N_RR N_RA N_AA TEST".split()
    split = [{l.split()[2]: l.split() for l in read(str(tmp_path / "split") + "_%s.regenie" % nm).splitlines()[1:]} for nm in ("Y1", "Y2")]
    assert len(rows) > 60
    for l in rows[1:]:
        t = l.split()
        v = int(t[2][1:])
        g, ival = obgen.dosage(probs[v, :, 0], probs[v, :, 1], miss[v])
        ok = ~miss[v]
        af = g[ok].sum() / (2 * ok.sum())
        info = 1 - ival[ok].sum() / (2 * ok.sum() * af * (1 - af))
        dd = probs[v, ok, 1].astype(int) + 2 * probs[v, ok, 0].astype(int)
        n_aa, n_rr = int((2 * dd >= 765).sum()), int((2 * dd < 255).sum())
        assert [int(x) for x in t[7:11]] == [int(ok.sum()), n_rr, int(ok.sum()) - n_rr - n_aa, n_aa], t
        assert abs(float(t[6]) - info) <= 2e-6 * max(1.0, abs(info)) and t[11] == "ADD"
        for k in range(2):
            s = split[k].get(t[2])
            cols = t[12 + 4 * k: 16 + 4 * k]
            assert cols == (["NA"] * 4 if s is None else s[9:13]), (t, s)


# ------------------------------------------------------------------- stored outputs of the compiled reference libraries
REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")


def ref_golden(name, compute):
    """What a library of oracle/_ref/ (compiled from the reference's sources by oracle/build_native.py) returned for a
    test's inputs, stored as tests/golden/ref/<name>.npz: the comparison then needs neither the library nor the reference's
    sources.  With RG_WRITE_REF_GOLDEN=1 in the environment, `compute()` runs the library and the file is rewritten."""
    path = os.path.join(REF_GOLDEN, name + ".npz")
    if os.environ.get("RG_WRITE_REF_GOLDEN") == "1":
        os.makedirs(REF_GOLDEN, exist_ok=True)
        np.savez_compressed(path, **compute())
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def sha256(a):
    """Digest of an exact (integer) result, stored in place of arrays too large to keep."""
    import hashlib
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def W_digest(W, n_rows=64, seed=0):
    """Level-0 predictors [P][N x R] too large to store whole: a fixed, seeded set of rows and every column's max |W|."""
    rows = np.sort(np.random.default_rng(seed).choice(W[0].shape[0], min(W[0].shape[0], n_rows), replace=False))
    return {"rows": rows, "W": np.stack([w[rows] for w in W]), "absmax": np.stack([np.abs(w).max(axis=0) for w in W])}


def W_rel_err(W, ref, prefix=""):
    """max over phenotypes of |W - W_ref| / max |W_ref| on the stored rows and of the columns' max |W| against the stored
    ones: both are bounded by the error over the whole matrix."""
    err = 0.0
    for p, w in enumerate(W):
        scale = ref[prefix + "absmax"][p].max()
        err = max(err, np.abs(w[ref[prefix + "rows"]] - ref[prefix + "W"][p]).max() / scale,
                  np.abs(np.abs(w).max(axis=0) - ref[prefix + "absmax"][p]).max() / scale)
    return float(err)
