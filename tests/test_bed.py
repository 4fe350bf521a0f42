"""PLINK 1 fileset (--bed): population.bed rows from k_bed (dnaf_generate_bed*) and population.bim from
SnpTable.bim_bytes().

The .bed bytes are checked with a numpy decoder written from the published format (np.unpackbits on the bytes, a
lookup of the four 2-bit values), not with the kernel's bit tricks, against genotypes parsed from the reference's own
row text and against the independent three-kernel export (dnaf_genotypes)."""
import gzip
import json
import os
import random

import numpy as np
import pytest

from tests.cases import GOLDEN, ROW_CASES, Snp, load_case, synth_case

MISSING = -1
# 2-bit value -> ALT copies (A1 = ALT, A2 = REF): 00 -> 2, 01 -> missing, 10 -> 1, 11 -> 0
_COPIES = np.array([2, MISSING, 1, 0], np.int8)


def decode_bed(data, n, rows, magic=True):
    """.bed bytes -> (ALT copies int8[rows, n] with -1 = missing, padding bits of every row's last byte)."""
    data = bytes(data)
    if magic:
        assert data[:3] == b"\x6c\x1b\x01"
        data = data[3:]
    pitch = (n + 3) // 4
    assert len(data) == rows * pitch
    bits = np.unpackbits(np.frombuffer(data, np.uint8).reshape(rows, pitch), axis=1, bitorder="little")
    val = bits[:, 0::2].astype(np.int64) | (bits[:, 1::2].astype(np.int64) << 1)    # [rows, 4 * pitch]
    return _COPIES[val[:, :n]], val[:, n:]


def copies_from_text(text, n):
    """ALT copies of every cell of VCF rows (biallelic): '.' -> missing, haploid 'a' -> 2a, 'a/b' -> a + b."""
    lines = text.split(b"\n")[:-1]
    out = np.zeros((len(lines), n), np.int8)
    for r, line in enumerate(lines):
        cells = line.split(b"\t")[9:] if n else []
        assert len(cells) == n
        for i, c in enumerate(cells):
            if c == b".":
                out[r, i] = MISSING
            elif len(c) == 1:
                out[r, i] = 2 * int(c)
            else:
                out[r, i] = int(c[:1]) + int(c[2:3])
    return out


def copies_from_genotypes(g):
    """The same from dnaf_genotypes' [rows][n][2] allele indices (0xFF = no such allele)."""
    g = g.astype(np.int16)
    hap = (g[..., 1] == 0xFF) & (g[..., 0] != 0xFF)
    out = np.where(hap, 2 * g[..., 0], g[..., 0] + g[..., 1]).astype(np.int8)
    out[g[..., 0] == 0xFF] = MISSING
    return out


def bim_python(table):
    lines = []
    for r in range(len(table)):
        k = int(table.n_alleles[r])
        lines.append("%s\trs%d\t0\t%d\t%s\t%s\n" % (table.chrom_labels[table.chrom_idx[r]], table.ids[r], table.position[r],
                                                   chr(table.nts[r, 1]) if k == 2 else "0", chr(table.nts[r, 0])))
    return "".join(lines).encode()


def _golden_table():
    from dna_factory_b200.snp import SNPTuples, SnpTable
    with open(os.path.join(GOLDEN, "cli_small", "snps.json")) as f:
        return SnpTable.from_snps([SNPTuples.from_json(line) for line in f])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bim_bytes_matches_per_line_rendering():
    from dna_factory_b200.snp import SnpTable
    labels = ["1", "22", "X", "Y", "MT", "10"]
    rs = np.random.RandomState(3)
    S = 300
    k = np.where(rs.rand(S) < 0.2, 1, 2).astype(np.uint8)
    nts = np.zeros((S, 4), np.uint8)
    nts[:, 0] = rs.choice(np.frombuffer(b"ACGT", np.uint8), S)
    nts[:, 1] = np.where(k == 2, rs.choice(np.frombuffer(b"ACGT", np.uint8), S), 0)
    cum = np.full((S, 4), 2.0)
    cum[:, 0] = np.where(k == 1, 1.0, 0.9)
    cum[:, 1] = 1.0
    pos = rs.randint(0, 250_000_000, S)
    pos[:3] = [0, 9, 10]
    ids = rs.randint(1, 10 ** 9, S)
    ids[:2] = [1, 1_000_000_000_000]
    t = SnpTable(ids, rs.randint(0, len(labels), S), labels, pos, k, nts, cum)
    assert (t.n_alleles == 1).any()
    assert t.bim_bytes() == bim_python(t)
    assert SnpTable([], [], labels, [], [], np.zeros((0, 4)), np.zeros((0, 4))).bim_bytes() == b""


def test_bim_bytes_of_the_golden_snps():
    t = _golden_table()
    assert len(t) == 400
    got = t.bim_bytes()
    assert got == bim_python(t)
    first = got.split(b"\n")[0].split(b"\t")
    assert first == [b"1", b"rs329", b"0", b"1798996", b"A", b"T"]   # snps.json line 1: {"T": 0.98, "A": 1.0}


def test_bim_bytes_refuses_multiallelic_rows():
    from dna_factory_b200.snp import SnpTable
    t = SnpTable([5], [0], ["1"], [10], [3], [[65, 67, 71, 0]], [[0.5, 0.8, 1.0, 2.0]])
    with pytest.raises(ValueError, match="alleles"):
        t.bim_bytes()


def test_bed_flag_parses():
    from dna_factory_b200 import pop_factory
    base = ["-s", "3", "-c", "4"]
    assert pop_factory.parse_cmd_args(base + ["--bed"]).bed is True
    assert pop_factory.parse_cmd_args(base).bed is False


def test_bed_with_a_multiallelic_snp_fails_before_the_vcf(tmp_path):
    from dna_factory_b200 import pop_factory
    with open(os.path.join(GOLDEN, "cli_small", "snps.json"), "rb") as f:
        lines = f.read().splitlines(keepends=True)
    lines.insert(5, b'{"id": 9001, "chromosome": "1", "position": 7000000, "tuples": {"A": 0.5, "C": 0.8, "G": 1.0}}\n')
    snps_gz = tmp_path / "snps_in.json.gz"
    with gzip.open(snps_gz, "wb") as g:
        g.write(b"".join(lines))
    out = tmp_path / "out"
    random.seed(1)
    with pytest.raises(ValueError, match="rs9001"):
        pop_factory.main(["-s", "5", "-c", "4", "--snps_file", str(snps_gz), "-p",
                          os.path.join(GOLDEN, "cli_small", "deleterious_config.yml"), "--outdir", str(out), "--seed", "7",
                          "--bed"])
    assert not (out / "population.vcf.gz").exists()
    assert not (out / "population.bed").exists()


def test_decoder_round_trips_a_hand_built_fileset():
    # 5 samples, 2 rows: ALT copies per cell, and the bytes the format spells out for them (sample i in byte i // 4,
    # bits 2(i % 4) and 2(i % 4) + 1; values 2 -> 00, missing -> 01, 1 -> 10, 0 -> 11; padding bits 0)
    copies = np.array([[2, 1, 0, MISSING, 2], [0, 0, 1, MISSING, 1]], np.int8)
    data = b"\x6c\x1b\x01" + bytes([0b01111000, 0b00000000, 0b01101111, 0b00000010])
    got, pad = decode_bed(data, 5, 2)
    assert np.array_equal(got, copies)
    assert not pad.any()
    got, pad = decode_bed(b"\x6c\x1b\x01" + bytes([0b01111000, 0b11000000, 0b01101111, 0b00000010]), 5, 2)
    assert np.array_equal(got, copies) and pad[0].tolist() == [0, 0, 3] and not pad[1].any()
    # whole bytes, no padding
    got, pad = decode_bed(bytes([0xE4]), 4, 1, magic=False)
    assert got.tolist() == [[2, MISSING, 1, 0]] and pad.shape == (1, 0)


# ------------------------------------------------------------------------------------------------------------- GPU
def _engine(case, chunk=None):
    from dna_factory_b200 import _native, host
    eng = _native.Engine(0)
    host.configure(eng, case.samples, case.snps)
    eng.set_row_base(case.row_begin)
    if chunk:
        eng.set_chunk_bytes(chunk)
    return eng


def _runs(ks):
    """Maximal runs [a, b) of rows with at most 2 alleles."""
    runs, a = [], None
    for r, k in enumerate(list(ks) + [9]):
        if k <= 2 and a is None:
            a = r
        elif k > 2 and a is not None:
            runs.append((a, r))
            a = None
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("name", ROW_CASES)
def test_bed_matches_the_reference_golden_rows(name):
    """X, Y and MT for both sexes, forced minors, u on a threshold, K = 1 rows, a row counter above 2^32, N = 0."""
    case = load_case(name)
    n = len(case.samples)
    lines = case.text.split(b"\n")[:-1]
    eng = _engine(case)
    runs = _runs([len(s.tuples) for s in case.snps])
    assert runs
    for a, b in runs:
        data, st = eng.generate_bed(a, b, case.seed)
        assert st["rows"] == b - a and st["calls"] == (b - a) * n
        got, pad = decode_bed(data, n, b - a, magic=False)
        assert not pad.any()
        want = copies_from_text(b"".join(ln + b"\n" for ln in lines[a:b]), n)
        assert np.array_equal(got, want), (name, a, b)


def _dense_case(n, seed):
    """A synthetic population with all four classes, K = 1 rows, and rare rows that carry overrides on most cases."""
    case = synth_case(n, 24, seed=seed, chroms=["1", "2", "X", "Y", "MT", "22"], n_del=6)
    rare = sorted(case.snps, key=lambda s: -s.tuples[0][1])[:3]
    case.snps.append(Snp(id=10_001, chromosome="7", position=5, tuples=[("G", 1.0)]))
    case.snps.append(Snp(id=10_002, chromosome="Y", position=6, tuples=[("A", 0.995), ("C", 1.0)]))
    case.snps.sort(key=lambda x: (x.chromosome, x.position))
    for i, smp in enumerate(case.samples):
        if not smp.is_control and i % 3 != 0:
            for s in rare + case.snps[-2:]:
                smp.deleterious_snps[s.id] = 0.5
    return case


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 4, 15, 16, 17, 4097, 20000, 100003])
def test_bed_matches_the_genotype_export(n):
    """k_bed against the three-kernel export (k_sample -> k_overrides -> k_export_genotypes) with the ploidy rules
    applied, at pitches that are and are not a multiple of 4 and with a partial last 16-sample group; a 4 KiB chunk
    makes every call many passes."""
    case = _dense_case(n, seed=n)
    S = len(case.snps)
    eng = _engine(case, chunk=4096)
    want = copies_from_genotypes(eng.genotypes(0, S, case.seed))
    data, st = eng.generate_bed(0, S, case.seed)
    got, pad = decode_bed(data, n, S, magic=False)
    assert np.array_equal(got, want)
    assert not pad.any()
    assert st["kernel_launches"] == -(-S // max(1, 4096 // ((n + 3) // 4)))
    assert st["ms_sample"] > 0 and st["ms_total"] >= st["ms_sample"]
    assert (st["bgzf_bytes"], st["bgzf_blocks"], st["text_bytes"]) == (0, 0, 0)


@pytest.mark.gpu
def test_bed_ranges_files_and_repeats(tmp_path):
    """Row ranges concatenate byte for byte, two contexts writing halves with pwrite give the one-call file, repeated
    calls are identical, and the device-only call reports what the host call reports."""
    from dna_factory_b200 import _native, host
    case = _dense_case(2500, seed=11)
    S = len(case.snps)
    eng = _engine(case, chunk=8192)
    whole, st = eng.generate_bed(0, S, case.seed)
    assert eng.generate_bed(0, S, case.seed)[0] == whole
    cut = [0, 1, 7, 7, S // 2, S - 1, S]
    assert b"".join(eng.generate_bed(a, b, case.seed)[0] for a, b in zip(cut, cut[1:])) == whole
    dev = eng.generate_bed_device(0, S, case.seed)
    assert {k: dev[k] for k in ("rows", "calls", "kernel_launches")} == {k: st[k] for k in ("rows", "calls", "kernel_launches")}
    pitch = eng.bed_pitch()
    path = tmp_path / "population.bed"
    fd = os.open(str(path), os.O_RDWR | os.O_CREAT | os.O_TRUNC, 0o644)
    try:
        os.write(fd, b"\x6c\x1b\x01")
        mid = S // 2
        rows, samples = host.override_pairs(case.samples, case.snps)
        for lo, hi in ((mid, S), (0, mid)):     # second half first: offsets, not the order of the writes, place rows
            with _native.Engine(0) as e:
                sex, ctl = host.flatten_samples(case.samples)
                e.set_samples(sex, ctl)
                e.set_snps(**host.slice_snps(host.flatten_snps(case.snps), lo, hi))
                e.set_overrides(*host.slice_overrides(rows, samples, lo, hi))
                e.set_row_base(lo)
                e.generate_bed_fd_at(0, hi - lo, case.seed, fd, 3 + lo * pitch)
    finally:
        os.close(fd)
    assert path.read_bytes() == b"\x6c\x1b\x01" + whole
    eng.close()


@pytest.mark.gpu
def test_bed_refuses_multiallelic_rows_before_any_work(tmp_path):
    from dna_factory_b200 import _native
    case = synth_case(40, 20, seed=5, exotic=True)    # rows with 3 and 4 alleles among biallelic ones
    eng = _engine(case)
    k = [len(s.tuples) for s in case.snps]
    bad = next(r for r, kr in enumerate(k) if kr > 2)
    out = np.full(20 * 10, 0xAB, np.uint8)
    with pytest.raises(_native.DnafError) as e:
        eng.generate_bed_into(0, 20, case.seed, out)
    assert e.value.code == _native.E_INPUT and ("row %d " % bad) in str(e.value)
    assert (out == 0xAB).all()
    path = tmp_path / "x.bed"
    fd = os.open(str(path), os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
    try:
        with pytest.raises(_native.DnafError):
            eng.generate_bed_fd_at(0, 20, case.seed, fd, 3)
    finally:
        os.close(fd)
    assert path.read_bytes() == b""
    a, b = _runs(k)[0]
    assert len(eng.generate_bed(a, b, case.seed)[0]) == (b - a) * 10    # the context is still usable
    eng.close()


def _cli(tmp_path, monkeypatch, out, extra):
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    meta = json.load(open(os.path.join(gold, "meta.json")))

    class FixedDatetime(pop_factory.datetime):
        @classmethod
        def now(cls, tz=None):
            return cls(2026, 1, 1, 12, 34, 56)

    monkeypatch.setattr(pop_factory, "datetime", FixedDatetime)
    random.seed(meta["python_random_seed"])
    pop_factory.main(meta["args"] + ["-p", os.path.join(gold, "deleterious_config.yml"), "--outdir", str(out),
                                     "--seed", str(meta["philox_seed"]), "--bed"] + extra)
    return gold, meta


@pytest.mark.gpu
def test_cli_bed_fileset(tmp_path, monkeypatch):
    """--bed on the pinned reference CLI run: the VCF and .fam stay the golden ones, the .bed decodes to the GTs of
    the decompressed VCF, the .bim lists the same rows, and --gpus 2 writes the same .bed and .bim."""
    import hashlib
    gold, meta = _cli(tmp_path, monkeypatch, tmp_path / "g1", [])
    out = tmp_path / "g1"
    vcf = gzip.decompress((out / "population.vcf.gz").read_bytes())
    assert hashlib.sha256(vcf).hexdigest() == meta["vcf_sha256"]
    assert (out / "population.fam").read_bytes() == open(os.path.join(gold, "population.fam"), "rb").read()
    fam = (out / "population.fam").read_text().splitlines()
    body = b"".join(ln + b"\n" for ln in vcf.split(b"\n")[:-1] if not ln.startswith(b"#"))
    n = len(fam)
    got, pad = decode_bed((out / "population.bed").read_bytes(), n, body.count(b"\n"))
    assert np.array_equal(got, copies_from_text(body, n)) and not pad.any()
    bim = (out / "population.bim").read_bytes()
    assert bim == _golden_table().bim_bytes()
    assert [ln.split(b"\t")[:3] for ln in body.splitlines()] == \
        [[f[0], f[3], f[1]] for f in (ln.split(b"\t") for ln in bim.splitlines())]
    _cli(tmp_path, monkeypatch, tmp_path / "g2", ["--gpus", "2"])
    for name in ("population.bed", "population.bim", "population.fam"):
        assert (tmp_path / "g2" / name).read_bytes() == (out / name).read_bytes(), name
