"""k_auto / k_lz allele draws and forced minors (GPU, -m gpu).

The draw keeps every 32-slot group in registers: the residual Philox calls work on whichever group is rotated into
slot 0, and forced minors are OR-ed in through per-word selects.  These rows are built to reach those paths: forced
minors in each of the four mask words of a span, on the last cells of rows and segments, many of them in one span,
thresholds next to 0 and next to 2^32 - 1, and sample counts whose last span is partial.  The text must be the
oracle's (oracle.rows_from_flat) at -z 2 (k_auto) and -z 6 (k_lz), and every BGZF block must inflate with a valid
CRC32 and ISIZE (oracle.bgzf_decompress checks both)."""
import numpy as np
import pytest

from tests.cases import Sample, Snp

pytestmark = pytest.mark.gpu

# reference-allele probabilities: thresholds next to 0 and next to 2^32 - 1 leave lanes undecided longest there
EDGE_P = [2.0 ** -32, 3 * 2.0 ** -32, 1e-6, 0.5, 1 - 1e-6, 1 - 3 * 2.0 ** -32, 1 - 2.0 ** -32]


def make_case(n, seed):
    """Biallelic autosome rows of n samples; every sample is a case, so that any cell can carry a forced minor."""
    rs = np.random.RandomState(seed)
    rows = []   # (reference-allele probability, forced-minor samples)
    every = np.arange(n)
    rows.append((0.3, every[every % 16 == 5]))                   # one forced cell in every 32-bit word of every span
    rows.append((0.7, every[every % 16 == 14]))
    rows.append((0.9, np.array([n - 1])))                        # the last cell of the row (a partial last span)
    rows.append((0.2, np.array([n - 2, n - 1])))
    rows.append((0.6, every[every % 2 == 0]))                    # together: the last cell of every segment
    rows.append((0.6, every[every % 2 == 1]))
    rows.append((0.95, every[:200]))                             # many forced minors in one span, and in the next
    rows.append((0.5, every[(every >= 64) & (every < 128)]))     # one whole span
    for p in EDGE_P:
        rows.append((p, np.array([], dtype=np.int64)))
        rows.append((p, rs.choice(n, size=9, replace=False)))
    for _ in range(6):
        rows.append(((1 + rs.randint(99)) * 0.005, rs.choice(n, size=rs.randint(0, 40), replace=False)))
    snps, forced = [], [dict() for _ in range(n)]
    for r, (p, who) in enumerate(rows):
        snp_id = r + 1
        snps.append(Snp(id=snp_id, chromosome="1" if r % 2 == 0 else "2", position=1000 + 10 * r,
                        tuples=[("A", p), ("G", 1.0)]))
        for i in who:
            forced[int(i)][snp_id] = 0.5
    snps.sort(key=lambda s: (s.chromosome, s.position))
    samples = [Sample(family_id=i + 1, person_id=500001 + i, father_id=0, mother_id=0, sex=1 + (i % 3 == 0),
                      is_control=False, deleterious_snps=forced[i]) for i in range(n)]
    return samples, snps


@pytest.fixture(scope="module")
def oracle_mod():
    from oracle import oracle
    oracle.build()
    return oracle


@pytest.mark.parametrize("n", [20001, 4097, 4160])
def test_auto_draw_matches_oracle(n, oracle_mod):
    from dna_factory_b200 import _native, host
    seed = 0xA5D0 + n
    samples, snps = make_case(n, seed=n)
    flat = oracle_mod.flatten(samples, snps)
    assert len(flat["over_row"]) > n, "the rows must carry forced minors"
    want = oracle_mod.rows_from_flat(flat, seed)[0].tobytes()
    with _native.Engine(0) as eng:
        host.configure(eng, samples, snps)
        for level in (2, 6):
            blob, st = eng.generate(0, len(snps), seed, level=level)
            text, blocks, _ = oracle_mod.bgzf_decompress(blob)   # raises on a bad CRC32 or ISIZE
            assert blocks == st["bgzf_blocks"]
            assert text == want, "-z %d, n = %d: text differs from the oracle" % (level, n)
