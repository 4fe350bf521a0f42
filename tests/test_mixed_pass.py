"""Mixed passes (GPU, -m gpu): a pass that opens with a run of autosome rows and ends with other rows (MT, X, Y, as
every sorted window does) runs the autosome run through k_auto's implicit descriptors and plans only the rest.  The
BGZF stream must be byte for byte the one of full planning (DNAF_FULL_PLAN=1, read once per process, hence the
child processes) and must inflate to the oracle's rows; a K = 3 row inside the autosome run keeps full planning."""
import json
import os
import re
import subprocess
import sys

import pytest

from tests.cases import synth_case

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AUTOSOMES = ["1", "2", "7", "12", "22"]
PASS_RE = re.compile(r"\[dnaf\] pass rows (\d+) implicit (\d+) ")
CASES = {"tail": (1500, 120, 5), "tail_two_segments": (17000, 48, 6), "k3_middle": (1500, 120, 7)}


def make_case(name):
    """Autosome rows, then MT / X / Y rows; 'k3_middle' turns one autosome row in the middle of the run into K = 3."""
    n, s, seed = CASES[name]
    case = synth_case(n, s, seed=seed, chroms=AUTOSOMES + ["MT", "X", "Y"])
    rx = first_other_row(case)
    assert 8 < rx < s - 8, "the seed must give an autosome run and a tail of other rows"
    if name == "k3_middle":
        case.snps[rx // 2].tuples = [("A", 0.55), ("C", 0.8), ("G", 1.0)]
    return case


def first_other_row(case):
    return next(i for i, snp in enumerate(case.snps) if snp.chromosome not in AUTOSOMES)


def scenarios(name, row_off):
    """(label, chunk bytes) with DNAF_RAMP=0, every pass one chunk: the autosome/other boundary rx in the middle of
    the single pass, one autosome row opening the second pass, one other row closing the first pass."""
    rx = first_other_row(make_case(name))
    out = [("middle", 256 << 20)]
    if name != "k3_middle":
        out += [("start", int(row_off[rx - 1])), ("end", int(row_off[rx + 1]))]
    return out


def child(name, scen, out_dir):
    """Runs in a child process: every scenario at -z 2 and -z 6, blobs to out_dir, pass lines on stderr."""
    from dna_factory_b200 import _native, host
    case = make_case(name)
    for label, chunk in scen:
        for level in (2, 6):
            with _native.Engine(0) as eng:
                host.configure(eng, case.samples, case.snps)
                eng.set_chunk_bytes(chunk)
                sys.stderr.write("[run] %s %d\n" % (label, level))
                sys.stderr.flush()
                blob, _ = eng.generate(0, len(case.snps), case.seed, level=level)
                sys.stderr.flush()
            with open(os.path.join(out_dir, "%s_z%d.bgzf" % (label, level)), "wb") as f:
                f.write(blob)


def run_child(name, scen, out_dir, full_plan):
    env = dict(os.environ, DNAF_RAMP="0", DNAF_TRACE="1")
    env.pop("DNAF_FULL_PLAN", None)
    if full_plan:
        env["DNAF_FULL_PLAN"] = "1"
    os.makedirs(out_dir, exist_ok=True)
    code = "import sys, json; sys.path.insert(0, %r); from tests.test_mixed_pass import child; child(%r, json.loads(%r), %r)" % (
        ROOT, name, json.dumps(scen), out_dir)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    passes, cur = {}, None
    for line in r.stderr.splitlines():
        if line.startswith("[run] "):
            label, level = line[6:].split()
            cur = passes.setdefault((label, int(level)), [])
        m = PASS_RE.search(line)
        if m and cur is not None:
            cur.append((int(m.group(1)), int(m.group(2))))
    blobs = {}
    for label, _ in scen:
        for level in (2, 6):
            with open(os.path.join(out_dir, "%s_z%d.bgzf" % (label, level)), "rb") as f:
                blobs[(label, level)] = f.read()
    return blobs, passes


@pytest.mark.parametrize("name", sorted(CASES))
def test_mixed_pass_stream_equals_full_planning(name, tmp_path):
    from oracle import oracle
    case = make_case(name)
    want, row_off = oracle.rows(case.samples, case.snps, case.seed, case.row_begin)
    scen = scenarios(name, row_off)
    new, new_passes = run_child(name, scen, str(tmp_path / "new"), full_plan=False)
    ref, ref_passes = run_child(name, scen, str(tmp_path / "full"), full_plan=True)
    rx = first_other_row(case)
    for label, _ in scen:
        for level in (2, 6):
            key = (label, level)
            assert new[key] == ref[key], "%s -z %d: the stream differs from full planning" % (label, level)
            assert oracle.bgzf_decompress(new[key])[0] == want, "%s -z %d: the text differs from the oracle" % (label, level)
            split = [(rows, imp) for rows, imp in new_passes[key] if 0 < imp < rows]
            assert not [p for p in ref_passes[key] if 0 < p[1] < p[0]], "DNAF_FULL_PLAN still split a pass"
            if name == "k3_middle":
                assert not split, "a pass with k_auto rows after its first other row must be planned whole"
            else:
                # the pass holding the boundary runs exactly the autosome rows before rx implicitly
                assert len(split) == 1, new_passes[key]
                rows, imp = split[0]
                expect = {"middle": (len(case.snps), rx), "start": (len(case.snps) - rx + 1, 1), "end": (rx + 1, rx)}[label]
                assert (rows, imp) == expect, (label, new_passes[key])
