"""CLI-level parity: `Ahsoka phase -g G -a A -o P -t 1` output text.

The committed tests/golden/*.ref-result.txt files were written by oracle/_ref/Ahsoka_ref — the
reference's src/*.cpp compiled VERBATIM (polyassembly.cpp, alignmentstoreadset.cpp,
chainstoreadset.cpp, graph.cpp, alignmentreader.cpp, argumentparser.cpp) against the WhatsHap
API shim of oracle/whatshap_shim — by tests/golden/make_golden.py.  They pin every
Ahsoka-owned stage (projection, filter, ordering, coverage, consensus, re-packing, emission and
the text format of README.md:28-42) to the reference text itself.

  * not gpu: host drop-in (flatten + emission) with the CPU oracle behind the C ABI
             (oracle/_ref/Ahsoka_flat_oracle, or oracle/_ref/Ahsoka_flat_oracle_standalone when the
             original's sources were not given at build time) must reproduce those files byte for byte;
  * gpu:     the same drop-in with the CUDA library behind the C ABI (ahsoka_b200/bin/Ahsoka_b200).
Neither test reads the original sources at run time (the binaries are built from them once, with AHSOKA_REFERENCE set).
"""
import json
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
# the drop-in with the CPU oracle behind the C ABI: linked with the original's host stages if built with AHSOKA_REFERENCE
FLAT_ORACLE = next((p for p in (os.path.join(REF_DIR, "Ahsoka_flat_oracle"), os.path.join(REF_DIR, "Ahsoka_flat_oracle_standalone"))
                    if os.path.exists(p)), None)
B200_CLI = os.path.join(ROOT, "ahsoka_b200", "bin", "Ahsoka_b200")

CASES = [c for c in json.load(open(os.path.join(GOLDEN, "index.json")))["cases"] if "ref_result" in c]


def _run_cli(exe, case, td, env=None):
    out = os.path.join(td, "out")
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([exe, "phase", "-g", os.path.join(GOLDEN, case["gfa"]), "-a", os.path.join(td, "reads.gaf"), "-o", out, "-t", "1"],
                       cwd=td, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=e, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return open(out + "-result.txt").read(), r.stdout


def _stage(case, td):
    # the reader writes <gaf stem>-alignment_identities.txt next to the GAF (alignmentreader.cpp:74-75): use a copy
    with open(os.path.join(GOLDEN, case["gaf"])) as f, open(os.path.join(td, "reads.gaf"), "w") as g:
        g.write(f.read())


def _hap_lines(stdout):
    # "hap:" blocks of alignmentstoreadset.cpp:479-486
    lines = stdout.split("\n")
    return [lines[i + 1] for i, l in enumerate(lines) if l.startswith("hap:") and i + 1 < len(lines)]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_flat_oracle_cli_matches_reference_verbatim(case):
    exe = FLAT_ORACLE
    if exe is None:
        pytest.skip("oracle/_ref/Ahsoka_flat_oracle_standalone not built")
    want = open(os.path.join(GOLDEN, case["ref_result"])).read()
    with tempfile.TemporaryDirectory() as td:
        _stage(case, td)
        got, _ = _run_cli(exe, case, td)
    assert got == want


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_reference_verbatim_binary_still_reproduces_golden(case):
    exe = os.path.join(REF_DIR, "Ahsoka_ref")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/Ahsoka_ref not built (needs the original Ahsoka sources at build time: AHSOKA_REFERENCE)")
    want = open(os.path.join(GOLDEN, case["ref_result"])).read()
    with tempfile.TemporaryDirectory() as td:
        _stage(case, td)
        got, _ = _run_cli(exe, case, td)
    assert got == want


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_b200_cli_matches_reference_verbatim(case):
    exe = B200_CLI
    if not os.path.exists(exe):
        pytest.skip("ahsoka_b200/bin/Ahsoka_b200 not built")
    want = open(os.path.join(GOLDEN, case["ref_result"])).read()
    with tempfile.TemporaryDirectory() as td:
        _stage(case, td)
        got, out_gpu = _run_cli(exe, case, td)
        assert got == want
        ora = FLAT_ORACLE
        if ora is not None:
            with tempfile.TemporaryDirectory() as td2:
                _stage(case, td2)
                _, out_cpu = _run_cli(ora, case, td2)
            assert _hap_lines(out_gpu) == _hap_lines(out_cpu)


# ---- BASELINE.json configs[0] (cfg1: one chain of 1000 bubbles, 2k reads) through the CLI.  The GFA / GAF pair is
# re-generated from the seed (14 MB of text is not committed); tests/golden/cfg1.inputs.md5 pins it to the files
# tests/golden/cfg1.ref-result.txt was produced from by oracle/_ref/Ahsoka_ref (reference sources verbatim + shim).
def _cfg1_inputs(td):
    import hashlib
    import sys
    sys.path.insert(0, ROOT)
    from ahsoka_b200 import synth
    synth.generate(synth.config("cfg1"), os.path.join(td, "cfg1"))
    md5 = [hashlib.md5(open(os.path.join(td, "cfg1" + ext), "rb").read()).hexdigest() for ext in (".gfa", ".gaf")]
    assert md5 == open(os.path.join(GOLDEN, "cfg1.inputs.md5")).read().split(), "generator drifted: cfg1 inputs differ from the golden run's"


def _cfg1_cli(exe):
    want = open(os.path.join(GOLDEN, "cfg1.ref-result.txt")).read()
    with tempfile.TemporaryDirectory() as td:
        _cfg1_inputs(td)
        out = os.path.join(td, "out")
        r = subprocess.run([exe, "phase", "-g", os.path.join(td, "cfg1.gfa"), "-a", os.path.join(td, "cfg1.gaf"), "-o", out, "-t", "1"],
                           cwd=td, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1200)
        assert r.returncode == 0, r.stderr[-2000:]
        assert open(out + "-result.txt").read() == want


def test_cfg1_flat_oracle_cli_matches_reference_verbatim():
    exe = FLAT_ORACLE
    if exe is None:
        pytest.skip("oracle/_ref/Ahsoka_flat_oracle_standalone not built")
    _cfg1_cli(exe)


@pytest.mark.gpu
def test_cfg1_b200_cli_matches_reference_verbatim():
    if not os.path.exists(B200_CLI):
        pytest.skip("ahsoka_b200/bin/Ahsoka_b200 not built")
    _cfg1_cli(B200_CLI)


# ---- <prefix>-chain<id>-readset_final.txt (reference src/alignmentstoreadset.cpp:298-303): pinned to what Ahsoka_ref
# (reference sources verbatim + shim) writes for the same fixture; ReadSet::toString() itself is the shim's format.
def _readset_dumps(exe, case):
    import glob
    with tempfile.TemporaryDirectory() as td:
        _stage(case, td)
        _run_cli(exe, case, td)
        return {os.path.basename(p): open(p).read() for p in sorted(glob.glob(os.path.join(td, "out-chain*-readset_final.txt")))}


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_flat_oracle_cli_readset_final_dumps_match_reference_verbatim(case):
    ref, exe = os.path.join(REF_DIR, "Ahsoka_ref"), FLAT_ORACLE
    if not os.path.exists(ref) or exe is None:
        pytest.skip("oracle/_ref/Ahsoka_ref not built (needs the original Ahsoka sources at build time: AHSOKA_REFERENCE)")
    want = _readset_dumps(ref, case)
    assert want and _readset_dumps(exe, case) == want


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_b200_cli_readset_final_dumps_match_reference_verbatim(case):
    # against the original's binary when it was built; else against the drop-in with the CPU oracle behind the C ABI
    ref = os.path.join(REF_DIR, "Ahsoka_ref")
    ref = ref if os.path.exists(ref) else FLAT_ORACLE
    if ref is None or not os.path.exists(B200_CLI):
        pytest.skip("binaries not built")
    want = _readset_dumps(ref, case)
    assert want and _readset_dumps(B200_CLI, case) == want


@pytest.mark.gpu
def test_b200_cli_exit_code_tells_when_a_chain_exceeds_a_build_limit():
    # a chain beyond a build limit is reported on stderr, gets header-only output — and the process exits with code 3, so that
    # a dropped chain cannot be mistaken for an empty one (the limit is lowered through the library's testing knob)
    if not os.path.exists(B200_CLI):
        pytest.skip("ahsoka_b200/bin/Ahsoka_b200 not built")
    import sys
    sys.path.insert(0, ROOT)
    from ahsoka_b200 import synth
    with tempfile.TemporaryDirectory() as td:
        synth.generate(synth.params(2, 3, 0, 60, depth=80.0, seed=7), os.path.join(td, "s"))
        cmd = [B200_CLI, "phase", "-g", "s.gfa", "-a", "s.gaf", "-o", "out", "-t", "1"]
        ok = subprocess.run(cmd, cwd=td, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert ok.returncode == 0 and "haplotype 0:" in open(os.path.join(td, "out-result.txt")).read()
        os.remove(os.path.join(td, "out-result.txt"))
        env = dict(os.environ, AHS_MAX_READS_CLUSTER="180")
        r = subprocess.run(cmd, cwd=td, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=600)
        assert r.returncode == 3 and "NOT phased" in r.stderr
        assert "haplotype 0:" not in open(os.path.join(td, "out-result.txt")).read()


def test_standalone_command_line_parser():
    # the parser a build without the original's sources links (ahsoka_b200/host/standalone/standalone.cpp): the sub-commands
    # and options of the original's CLI; a wrong command line exits with 1 and says why, -h with 0, an option registered for
    # another sub-command is ignored, as the original's parser does
    exe = os.path.join(REF_DIR, "Ahsoka_flat_oracle_standalone")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/Ahsoka_flat_oracle_standalone not built")
    case = CASES[0]
    with tempfile.TemporaryDirectory() as td:
        _stage(case, td)
        gfa = os.path.join(GOLDEN, case["gfa"])

        def run(*args):
            return subprocess.run([exe] + list(args), cwd=td, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        for args, why in ((["phase", "-g", gfa, "-a", "reads.gaf"], "missing mandatory option -o"),
                          (["phase", "-g", gfa, "-a", "reads.gaf", "-o", "out", "-z", "1"], "unknown option -z"),
                          (["phase", "-g", gfa, "-a", "reads.gaf", "-o"], "option -o needs a value"),
                          (["bogus", "-g", gfa], "unknown sub-command 'bogus'"),
                          ([], "unknown sub-command ''")):
            r = run(*args)
            assert r.returncode == 1 and why in r.stderr and "usage: Ahsoka" in r.stderr, (args, r.returncode, r.stderr[-500:])
        r = run("phase", "-h")
        assert r.returncode == 0 and "usage: Ahsoka" in r.stderr
        r = run("only-bubbles", "-g", gfa, "-o", "bub", "-k", "ignored")
        assert r.returncode == 0 and os.path.exists(os.path.join(td, "bub-bubbleinfo.txt"))
        r = run("phase", "-g" + gfa, "-a", "reads.gaf", "-o", "out", "-t", "1")
        assert r.returncode == 0 and open(os.path.join(td, "out-result.txt")).read() == open(os.path.join(GOLDEN, case["ref_result"])).read()
