"""Host rows either side of the phasing call (SURVEY §8 f1, f2, f4): the native GAF reader
(ahsoka_b200/host/gaf_reader.cpp) and allele-path enumeration (chain_alleles.cpp) against the
reference's own functions.

oracle/_ref/Ahsoka_flat_oracle (built when AHSOKA_REFERENCE names the original's sources) links BOTH: the
reference translation units alignmentreader.cpp / chainstoreadset.cpp compiled where they lie, and this repo's
replacements; AHSOKA_HOST=reference selects the former.  Everything observable must then be byte-identical between
the two: the flattened batch handed to ahs_phase_batch (AHSOKA_DUMP_BATCH), the <gaf stem>-alignment_identities.txt
side file, -result.txt, -bubbleinfo.txt and stdout.  Without that binary the same tests run this repo's host stages
alone (oracle/_ref/Ahsoka_flat_oracle_standalone) and keep every assertion that does not need the original's
functions: the golden files written by the original, exit codes and messages, determinism.
"""
import json
import os
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
EXE_REF = os.path.join(ROOT, "oracle", "_ref", "Ahsoka_flat_oracle")                    # linked with the original's host stages
HAS_REF = os.path.exists(EXE_REF)
EXE = EXE_REF if HAS_REF else os.path.join(ROOT, "oracle", "_ref", "Ahsoka_flat_oracle_standalone")
CASES = [c for c in json.load(open(os.path.join(GOLDEN, "index.json")))["cases"] if "ref_result" in c]

pytestmark = pytest.mark.skipif(not os.path.exists(EXE), reason="oracle/_ref/Ahsoka_flat_oracle_standalone not built")


def test_reference_checker_is_built_when_the_original_is_given():
    # a build with AHSOKA_REFERENCE must leave the reference-linked checker: the comparisons below then must not quietly
    # fall back to this repo's host stages alone
    if not os.environ.get("AHSOKA_REFERENCE"):
        pytest.skip("AHSOKA_REFERENCE not set")
    assert HAS_REF, "AHSOKA_REFERENCE is set but oracle/_ref/Ahsoka_flat_oracle was not built"


def _run(td, tag, gfa_text, gaf_bytes, host, ploidy=2, expect_ok=True):
    d = os.path.join(td, tag)
    os.makedirs(d)
    open(os.path.join(d, "g.gfa"), "w").write(gfa_text)
    open(os.path.join(d, "reads.gaf"), "wb").write(gaf_bytes)
    env = dict(os.environ, AHSOKA_DUMP_BATCH=os.path.join(d, "batch.bin"), AHSOKA_PLOIDY=str(ploidy))
    if host == "reference":
        env["AHSOKA_HOST"] = "reference"
    else:
        env.pop("AHSOKA_HOST", None)
    r = subprocess.run([EXE, "phase", "-g", "g.gfa", "-a", "reads.gaf", "-o", "out", "-t", "1"], cwd=d,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, env=env)
    if not expect_ok:
        return r
    assert r.returncode == 0, r.stderr[-2000:]
    out = {"stdout": r.stdout}
    for f in ("batch.bin", "reads-alignment_identities.txt", "out-result.txt", "out-bubbleinfo.txt"):
        out[f] = open(os.path.join(d, f), "rb").read()
    return out


def _both(gfa_text, gaf_bytes, ploidy=2):
    """The native host's outputs, checked against the reference's functions when the checker links them."""
    with tempfile.TemporaryDirectory() as td:
        nat = _run(td, "nat", gfa_text, gaf_bytes, "native", ploidy)
        if HAS_REF:
            ref = _run(td, "ref", gfa_text, gaf_bytes, "reference", ploidy)
            for k in ref:
                assert ref[k] == nat[k], "native host differs from the reference's functions in " + k
    return nat


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_native_host_matches_reference_functions_on_golden_inputs(case):
    gfa = open(os.path.join(GOLDEN, case["gfa"])).read()
    gaf = open(os.path.join(GOLDEN, case["gaf"]), "rb").read()
    out = _both(gfa, gaf)
    # ... and the result is still the reference-verbatim binary's
    assert out["out-result.txt"] == open(os.path.join(GOLDEN, case["ref_result"]), "rb").read()


def test_identities_side_file_matches_reference_verbatim_binary():
    # tests/golden/dip_a-alignment_identities.txt was written by oracle/_ref/Ahsoka_ref (reference reader, verbatim)
    case = next(c for c in CASES if c["name"] == "dip_a")
    out = _both(open(os.path.join(GOLDEN, case["gfa"])).read(), open(os.path.join(GOLDEN, case["gaf"]), "rb").read())
    assert out["reads-alignment_identities.txt"] == open(os.path.join(GOLDEN, "dip_a-alignment_identities.txt"), "rb").read()


def _quirky_gaf(lines):
    """Every tolerated irregularity of reference src/alignmentreader.cpp:78-183 in one file."""
    out = []
    n = len(lines)
    for i, l in enumerate(lines):
        f = l.split(b"\t")
        if i % 11 == 0:
            out.append(b"")                                             # blank line (:84)
        if i % 7 == 1:
            l = b" ".join(f)                                            # any whitespace separates fields
        elif i % 7 == 2:
            l = l + b"\textra:Z:field"                                  # tokens after the 16th are never read
        elif i % 7 == 3:
            f[15] = b"id:f:x:" + f[15].split(b":")[-1]                  # value = text after the LAST ':' (:120-134)
            l = b"\t".join(f)
        elif i % 7 == 4:
            l = l + b"\r"                                               # CRLF: '\r' is whitespace to operator>>
        elif i % 7 == 5:
            f[5] = f[5].replace(b">", b">>", 1).replace(b"<", b"<<", 1)  # doubled direction characters (:143-149)
            l = b"\t".join(f)
        out.append(l)
        if i % 13 == 0:
            out.append(l)                                               # identical adjacent line
        if i % 17 == 0:
            out.append(lines[(i * 5 + 3) % n])                          # an earlier/later line repeated out of place
        if i % 19 == 0:
            g = list(f)
            g[5] = g[5] + b">utg9999999l"                               # node that is not in the graph → chain 0 (:180)
            out.append(b"\t".join(g))
        if i % 23 == 0:
            g = list(f)
            g[5] = g[5].replace(b"utg00", b"u", 1)                      # other spelling, same raw id (:48-54)
            out.append(b"\t".join(g))
        if i % 31 == 0:
            g = list(f)
            g[5] = g[5] + lines[(i * 7 + 11) % n].split(b"\t")[5] + g[5]    # one line through several chains, one of them twice
            out.append(b"\t".join(g))
        if i % 29 == 0:
            g = list(f)
            g[15] = b"id:f:9.3e-1"
            g[7] = b"+12junk"                                           # stoi stops at the first non-digit
            out.append(b"\t".join(g))
    body = b"\n".join(out) + b"\n"
    return body + lines[0]                                              # unterminated last line is dropped (:82)


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_native_reader_reproduces_reader_quirks(case):
    gfa = open(os.path.join(GOLDEN, case["gfa"])).read()
    lines = open(os.path.join(GOLDEN, case["gaf"]), "rb").read().split(b"\n")
    lines = [l for l in lines if l]
    _both(gfa, _quirky_gaf(lines))


def test_unterminated_last_line_is_dropped():
    case = CASES[0]
    gfa = open(os.path.join(GOLDEN, case["gfa"])).read()
    gaf = open(os.path.join(GOLDEN, case["gaf"]), "rb").read()
    assert gaf.endswith(b"\n")
    a = _both(gfa, gaf)
    b = _both(gfa, gaf[:-1])
    assert a["reads-alignment_identities.txt"].count(b"\n") == b["reads-alignment_identities.txt"].count(b"\n") + 1
    with tempfile.TemporaryDirectory() as td:      # empty and missing-newline-only files: no alignments, header-only result
        e = _run(td, "empty", gfa, b"", "native")
        if HAS_REF:
            assert e == _run(td, "empty_ref", gfa, b"", "reference")
    assert e["out-result.txt"] and b"haplotype" not in e["out-result.txt"]


MALFORMED = {
    "short": lambda f: f[:15],
    "no_id_tag": lambda f: f[:15] + [b"dv:f:0.1"],
    "id_not_float": lambda f: f[:15] + [b"id:f:abc"],
    "path_without_direction": lambda f: f[:5] + [f[5][1:]] + f[6:],
    "node_without_digits": lambda f: f[:5] + [f[5] + b">utgl"] + f[6:],
    "node_id_overflow": lambda f: f[:5] + [f[5] + b">utg99999999999l"] + f[6:],
    "start_not_int": lambda f: f[:7] + [b"x"] + f[8:],
}


@pytest.mark.parametrize("kind", sorted(MALFORMED))
def test_malformed_lines_fail_loudly_where_the_reference_dies(kind):
    case = CASES[0]
    gfa = open(os.path.join(GOLDEN, case["gfa"])).read()
    lines = [l for l in open(os.path.join(GOLDEN, case["gaf"]), "rb").read().split(b"\n") if l]
    lines[5] = b"\t".join(MALFORMED[kind](lines[5].split(b"\t")))
    gaf = b"\n".join(lines) + b"\n"
    with tempfile.TemporaryDirectory() as td:
        nat = _run(td, "nat", gfa, gaf, "native", expect_ok=False)
        if HAS_REF:
            assert _run(td, "ref", gfa, gaf, "reference", expect_ok=False).returncode != 0, "the reference's reader accepted this line"
    assert nat.returncode == 65
    assert b"reads.gaf:6:" in nat.stderr


def _synth_text(prm):
    from ahsoka_b200 import synth
    with tempfile.TemporaryDirectory() as td:
        synth.generate(prm, os.path.join(td, "x"))
        return open(os.path.join(td, "x.gfa")).read(), open(os.path.join(td, "x.gaf"), "rb").read()


def test_allele_paths_of_multi_allele_bubbles():
    # bubbles with 3 inner nodes take findPathsComplex (chainstoreadset.cpp:84-116): paths start at the SINK
    from ahsoka_b200 import synth
    gfa, gaf = _synth_text(synth.params(3, 5, 1, 10, depth=12.0, seed=311))
    _both(gfa, gaf, ploidy=3)


def test_allele_paths_of_nested_bubbles():
    # put a node in series behind one inner node of some bubbles: the bubble then has three inner nodes and one
    # allele path of four nodes (depth-first enumeration, addSequence chainstoreadset.cpp:44-82)
    from ahsoka_b200 import synth
    gfa, gaf = _synth_text(synth.params(2, 4, 1, 8, depth=10.0, seed=312))
    L = [l.split("\t") for l in gfa.split("\n") if l.startswith("L")]
    S = [l for l in gfa.split("\n") if l.startswith("S")]
    nxt = len(S) + 1
    # plus-strand links in file order: flank→a0, then per allele (anchor→inner, inner→next anchor)
    plus = [l for l in L if l[2] == "+"]
    outdeg = {}
    for l in plus:
        outdeg[l[1]] = outdeg.get(l[1], 0) + 1
    inner_out = [l for l in plus if outdeg.get(l[1], 0) == 1 and sum(1 for m in plus if m[3] == l[1]) == 1 and
                 outdeg.get(next(m[1] for m in plus if m[3] == l[1]), 0) == 2]
    assert len(inner_out) > 8
    edited = 0
    new_L = list(L)
    for l in inner_out[1::5]:
        name = "utg%07dl" % nxt
        nxt += 1
        S.append("S\t%s\tA" % name)
        inner, anchor = l[1], l[3]
        new_L = [m for m in new_L if not (m[1] == inner and m[2] == "+" and m[3] == anchor) and not (m[1] == anchor and m[2] == "-" and m[3] == inner)]
        for a, b in ((inner, name), (name, anchor)):
            new_L.append(["L", a, "+", b, "+", "0M"])
            new_L.append(["L", b, "-", a, "-", "0M"])
        edited += 1
    assert edited >= 2
    gfa2 = "\n".join(S + ["\t".join(m) for m in new_L]) + "\n"
    out = _both(gfa2, gaf)
    assert out["out-bubbleinfo.txt"].count(b"bubble id") > 0


def _messy_gfa(seed):
    """Random small graphs: bubble chains with tips, loops, cross links, one-sided links, repeated S lines, other
    record types — every branch of Graph::findBubble (graph.cpp:381-500) gets exercised."""
    import random
    rng = random.Random(seed)
    lines = ["H\tVN:Z:1.0"]
    n = rng.randint(6, 40)
    ids = list(range(1, n + 1))
    rng.shuffle(ids)
    for i in ids:
        lines.append("S\tutg%06dl\t%s" % (i, "ACGT"[: rng.randint(1, 4)]))
    links = set()

    def link(a, sa, b, sb, both=True):
        links.add((a, sa, b, sb))
        if both:
            links.add((b, "-" if sb == "+" else "+", a, "-" if sa == "+" else "+"))

    # a backbone of bubbles / linear stretches
    cur = 1
    nxt = 2
    while nxt + 3 <= n:
        kind = rng.random()
        if kind < 0.55:                      # simple bubble cur -> {a, b} -> c
            a, b, c = nxt, nxt + 1, nxt + 2
            for x in (a, b):
                link(cur, "+", x, "+"); link(x, "+", c, "+")
            cur, nxt = c, nxt + 3
        elif kind < 0.7:                     # three-allele bubble
            if nxt + 4 > n:
                break
            a, b, c, e = nxt, nxt + 1, nxt + 2, nxt + 3
            for x in (a, b, c):
                link(cur, "+", x, "+"); link(x, "+", e, "+")
            cur, nxt = e, nxt + 4
        elif kind < 0.85:                    # linear step
            link(cur, "+", nxt, "+")
            cur, nxt = nxt, nxt + 1
        else:                                # nested: cur -> a -> b -> c, cur -> d -> c
            if nxt + 4 > n:
                break
            a, b, d, c = nxt, nxt + 1, nxt + 2, nxt + 3
            link(cur, "+", a, "+"); link(a, "+", b, "+"); link(b, "+", c, "+"); link(cur, "+", d, "+"); link(d, "+", c, "+")
            cur, nxt = c, nxt + 4
    for _ in range(rng.randint(0, 4)):      # noise: tips, cross links, loops, one-sided links, inversions
        a, b = rng.randint(1, n), rng.randint(1, n)
        link(a, rng.choice("+-"), b, rng.choice("+-"), both=rng.random() < 0.7)
    out = list(links)
    rng.shuffle(out)
    for a, sa, b, sb in out:
        lines.append("L\tutg%06dl\t%s\tutg%06dl\t%s\t%dM" % (a, sa, b, sb, rng.choice([0, 0, 17])))
    if rng.random() < 0.3:
        lines.insert(rng.randint(1, n), "")           # blank line
    if rng.random() < 0.3:
        lines.append("P\tpath1\tutg000001l+\t*")      # other record types are skipped (:194)
    text = "\n".join(lines) + "\n"
    if rng.random() < 0.2:
        text += "S\tutg999999l\tA"                    # unterminated last line is dropped (:192)
    return text


def _only_bubbles(td, tag, gfa_text, host):
    d = os.path.join(td, tag)
    os.makedirs(d)
    open(os.path.join(d, "g.gfa"), "w").write(gfa_text)
    env = dict(os.environ)
    env.pop("AHSOKA_HOST", None)
    if host == "reference":
        env["AHSOKA_HOST"] = "reference"
    try:
        r = subprocess.run([EXE, "only-bubbles", "-g", "g.gfa", "-o", "out"], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=20, env=env)
    except subprocess.TimeoutExpired:
        return None
    if r.returncode != 0:
        return None
    return r.stdout, open(os.path.join(d, "out-bubbleinfo.txt"), "rb").read()


def test_bubble_detection_on_messy_graphs():
    ok = 0
    with_bubbles = 0
    with tempfile.TemporaryDirectory() as td:
        for seed in range(150):
            gfa = _messy_gfa(seed)
            if not HAS_REF:         # this repo's detection alone: it finishes on every graph and finds the chains it finds with the original
                nat = _only_bubbles(td, "n%d" % seed, gfa, "native")
                if nat is not None:
                    ok += 1
                    with_bubbles += b"bubble id" in nat[1]
                    _run(td, "pn%d" % seed, gfa, b"", "native", expect_ok=False)       # terminates (else TimeoutExpired)
                continue
            ref = _only_bubbles(td, "r%d" % seed, gfa, "reference")
            if ref is None:
                continue        # the reference itself crashes or does not terminate on this graph
            nat = _only_bubbles(td, "n%d" % seed, gfa, "native")
            assert nat is not None, "native detection failed where the reference ran (seed %d)" % seed
            assert nat == ref, "bubble chains differ from the reference's (seed %d)" % seed
            ok += 1
            with_bubbles += b"bubble id" in ref[1]
            # and the stages behind it (reader's chain lookup, allele paths, flattening) on the same graph
            try:
                r2 = _run(td, "pr%d" % seed, gfa, b"", "reference")
            except (AssertionError, subprocess.TimeoutExpired):
                continue        # the reference's allele-path enumeration dies on this bubble
            n2 = _run(td, "pn%d" % seed, gfa, b"", "native")
            assert r2 == n2, "seed %d" % seed
    assert ok >= 100 and with_bubbles >= 80, (ok, with_bubbles)


MALFORMED_GFA = {
    "s_without_sequence": "S\tutg000001l\n",
    "s_without_digits": "S\tutgl\tA\n",
    "l_bad_orientation": "S\tu1\tA\nS\tu2\tA\nL\tu1\t*\tu2\t+\t0M\n",
    "l_star_overlap": "S\tu1\tA\nS\tu2\tA\nL\tu1\t+\tu2\t+\t*\n",
    "l_negative_overlap": "S\tu1\tA\nS\tu2\tA\nL\tu1\t+\tu2\t+\t-3M\n",
}


@pytest.mark.parametrize("kind", sorted(MALFORMED_GFA))
def test_malformed_gfa_fails_loudly_where_the_reference_dies(kind):
    with tempfile.TemporaryDirectory() as td:
        if HAS_REF:
            assert _only_bubbles(td, "ref", MALFORMED_GFA[kind], "reference") is None
        d = os.path.join(td, "nat")
        os.makedirs(d)
        open(os.path.join(d, "g.gfa"), "w").write(MALFORMED_GFA[kind])
        r = subprocess.run([EXE, "only-bubbles", "-g", "g.gfa", "-o", "out"], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=20)
    assert r.returncode == 66 and b"g.gfa:" in r.stderr


def _cli_files(exe, td, tag, gfa_text, gaf_bytes, ploidy):
    d = os.path.join(td, tag)
    os.makedirs(d)
    open(os.path.join(d, "g.gfa"), "w").write(gfa_text)
    open(os.path.join(d, "reads.gaf"), "wb").write(gaf_bytes)
    env = dict(os.environ, AHSOKA_PLOIDY=str(ploidy))
    env.pop("AHSOKA_HOST", None)
    r = subprocess.run([exe, "phase", "-g", "g.gfa", "-a", "reads.gaf", "-o", "out", "-t", "1"], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout, open(os.path.join(d, "out-result.txt"), "rb").read(), open(os.path.join(d, "out-bubbleinfo.txt"), "rb").read()


@pytest.mark.gpu
@pytest.mark.parametrize("ploidy,seed", [(2, 411), (3, 412), (4, 413)])
def test_b200_cli_equals_oracle_cli_on_polyploid_graphs(ploidy, seed):
    # the whole drop-in (native host stages + CUDA library) against the same host with the CPU oracle behind the C ABI
    from ahsoka_b200 import synth
    cuda_exe = os.path.join(ROOT, "ahsoka_b200", "bin", "Ahsoka_b200")
    if not os.path.exists(cuda_exe):
        pytest.skip("ahsoka_b200/bin/Ahsoka_b200 not built")
    gfa, gaf = _synth_text(synth.params(ploidy, 12, 1, 14, depth=12.0 * ploidy, seed=seed))
    with tempfile.TemporaryDirectory() as td:
        assert _cli_files(cuda_exe, td, "cuda", gfa, gaf, ploidy) == _cli_files(EXE, td, "cpu", gfa, gaf, ploidy)


def test_reader_thread_count_does_not_change_the_batch():
    # a GAF above 1 MB is parsed in line-aligned slabs on several threads and merged in file order: same batch, same side file
    from ahsoka_b200 import synth
    gfa, gaf = _synth_text(synth.params(2, 60, 1, 30, depth=25.0, dup_lines=200, seed=515))
    assert len(gaf) > (1 << 20)
    outs = []
    with tempfile.TemporaryDirectory() as td:
        for t in (2, 3, 7):
            d = os.path.join(td, "t%d" % t)
            os.makedirs(d)
            open(os.path.join(d, "g.gfa"), "w").write(gfa)
            open(os.path.join(d, "reads.gaf"), "wb").write(gaf)
            env = dict(os.environ, AHSOKA_DUMP_BATCH=os.path.join(d, "batch.bin"))
            env.pop("AHSOKA_HOST", None)
            r = subprocess.run([EXE, "phase", "-g", "g.gfa", "-a", "reads.gaf", "-o", "out", "-t", str(t)], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, env=env)
            assert r.returncode == 0, r.stderr[-2000:]
            outs.append((open(os.path.join(d, "batch.bin"), "rb").read(), open(os.path.join(d, "reads-alignment_identities.txt"), "rb").read(),
                         open(os.path.join(d, "out-result.txt"), "rb").read()))
        ref = _run(td, "ref", gfa, gaf, "reference") if HAS_REF else None
    assert outs[0] == outs[1] == outs[2]
    if ref is not None:
        assert outs[0] == (ref["batch.bin"], ref["reads-alignment_identities.txt"], ref["out-result.txt"])
