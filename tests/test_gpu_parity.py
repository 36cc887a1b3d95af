"""-m gpu: the CUDA path, through the C ABI, against the CPU oracle on the same seeded inputs.
Bar: bit-exact on every output array (integer / index work; dp_cost is integer valued)."""
import os

import numpy as np
import pytest

from ahsoka_b200 import api, synth
from tests.oracle_binding import oracle_phase

pytestmark = pytest.mark.gpu


def _check(batch, **kw):
    got = api.phase_batch(batch, **kw)
    want = oracle_phase(batch)
    bad = got.diff(want)
    assert not bad, f"GPU differs from oracle in {bad}"
    return got


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_diploid_small_chains(seed):
    got = _check(synth.generate(synth.params(2, 40, 1, 24, depth=30.0, seed=seed)))
    assert got.n_chains_ok > 30


@pytest.mark.parametrize("mean_len,n_chains,seed", [(80, 30, 71), (110, 40, 74), (140, 12, 72)])
def test_diploid_mid_and_big_chains(mean_len, n_chains, seed):
    # ~100, ~145 and ~180 final reads per chain: the large shared-memory classes (up to 160 reads, 1024 threads with
    # 9-13 pair slots each) and, above, the HBM-resident scoring / cluster-editing path
    got = _check(synth.generate(synth.params(2, n_chains, 1, mean_len, depth=30.0, seed=seed)))
    assert got.n_chains_ok == n_chains


def test_long_chains_low_depth_wide_rate_keys():
    # ~400 bubbles, ~70 final reads per chain: shared-memory scoring with the 62-bit rate keys (overlaps may exceed 255)
    got = _check(synth.generate(synth.params(2, 8, 1, 400, depth=4.0, seed=73)))
    assert got.n_chains_ok == 8


def test_cfg3_sample_triploid_chains_up_to_150_reads():
    got = _check(synth.generate(synth.config("cfg3", 0.01)))
    assert got.n_chains_ok > 150
    assert int(np.diff(got.read_off).max()) > 128


def test_cfg2_sample():
    got = _check(synth.generate(synth.config("cfg2", 0.01)))
    assert got.n_chains_ok > 400


def test_diploid_tiny_and_trivial_chains():
    # chains of 1..6 bubbles: <=1 bubble is header-only (status 1), very short chains often end empty (status 2)
    _check(synth.generate(synth.params(2, 60, 1, 3, min_len=1, depth=12.0, seed=11)))


def test_diploid_low_depth_empty_chains():
    got = _check(synth.generate(synth.params(2, 50, 1, 10, depth=2.0, seed=5)))
    assert (got.status == 2).any()


def test_cfg1_one_long_chain():
    got = _check(synth.generate(synth.config("cfg1")))
    assert got.n_chains_ok == 1 and got.n_cells > 15000


def test_multiline_reads():
    # same read name on two GAF lines with different identity (SURVEY A#3)
    _check(synth.generate(synth.params(2, 30, 1, 30, depth=25.0, dup_lines=300, seed=21)))


@pytest.mark.parametrize("ploidy,seed", [(3, 31), (4, 41), (5, 51), (6, 61)])
def test_polyploid(ploidy, seed):
    # ploidy 3, 4: ordered tuples (rule R3); ploidy 5, 6: canonical tuples over the first p + 2 clusters (rule R3c)
    got = _check(synth.generate(synth.params(ploidy, 12, 1, 30, depth=10.0 * ploidy, seed=seed)))
    assert got.n_chains_ok == 12


def test_hexaploid_many_alleles_and_short_chains():
    _check(synth.generate(synth.params(6, 40, 1, 8, min_len=1, depth=50.0, max_alleles=12, seed=62)))
    _check(synth.generate(synth.params(5, 10, 1, 60, depth=30.0, max_alleles=3, seed=52)))          # 2-bit codes at ploidy 5


def test_cfg5_sample_hexaploid_skewed_chain_sizes():
    # BASELINE configs[4] at reduced chain length: ploidy 6, 80x, Zipf-skewed sizes with one forced 600-bubble chain
    # (~2,000 final reads: the big-chain cluster editing + the canonical-tuple DP over 600 columns)
    b = synth.generate(synth.params(6, 24, 2, 500, 2, 600, 1.2, 1, depth=80.0, seed=0xA450CA05))
    got = _check(b)
    assert got.n_chains_ok >= 20 and int(np.diff(got.read_off).max()) > 1500


def test_four_bit_codes_diploid_many_alleles():
    _check(synth.generate(synth.params(2, 20, 1, 20, depth=30.0, max_alleles=6, seed=51)))


def test_resident_mode_same_result():
    b = synth.generate(synth.params(2, 30, 1, 30, depth=30.0, seed=61))
    _check(b, resident_iters=2, warmup=1)


def test_zero_copy_views_and_release():
    b = synth.generate(synth.params(2, 20, 1, 20, depth=30.0, seed=81))
    want = oracle_phase(b)
    got = api.phase_batch(b, copy=False)
    assert not got.diff(want)
    # the output buffers are still owned by the library: a second call on the device must be refused ...
    with pytest.raises(RuntimeError):
        api.phase_batch(b)
    got.release()
    # ... and accepted again after the release
    assert not api.phase_batch(b).diff(want)


def _broken(b, **kw):
    import copy
    c = copy.copy(b)
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def test_malformed_batches_are_rejected_not_mis_phased():
    b = synth.generate(synth.params(2, 8, 1, 12, depth=20.0, seed=91))
    er = b.entry_read.copy(); er[3] = 10 ** 6
    with pytest.raises(RuntimeError, match="entry_read"):
        api.phase_batch(_broken(b, entry_read=er))
    ao = b.allele_off.copy(); ao[5], ao[6] = ao[6] + 1, ao[5]
    with pytest.raises(RuntimeError, match="monotone"):
        api.phase_batch(_broken(b, allele_off=ao))
    so = b.stage_a_order.copy(); so[1] = so[0]
    with pytest.raises(RuntimeError, match="permutation"):
        api.phase_batch(_broken(b, stage_a_order=so))
    eo = b.enode_off.copy(); eo[2] = eo[3] + 5
    with pytest.raises(RuntimeError, match="monotone"):
        api.phase_batch(_broken(b, enode_off=eo))
    # the library is still usable afterwards
    assert not api.phase_batch(b).diff(oracle_phase(b))


def test_cfg2_full_size_against_oracle():
    # BASELINE configs[1] at full size: 50k chains, 2M bubbles, 45.7M cells — the bench workload itself
    b = synth.generate(synth.config("cfg2"))
    got = api.phase_batch(b, copy=False)
    want = oracle_phase(b, os.cpu_count() or 1)
    try:
        assert not got.diff(want)
        assert got.n_chains_ok == 50000 and got.n_cells == want.n_cells
    finally:
        got.release()


def test_chains_are_independent_permutation_property():
    # size-independent property: phasing a permutation of the chains gives the permuted result
    b = synth.generate(synth.config("cfg2", 0.02))
    perm = np.random.default_rng(3).permutation(b.n_chains)
    r1 = api.phase_batch(b)
    r2 = api.phase_batch(b.select(perm))
    assert np.array_equal(r2.status, r1.status[perm]) and np.array_equal(r2.dp_cost, r1.dp_cost[perm])
    assert np.array_equal(r2.n_clusters, r1.n_clusters[perm])
    for k, c in enumerate(perm[:200]):
        a0, a1 = r1.read_off[c], r1.read_off[c + 1]
        b0, b1 = r2.read_off[k], r2.read_off[k + 1]
        assert np.array_equal(r1.read_cluster[a0:a1], r2.read_cluster[b0:b1])
        p0, p1 = r1.pos_off[c] * 2, r1.pos_off[c + 1] * 2
        q0, q1 = r2.pos_off[k] * 2, r2.pos_off[k + 1] * 2
        assert np.array_equal(r1.hap_allele[p0:p1], r2.hap_allele[q0:q1]) and np.array_equal(r1.path[p0:p1], r2.path[q0:q1])


def test_phasing_recovers_the_simulated_haplotypes():
    # domain property at size: with 5 % allele error the emitted haplotypes agree with the truth at > 95 % of the
    # covered positions of long enough chains (up to the haplotype swap)
    b = synth.generate(synth.config("cfg2", 0.02))
    r = api.phase_batch(b)
    truth = b.truth["hap_allele"].reshape(-1, 2)
    agree = tot = 0
    for c in range(b.n_chains):
        if r.status[c] != 0:
            continue
        q0, q1 = int(r.pos_off[c]), int(r.pos_off[c + 1])
        if q1 - q0 < 10:
            continue
        gb = int(b.bubble_off[c]) + r.pos[q0:q1]
        t = truth[gb]
        h = r.hap_allele[q0 * 2:q1 * 2].reshape(-1, 2)
        same = int((h == t).all(axis=1).sum()); swap = int((h == t[:, ::-1]).all(axis=1).sum())
        agree += max(same, swap); tot += q1 - q0
    assert tot > 1000 and agree / tot > 0.95


def test_multi_device_lpt_gather():
    # one batch dealt over the devices of the box (heavy chains one by one, the tail in ranges of consecutive chains,
    # LPT), every device writing its ranges straight into the output arrays.  Needs >= 2 GPUs: on a one-GPU box the
    # same assertion runs inside `bench.py --gpus 2` (key "multi" of the JSON line).
    n = api.load_library().ahs_device_count()
    if n < 2:
        pytest.skip("needs two CUDA devices")
    b = synth.generate(synth.config("cfg2", 0.02))
    want = oracle_phase(b)
    for devs in ([0, 1], list(range(n))):
        got = api.phase_batch(b, devices=devs)
        assert not got.diff(want)
    skew = synth.generate(synth.params(2, 300, 2, 40, 2, 400, 1.2, 3, depth=30.0, seed=77))       # Zipf-skewed chain sizes
    assert not api.phase_batch(skew, devices=[0, 1]).diff(oracle_phase(skew))
    with pytest.raises(RuntimeError, match="listed twice"):
        api.phase_batch(b, devices=[0, 0])


def test_multi_device_call_on_one_device_equals_single_call():
    # the multi-device entry point with one device is the single-device path (runs on any box)
    b = synth.generate(synth.config("cfg2", 0.01))
    assert not api.phase_batch(b, devices=[0]).diff(oracle_phase(b))


@pytest.mark.parametrize("desc", [False, True])
def test_std_sort_replay_including_the_heap_sort_fallback(desc):
    # ReadSet::sort() (alignmentstoreadset.cpp:297) and the cluster sort (:720) are libstdc++ std::sort calls with a
    # comparator on the key only; the device replays them move for move.  Inputs: ties, already sorted keys (what
    # ReadSet::sort sees), permutations, and McIlroy's adversary, which drives introsort into its heap-sort fall-back.
    from tests.oracle_binding import oracle_antiqsort, oracle_std_sort
    rng = np.random.default_rng(5)
    for n in (0, 1, 2, 15, 16, 17, 33, 100, 128, 129, 1000, 8191, 20000):
        cases = [rng.integers(0, 50, n), np.sort(rng.integers(0, max(2, n // 8), n)), rng.permutation(n)]
        k = oracle_antiqsort(n)
        cases.append(-k if desc else k)
        for keys in cases:
            vals = np.arange(n, dtype=np.int32)
            gk, gv = api.debug_std_sort(keys, vals, desc)
            wk, wv = oracle_std_sort(keys, vals, desc)
            assert np.array_equal(gk, wk) and np.array_equal(gv, wv), (n, desc)


def test_cfg4_shape_tetraploid_chains_of_200_to_330_reads():
    # BASELINE configs[3] at its shape: ploidy 4, 60x -> 200-330 final reads per chain: HBM-resident scoring, the
    # big-chain cluster editing (k_cluster_sparse, chains above 160 reads) and the 4096-state threading DP together
    b = synth.generate(synth.config("cfg4", 0.005))
    got = _check(b)
    assert b.ploidy == 4 and got.n_chains_ok == b.n_chains
    assert int(np.diff(got.read_off).max()) > 250


def test_tetraploid_more_than_eight_alleles():
    # ploidy 4 with up to 12 alleles per bubble: 4-bit codes and 8 clusters per DP column
    got = _check(synth.generate(synth.params(4, 10, 1, 30, depth=60.0, max_alleles=12, seed=77)))
    assert got.n_chains_ok == 10


def test_randomised_shapes_twice_each():
    # chain length 3..120, depth 3..90, ploidy 2..4, up to 12 alleles, duplicated read names, error / missing rates:
    # every case bit-identical to the oracle, in two consecutive runs (a data race would show up as a flaky diff)
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(api.ROOT, "tests", "stress_gpu.py"), "30", "4242"], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stdout[-2000:]


def test_build_limits_are_reported_not_mis_phased():
    import copy
    b = synth.generate(synth.params(2, 6, 1, 12, depth=20.0, seed=97))
    b5 = copy.copy(b); b5.ploidy = 7
    with pytest.raises(RuntimeError, match=r"failed \(3\).*ploidy"):          # AHS_ERR_LIMIT
        api.phase_batch(b5)
    # a bubble with 16 alleles: more than the 4-bit codes hold
    wide = synth.generate(synth.params(2, 4, 1, 8, depth=20.0, max_alleles=15, seed=98))
    ao = wide.allele_off.copy(); no = wide.anode_off.copy()
    k0 = int(np.argmax(np.diff(ao)))                                       # widen its largest bubble to 16 alleles by repeating one path
    extra = 16 - int(ao[k0 + 1] - ao[k0])
    a_last = int(ao[k0 + 1]) - 1
    path = wide.anode[no[a_last]:no[a_last + 1]]
    new_anode = np.concatenate([wide.anode[:no[a_last + 1]]] + [path] * extra + [wide.anode[no[a_last + 1]:]])
    new_no = np.concatenate([no[:a_last + 2], no[a_last + 1] + len(path) * np.arange(1, extra + 1), no[a_last + 2:] + len(path) * extra])
    new_ao = ao.copy(); new_ao[k0 + 1:] += extra
    w2 = copy.copy(wide); w2.allele_off, w2.anode_off, w2.anode = new_ao, new_no.astype(np.int64), new_anode.astype(np.int32)
    with pytest.raises(RuntimeError, match=r"failed \(3\).*15 alleles"):
        api.phase_batch(w2)
    # a chain with more final reads than cluster editing accepts (65,535; lowered here through the testing knob): reported
    # per chain, the other chains are phased
    big = synth.generate(synth.params(2, 1, 0, 300, depth=80.0, seed=99))
    small = synth.generate(synth.params(2, 5, 1, 12, depth=20.0, seed=100))
    os.environ["AHS_MAX_READS_CLUSTER"] = "500"
    try:
        got = api.phase_batch(big)
    finally:
        del os.environ["AHS_MAX_READS_CLUSTER"]
    assert int(got.status[0]) == 3 and got.read_off[-1] == 0               # AHS_CHAIN_TOO_LARGE, nothing emitted for it
    assert not api.phase_batch(small).diff(oracle_phase(small))


def test_long_chains_of_thousands_of_reads():
    # a chain of 600 bubbles at 80x (~2,100 final reads, 80 k edges, neighbourhoods of > 1,000 nodes) and chains just above
    # 1,024 reads: edge slots + lists + maximum tree (k_cluster_sparse), both block sizes
    b = synth.generate(synth.params(2, 1, 0, 600, depth=80.0, seed=99))
    got = _check(b)
    assert got.n_chains_ok == 1 and int(np.diff(got.read_off).min()) > 2000
    b = synth.generate(synth.params(3, 3, 0, 700, depth=45.0, seed=98))
    got = _check(b)
    assert got.n_chains_ok == 3 and int(np.diff(got.read_off).min()) > 1024


@pytest.mark.parametrize("chunks", ["1", "2", "4"])
def test_chunked_call_is_result_identical(chunks, monkeypatch):
    # a large call runs as several chunks of chains in flight (H2D of chunk k+1 under the clustering of chunk k):
    # same result for every chunk count
    b = synth.generate(synth.config("cfg2", 0.25))
    want = oracle_phase(b, os.cpu_count() or 1)
    monkeypatch.setenv("AHS_CHUNKS", chunks)
    assert not api.phase_batch(b).diff(want)


_DEL_ANODE = [1, 2, 4, 1, 3, 4,   4, 5, 7, 7, 4,   7, 8, 10, 7, 9, 10]
_DEL_ANODE_OFF = [0, 3, 6, 9, 11, 14, 17]
_DEL_ALLELE_OFF = [0, 2, 4, 6]
_DEL_READS = [[1, 2, 4, 5, 7, 8, 10], [1, 3, 4, 7, 9, 10], [1, 2, 4], [7, 8, 10, 4, 5], [1, 3, 4, 5, 7, 9, 10]]


def deletion_allele_chain():
    """One diploid chain of three bubbles whose middle bubble has the allele path 7-4: two nodes, no inner node."""
    n = len(_DEL_READS)
    return api.Batch(2, [0], [0, 3], _DEL_ALLELE_OFF, _DEL_ANODE_OFF, _DEL_ANODE, [2, 1, 0], [0, n], [0, n],
                     np.cumsum([0] + [len(x) for x in _DEL_READS]), sum(_DEL_READS, []), list(range(n)), [0.99] * n)


def test_deletion_allele_matches_every_entry():
    # allele path of two nodes (no inner node): stage B matches it for every entry of the chain (SURVEY A#9); same hand-made
    # chain as tests/test_oracle_cpu.py, alone and next to ordinary chains (the per-chain "has universal allele" flag)
    from ahsoka_b200.api import Batch
    anode, anode_off, allele_off, reads = _DEL_ANODE, _DEL_ANODE_OFF, _DEL_ALLELE_OFF, _DEL_READS
    enode = sum(reads, [])
    enode_off = np.cumsum([0] + [len(x) for x in reads])
    got = _check(deletion_allele_chain())
    assert got.status[0] == 0
    # the same chain between two synthetic ones
    s = synth.generate(synth.params(2, 2, 1, 12, depth=20.0, seed=333))
    nb, na, nan_, nr, ne, nen = (int(s.bubble_off[1]), int(s.allele_off[s.bubble_off[1]]), int(s.anode_off[s.allele_off[s.bubble_off[1]]]),
                                 int(s.read_off[1]), int(s.entry_off[1]), int(s.enode_off[s.entry_off[1]]))
    cat = np.concatenate
    mixed = Batch(2, [int(s.chain_id[0]), 777, int(s.chain_id[1])],
                  cat([s.bubble_off[:2], [nb + 3], s.bubble_off[2:] + 3]),
                  cat([s.allele_off[:nb + 1], na + np.array(allele_off[1:]), s.allele_off[nb + 1:] + 6]),
                  cat([s.anode_off[:na + 1], nan_ + np.array(anode_off[1:]), s.anode_off[na + 1:] + len(anode)]),
                  cat([s.anode[:nan_], np.array(anode) + 10 ** 6, s.anode[nan_:]]),
                  cat([s.stage_a_order[:nb], [2, 1, 0], s.stage_a_order[nb:]]),
                  cat([s.read_off[:2], [nr + len(reads)], s.read_off[2:] + len(reads)]),
                  cat([s.entry_off[:2], [ne + len(reads)], s.entry_off[2:] + len(reads)]),
                  cat([s.enode_off[:ne + 1], nen + enode_off[1:], s.enode_off[ne + 1:] + len(enode)]),
                  cat([s.enode[:nen], np.array(enode) + 10 ** 6, s.enode[nen:]]),
                  cat([s.entry_read[:ne], np.arange(len(reads)), s.entry_read[ne:]]),
                  cat([s.entry_identity[:ne], np.full(len(reads), 0.99, dtype=np.float32), s.entry_identity[ne:]]))
    got = _check(mixed)
    assert list(got.status) == [0, 0, 0]


def test_cfg5_chain_of_five_thousand_bubbles_against_the_truth():
    # BASELINE configs[4] at its shape: ploidy 6, 80x, one chain of 5,000 bubbles (~17,500 final reads, 0.7 M edges) next to
    # short ones.  The CPU oracle needs hours for such a chain (dense n x n state), so this is a property test at size: every
    # chain is phased, the reads of the long chain fall into about ploidy clusters, and the emitted haplotypes carry the
    # generator's true allele multiset at > 99 % of its positions (labels are arbitrary, the multiset is not).
    b = synth.generate(synth.params(6, 6, 2, 500, 2, 5000, 1.2, 1, depth=80.0, seed=0xA450CA05))
    r = api.phase_batch(b)
    p = 6
    assert (r.status == 0).all()
    nr = np.diff(r.read_off)
    c = int(np.argmax(nr))
    assert int(np.diff(b.bubble_off)[c]) == 5000 and int(nr[c]) > 15000
    assert 6 <= int(r.n_clusters[c]) <= 16
    q0, q1 = int(r.pos_off[c]), int(r.pos_off[c + 1])
    truth = b.truth["hap_allele"].reshape(-1, p)[int(b.bubble_off[c]) + r.pos[q0:q1]]
    hap = r.hap_allele[q0 * p:q1 * p].reshape(-1, p)
    same = int((np.sort(truth, axis=1) == np.sort(hap, axis=1)).all(axis=1).sum())
    assert q1 - q0 > 4900 and same > 0.99 * (q1 - q0)
    # every read of the chain has a cluster, cluster ids are dense
    cl = r.read_cluster[int(r.read_off[c]):int(r.read_off[c + 1])]
    assert set(np.unique(cl).tolist()) == set(range(int(r.n_clusters[c])))


def test_committed_golden_fixtures():
    # tests/golden/*.batch.npz -> *.result.npz (written by tests/golden/make_golden.py from the CPU oracle; the same files pin
    # the oracle itself in tests/test_oracle_cpu.py): ploidy 2-6, duplicated read names, a chain above 160 reads
    import json
    golden = os.path.join(api.ROOT, "tests", "golden")
    cases = json.load(open(os.path.join(golden, "index.json")))["cases"]
    assert len(cases) >= 8
    for case in cases:
        b = api.Batch.load(os.path.join(golden, case["batch"]))
        want = np.load(os.path.join(golden, case["result"]))
        got = api.phase_batch(b)
        for k in got.ARRAYS:
            assert np.array_equal(getattr(got, k), want[k]), (case["name"], k)
