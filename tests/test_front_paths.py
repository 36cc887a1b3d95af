"""-m gpu: the front end's two data placements on the same edge cases.

A batch runs its front end (projection, stage A, boundary set, stage B, filter, read order) in k_chain_front, one block per
chain out of shared memory, when every chain fits the block's budget, and in the kernel sequence of k_project.cuh otherwise.
Both call the same rule functions.  Each case runs twice: alone (every chain fits: k_chain_front) and with one chain
appended whose read x bubble mask alone exceeds the budget (the whole batch: the sequence).  Both runs must match the CPU
oracle, and the small chains' results must be the same in both."""
import copy
import functools
import json
import os

import numpy as np
import pytest

from ahsoka_b200 import api, synth
from tests.oracle_binding import oracle_phase
from tests.test_gpu_parity import deletion_allele_chain

pytestmark = pytest.mark.gpu

FRONT_BUDGET = 96 * 1024            # FR_SMEM_CAP (k_front.cuh): shared memory of one k_chain_front block


def _dims(b, c):
    B = int(b.bubble_off[c + 1] - b.bubble_off[c])
    R = int(b.read_off[c + 1] - b.read_off[c])
    NA = int(b.allele_off[b.bubble_off[c + 1]] - b.allele_off[b.bubble_off[c]])
    e0, e1 = int(b.entry_off[c]), int(b.entry_off[c + 1])
    return B, R, NA, e1 - e0, int(b.enode_off[e1] - b.enode_off[e0])


def _front_bytes_bound(b, c):
    """An upper bound of fr_layout(...).total of chain c: its arrays plus every alignment gap."""
    B, R, NA, NE, NEN = _dims(b, c)
    cap = 4
    while cap < 4 * NA:
        cap <<= 1
    return (NEN + 8) * 4 + cap * 8 + R * 62 + NA * 20 + (NE + 1) * 4 + B * 13 + R * B * 2 + 256


@functools.lru_cache(maxsize=None)
def _large_chain(ploidy):
    # ~375 reads x 200 bubbles: a 146 KB mask
    return synth.generate(synth.params(ploidy, 1, 0, 200, depth=30.0))


def _append(a, b):
    """a's chains followed by b's; b's node ids and chain ids are moved above a's."""
    cat = np.concatenate

    def off(x, y):
        return cat([x, y[1:] - y[0] + x[-1]])
    node = int(max(a.anode.max(initial=0), a.enode.max(initial=0))) + 1
    return api.Batch(a.ploidy, cat([a.chain_id, b.chain_id + int(a.chain_id.max(initial=0)) + 1]), off(a.bubble_off, b.bubble_off),
                     off(a.allele_off, b.allele_off), off(a.anode_off, b.anode_off), cat([a.anode, b.anode + node]),
                     cat([a.stage_a_order, b.stage_a_order]), off(a.read_off, b.read_off), off(a.entry_off, b.entry_off),
                     off(a.enode_off, b.enode_off), cat([a.enode, b.enode + node]), cat([a.entry_read, b.entry_read]),
                     cat([a.entry_identity, b.entry_identity]))


def _with_large_chain(small):
    for c in range(small.n_chains):
        assert _front_bytes_bound(small, c) <= FRONT_BUDGET, f"chain {c} does not fit k_chain_front"
    big = _large_chain(int(small.ploidy))
    B, R = _dims(big, 0)[:2]
    assert R * B * 2 > FRONT_BUDGET, "the appended chain fits k_chain_front"
    return _append(small, big)


def _first_chains(res, C):
    """Every result array restricted to the first C chains."""
    nr = int(res.read_off[C])
    nc = int(res.cell_off[nr])
    npos = int(res.pos_off[C])
    cut = {"status": C, "n_clusters": C, "dp_cost": C, "maxpos": C, "read_off": C + 1, "pos_off": C + 1,
           "read_id": nr, "read_mapq": nr, "read_cluster": nr, "cell_off": nr + 1, "cell_pos": nc, "cell_allele": nc,
           "pos": npos, "path": npos * res.ploidy, "hap_allele": npos * res.ploidy}
    assert set(cut) == set(res.ARRAYS)
    return {k: getattr(res, k)[:n] for k, n in cut.items()}


def _phase_checked(batch):
    got = api.phase_batch(batch)
    bad = got.diff(oracle_phase(batch))
    assert not bad, f"GPU differs from oracle in {bad}"
    return got


def _both_paths(small):
    joint_batch = _with_large_chain(small)
    alone = _phase_checked(small)
    joint = _phase_checked(joint_batch)
    a, j = _first_chains(alone, small.n_chains), _first_chains(joint, small.n_chains)
    bad = [k for k in a if not np.array_equal(a[k], j[k])]
    assert not bad, f"the small chains' results depend on the front-end path in {bad}"
    return alone


def test_deletion_allele_chain():
    assert _both_paths(deletion_allele_chain()).status[0] == 0


@pytest.mark.parametrize("p", [
    pytest.param(synth.params(2, 60, 1, 3, min_len=1, depth=12.0, seed=11), id="tiny_and_trivial_chains"),
    pytest.param(synth.params(2, 50, 1, 10, depth=2.0, seed=5), id="low_depth_empty_chains"),
    pytest.param(synth.params(2, 30, 1, 30, depth=25.0, dup_lines=300, seed=21), id="multiline_reads"),
    pytest.param(synth.params(2, 20, 1, 20, depth=30.0, max_alleles=6, seed=51), id="four_bit_codes_diploid"),
    pytest.param(synth.params(4, 10, 1, 30, depth=60.0, max_alleles=12, seed=77), id="four_bit_codes_tetraploid"),
    pytest.param(synth.params(5, 12, 1, 30, depth=50.0, seed=51), id="ploidy5"),
    pytest.param(synth.params(6, 12, 1, 30, depth=60.0, seed=61), id="ploidy6"),
])
def test_synthetic(p):
    _both_paths(synth.generate(p))


def _golden_cases():
    golden = os.path.join(api.ROOT, "tests", "golden")
    return [os.path.join(golden, c["batch"]) for c in json.load(open(os.path.join(golden, "index.json")))["cases"]]


# dip_200_reads (one chain of 200 reads) is above the budget by itself: test_committed_golden_fixtures runs it in the sequence
@pytest.mark.parametrize("path", [p for p in _golden_cases() if "dip_200_reads" not in p], ids=os.path.basename)
def test_golden_fixture(path):
    _both_paths(api.Batch.load(path))


def _malformed(b, kind):
    c = copy.copy(b)
    if kind == "entry_read_out_of_range":
        c.entry_read = b.entry_read.copy(); c.entry_read[3] = 10 ** 6
    elif kind == "allele_off_not_monotone":
        c.allele_off = b.allele_off.copy(); c.allele_off[5], c.allele_off[6] = b.allele_off[6] + 1, b.allele_off[5]
    elif kind == "stage_a_order_repeats":
        c.stage_a_order = b.stage_a_order.copy(); c.stage_a_order[1] = b.stage_a_order[0]
    elif kind == "stage_a_order_out_of_range":
        c.stage_a_order = b.stage_a_order.copy(); c.stage_a_order[1] = 10 ** 6
    else:
        assert kind == "enode_off_not_monotone"
        c.enode_off = b.enode_off.copy(); c.enode_off[2] = b.enode_off[3] + 5
    return c


@pytest.mark.parametrize("kind,message", [("entry_read_out_of_range", "entry_read"), ("allele_off_not_monotone", "monotone"),
                                          ("stage_a_order_repeats", "permutation"), ("stage_a_order_out_of_range", "permutation"),
                                          ("enode_off_not_monotone", "monotone")])
def test_malformed_batch_is_rejected(kind, message):
    # the errors sit in the small chains; with the large chain appended the sequence reports them
    small = synth.generate(synth.params(2, 8, 1, 12, depth=20.0, seed=91))
    joint = _with_large_chain(small)
    for b in (small, joint):
        with pytest.raises(RuntimeError, match=message):
            api.phase_batch(_malformed(b, kind))
    assert not api.phase_batch(joint).diff(oracle_phase(joint))          # the library is still usable afterwards
