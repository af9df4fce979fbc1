"""The general BQSR gather path on the reads that neither the count kernel nor bqsr_chunk_kernel<false> take: reads hit by more
than 4 known-site ranges (their skip mask is a 512-bit word) and reads longer than --max-cycle.  Bit-exact against the oracle
for output order, FLAG, table counters, EmpiricalQuality, report text and QUAL bytes, with the tables built for the test's
own --max-cycle."""
import numpy as np
import pytest

from elprep_b200 import synth
from util import gpu_pipeline, oracle_pipeline, oracle_tables_dense

pytestmark = pytest.mark.gpu

SMALL = [("chr20", 600_000), ("chr21", 300_000), ("chrM", 16_569)]


def _compare(g, o, max_cycle, qual=True):
    assert np.array_equal(g["perm"], o["perm"]), "output order differs"
    assert np.array_equal(g["flag"], o["flag"]), "FLAG differs"
    assert np.array_equal(g["qual_off"], o["qual_off"])
    d, e = oracle_tables_dense(o["tables"], max_cycle)
    assert np.array_equal(g["tables"], d), "BQSR table counters differ"
    assert np.array_equal(g["emp"], e), "EmpiricalQuality differs"
    assert g["report"] == o["report"], "recalibration report text differs"
    if qual:
        assert np.array_equal(g["qual"], o["qual"]), "QUAL bytes differ"


def _sites_per_read(b, sites):
    """known-site ranges inside the aligned reference span of every mapped read (0 for the others)"""
    n = b.n
    ops, lens = b.cigar & 15, (b.cigar >> 4).astype(np.int64)
    read_of = np.repeat(np.arange(n), np.diff(b.cigar_off.astype(np.int64)))
    span = np.bincount(read_of, weights=lens * np.isin(ops, (0, 2, 3, 7, 8)), minlength=n).astype(np.int64)
    out = np.zeros(n, np.int64)
    for ci, s in enumerate(sites):
        k = np.nonzero((b.refid == ci) & ((b.flag & 4) == 0) & (span > 0))[0]
        lo, hi = b.pos[k].astype(np.int64), b.pos[k].astype(np.int64) + span[k] - 1
        out[k] = np.searchsorted(s[:, 0], hi, side="right") - np.searchsorted(s[:, 1], lo, side="left")
    return out


@pytest.mark.parametrize("wide_quals", [False, True])
def test_dense_known_sites(wide_quals):
    """a 1-bp known site every 23 bp: a 150-base read holds 6-7 of them, so its skip mask takes the 512-bit overflow form"""
    w = synth.make_workload(1_500, SMALL, seed=61, wide_quals=wide_quals)
    w.sites = [np.repeat(np.arange(1, ln + 1, 23, dtype=np.int32)[:, None], 2, axis=1) for _, ln in SMALL]
    assert int((_sites_per_read(w.batch, w.sites) > 4).sum()) > 1000
    _compare(gpu_pipeline(w, n_batches=2), oracle_pipeline(w), 500)


def _long_reads(mask):
    """150-base reads under --max-cycle 100; with `mask`, every base whose cycle exceeds 100 gets QUAL 2 (never counted).  The
    cycle magnitude of stored base i is i+1 (forward) or L-i (reversed); clipping never makes it larger."""
    w = synth.make_workload(1_500, SMALL, seed=62, L=150)
    b = w.batch
    assert int(b.lseq.max()) == 150
    if mask:
        qo = b.qual_off.astype(np.int64)
        for r in range(b.n):
            L = int(b.lseq[r])
            i = np.arange(L)
            cyc = L - i if b.flag[r] & 0x10 else i + 1
            b.qual[qo[r]:qo[r] + L][cyc > 100] = 2
    return w


def test_reads_longer_than_max_cycle():
    """gather and apply both succeed; QUAL bytes are not compared: bqsr_apply_kernel leaves every base of a 16-base chunk that
    also holds a cycle beyond --max-cycle unrecalibrated, where the oracle recalibrates the chunk's other bases"""
    w = _long_reads(mask=True)
    _compare(gpu_pipeline(w, max_cycle=100), oracle_pipeline(w, max_cycle=100), 100, qual=False)


def test_cycle_beyond_max_cycle_is_an_error():
    from elprep_b200 import device
    w = _long_reads(mask=False)
    with pytest.raises(ValueError, match="cycle value exceeds maximum cycle value"):
        oracle_pipeline(w, max_cycle=100)
    with pytest.raises(device.ElprepError) as ei:
        gpu_pipeline(w, max_cycle=100)
    assert ei.value.code == -12 and "cycle value exceeds maximum cycle value" in str(ei.value)
