"""The decode choice of the normcounts worker (normcounts.normcounts_region) and the phase edges (phaselib.edge_table)
on the CPU: with the oracle stand-in context, which has no device decoder, decode="device" falls back to the host
decoder and still reproduces the reference's outputs; a bad decode value is refused; "auto" keeps small inputs on the
host decoder (worker.choose_decode)."""
import json
import os

import numpy as np
import pytest

import cases
import parity
from himut_b200 import bamdec, normcounts, phaselib, worker
from standin import OracleContext
from test_worker_host import _inputs, mk_edges, octx  # noqa: F401  (octx: the stand-in fixture)


def _norm_region(ctx, c, tmp_path, decode):
    bam, common, pon = _inputs(c, tmp_path)
    ctx.set_params(c["params"])
    ctx.set_site_sets(c["common"], c["pon"])
    if c["phase"] is not None:
        ctx.set_phase_sets(c["phase"])
    loci = [(cases.CHROM, s, e) for s, e in c["chunks"]]
    return normcounts.normcounts_region(ctx, bam, cases.CHROM, c["ref"].encode(), loci, c["phase_sets"], decode=decode)


def _check_norm(got, name):
    e = parity.load_golden(name)["expected"]
    ccs, rt, log, ties, num_ccs = got
    if ties:
        pytest.skip("%d alt ties: the reference's own result depends on PYTHONHASHSEED here" % ties)
    assert np.array_equal(ccs, parity.tri_dict_to_bins(e["ccs_tri2count"]))
    assert np.array_equal(rt, parity.tri_dict_to_bins(e["ref_tri2count"]))
    assert [int(v) for v in log] == e["log"] and num_ccs == e["log"][0]


@pytest.mark.parametrize("name", ["norm_basic", "norm_phase", "norm_adversarial"])
def test_normcounts_region_device_falls_back_to_the_host(octx, name, tmp_path, monkeypatch):
    if name == "norm_adversarial":
        monkeypatch.setattr(worker, "GROUP_SPAN", 1200)
    c = cases.build_case(name)
    before = octx.uploads
    got = _norm_region(octx, c, tmp_path, "device")
    assert octx.uploads > before
    _check_norm(got, name)


def _edges(ctx, tmp_path, name, decode):
    """-> (the table's non-empty (i, j, counts) rows, hetSNPs numbered as get_edges numbers them; the reference's)"""
    batch, hetsnp_lst, h2i, n, min_bq, min_mapq = mk_edges.inputs(name)
    path = str(tmp_path / "e.bam")
    bamdec.write_batch_bam(path, "chr1", n, batch)
    hpos = np.array([h[0] for h in hetsnp_lst], np.int32)
    href = np.array([phaselib.BASE2CODE[h[1]] for h in hetsnp_lst], np.uint8)
    hidx = [h2i[h] for h in hetsnp_lst]
    table = phaselib.edge_table(ctx, path, "chr1", hpos, href, min_bq, min_mapq, decode=decode)
    a, d = np.nonzero(table.any(axis=2))
    rows = sorted([hidx[x], hidx[x + y + 1]] + [int(v) for v in table[x, y]] for x, y in zip(a.tolist(), d.tolist()))
    want = json.load(open(os.path.join(cases.GOLDEN_DIR, "edges.json")))["expected"][name]
    return rows, sorted(want)


@pytest.mark.parametrize("name", ["plain", "bq0_counts_deletions"])
def test_edge_table_device_falls_back_to_the_host(octx, tmp_path, monkeypatch, name):
    monkeypatch.setattr(worker, "GROUP_SPAN", 37_000)
    rows, want = _edges(octx, tmp_path, name, "device")
    assert rows == want


def test_bad_decode_value_is_refused(octx, tmp_path):
    c = cases.build_case("norm_basic")
    with pytest.raises(ValueError):
        _norm_region(octx, c, tmp_path, "gpu")
    with pytest.raises(ValueError):
        _edges(octx, tmp_path, "plain", "fast")
    with pytest.raises(ValueError):
        worker.choose_decode("Device", octx, None, "chr1", 0, 1, 1, 1)


class _DecodingStandIn(OracleContext):
    """a stand-in that claims the device decoder: "auto" must not take it for small inputs"""

    def decode_region(self, *a, **k):
        raise AssertionError("decode_region called below the threshold")


def test_auto_stays_on_the_host_below_the_threshold(tmp_path, monkeypatch):
    ctx = _DecodingStandIn()
    monkeypatch.setattr(worker, "context", lambda: ctx)
    plain = worker.RegionSource.batch
    monkeypatch.setattr(worker.RegionSource, "batch",
                        lambda self, chrom, loci, phase_sets=None, seq=True, **kw: plain(self, chrom, loci, phase_sets, seq=True, **kw))
    c = cases.build_case("norm_basic")
    _check_norm(_norm_region(ctx, c, tmp_path, "auto"), "norm_basic")
    rows, want = _edges(ctx, tmp_path, "plain", "auto")
    assert rows == want
    with pytest.raises(AssertionError):  # the stand-in is asked when the device decoder is forced
        _norm_region(ctx, c, tmp_path, "device")


class _Plan:
    def __init__(self, comp_bytes):
        self.comp_bytes = comp_bytes


class _Reader:
    def __init__(self, comp_bytes, has_index=True):
        self.comp_bytes, self.has_index = comp_bytes, has_index

    def plan(self, chrom, lo, hi):
        return _Plan(self.comp_bytes)


def test_choose_decode():
    dev, host = _DecodingStandIn(), OracleContext()
    m = normcounts.DEVICE_DECODE_MIN_BYTES
    assert worker.choose_decode("auto", dev, _Reader(3 * m), "chr1", 0, 10, 3, m) == "device"
    assert worker.choose_decode("auto", dev, _Reader(3 * m - 1), "chr1", 0, 10, 3, m) == "host"
    assert worker.choose_decode("auto", dev, _Reader(3 * m), "chr1", None, None, 3, m) == "host"  # no chunks
    assert worker.choose_decode("auto", dev, _Reader(3 * m, has_index=False), "chr1", 0, 10, 3, m) == "host"
    assert worker.choose_decode("device", dev, _Reader(0), "chr1", 0, 10, 1, m) == "device"
    assert worker.choose_decode("device", dev, _Reader(0, has_index=False), "chr1", 0, 10, 1, m) == "host"
    assert worker.choose_decode("device", host, _Reader(3 * m), "chr1", 0, 10, 1, m) == "host"
    assert worker.choose_decode("host", dev, _Reader(3 * m), "chr1", 0, 10, 1, m) == "host"
