"""The callable-base track of `himut normcounts` on the device (HM_OPT_CALLABLE_TRACK): the runs k_track_count /
k_track_emit build from what k_norm_bits, the exact pass and k_norm_tiles_tma store equal the oracle's record for
record on every route, and switching the track on changes none of the tallies.  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest

import cases
import test_genotype_edges as tge
import test_norm_cert
from himut_b200 import abi, gtmodel, normcounts, synth
from test_callable_track import NORM_CASES, check_runs_shape, oracle_track, overlap_case, run_sums, tracked, tri_bins
from test_gpu_csi import LONG, N, _base, long_contig  # noqa: F401  (module fixture)
from test_gpu_fullsize import CONTIG, big  # noqa: F401  (module fixture)

pytestmark = pytest.mark.gpu


def track_on_off(ctx, ref, table):
    """normcounts_chunks with the track off, then on -> (tallies, runs); the tallies must be bit-identical"""
    off = ctx.normcounts_chunks(ref, table)
    assert ctx.last_callable_runs().size == 0
    ctx.callable_track(True)
    try:
        on = ctx.normcounts_chunks(ref, table)
        runs = ctx.last_callable_runs()
    finally:
        ctx.callable_track(False)
    for a, b in zip(off[:3], on[:3]):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    assert off[3] == on[3]
    return on, runs


def case_on_device(ctx, c):
    ctx.set_params(c["params"])
    ctx.set_site_sets(c["common"], c["pon"])
    if c["phase"] is not None:
        ctx.set_phase_sets(c["phase"])
    ctx.upload(c["batch"])
    return track_on_off(ctx, c["ref"].encode(), c["chunk_table"])


def same_as_oracle(ctx, c):
    g, runs = case_on_device(ctx, c)
    o = oracle_track(c)
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and list(g[2]) == list(o[2])
    check_runs_shape(runs, c["chunk_table"])
    assert runs.size == o[4].size and np.array_equal(runs, o[4]), _first_diff(runs, o[4])
    return g, runs


def _first_diff(a, b):
    for i, (x, y) in enumerate(zip(a.tolist(), b.tolist())):
        if x != y:
            return "run %d: device %r, oracle %r" % (i, x, y)
    return "lengths %d vs %d" % (a.size, b.size)


@pytest.mark.parametrize("name", NORM_CASES)
def test_golden_cases(ctx, name):
    _g, runs = same_as_oracle(ctx, cases.build_case(name))
    assert runs.size > 100


@pytest.mark.parametrize("seed", list(cases.RANDOM_NORM_SEEDS) + list(cases.RANDOM_LONG_NORM_SEEDS))
def test_random_sweep_norm(ctx, seed):
    c = cases.random_case("norm", seed)
    if c is None:
        pytest.skip("no phase set")
    same_as_oracle(ctx, c)


@pytest.mark.parametrize("seed", list(cases.RANDOM_CALL_SEEDS) + list(cases.RANDOM_LONG_CALL_SEEDS) + list(cases.RANDOM_DUPNAME_CALL_SEEDS))
def test_random_sweep_call_seeds(ctx, seed):
    c = cases.random_case("call", seed)
    if c is None:
        pytest.skip("no phase set")
    same_as_oracle(ctx, c)


@pytest.mark.parametrize("prior,min_gq,min_bq", [(1e-3, 20, 20), (1e-3, 60, 60), (5e-4, 99, 93)])
def test_pure_columns_at_the_certificate_edge(ctx, prior, min_gq, min_bq):
    """the columns of test_genotype_edges at thr[n] - 1, thr[n], thr[n] + 1: certified ones are stored by k_norm_bits,
    the others by k_norm_reduce"""
    cert = test_norm_cert.make_cert(prior, min_gq, min_bq)
    depths = sorted({max(cert["n_min"], 1), cert["n_min"] + 1, 2, 5, 17, 40, 100, 200, 255})
    b, ref, n_yes, n_no, _touched = tge.pure_edge_batch(cert, min_bq, depths)
    p = gtmodel.make_params(**cases.call_args(min_qv=0, min_mapq=0, qlen_lower_limit=0, qlen_upper_limit=1000,
                                              min_sequence_identity=0.0, min_trim=0.0, md_threshold=1000,
                                              germline_snv_prior=prior, min_gq=min_gq, min_bq=min_bq))
    c = dict(params=p, batch=b, ref=ref.decode(), chunk_table=b.chunk_table([(0, len(ref))]), common=None, pon=None, phase=None)
    same_as_oracle(ctx, c)
    assert "k_norm_bits" in tge.kernels(ctx)
    assert ctx.last_norm_exact_sites() >= n_no


def _synth_case(d, p, loci):
    return dict(params=p, batch=d.batch, ref=d.ref.decode(), chunk_table=d.batch.chunk_table(loci), common=None, pon=None, phase=None)


def test_deep_pileup(ctx):
    """400x: more than 255 reads per span, so every position goes to the exact pass (values above 255)"""
    d = synth.generate(30_000, seed=34, depth=400.0)
    c = _synth_case(d, gtmodel.make_params(**cases.call_args(md_threshold=1000)), [(0, 12_345), (12_345, 30_000)])
    _g, runs = same_as_oracle(ctx, c)
    assert ctx.last_norm_exact_sites() > 25_000
    assert int(runs["value"].max()) > 255


def test_overlapping_chunk_list(ctx):
    d, p, loci, _table = overlap_case()
    same_as_oracle(ctx, _synth_case(d, p, loci))


@pytest.mark.parametrize("loci", [[(0, 40_000), (40_000, 100_000)], [(-500, 40_000), (30_000, 100_000)]])
def test_single_pass_route(ctx, loci):
    """min_bq 0 lies outside the certified domain (and so does a chunk that starts below 0): k_norm_tiles_tma stores"""
    d = synth.generate(100_000, seed=37)
    c = _synth_case(d, gtmodel.make_params(**cases.call_args(min_bq=0)), loci)
    _g, runs = same_as_oracle(ctx, c)
    assert "k_norm_tiles_tma" in tge.kernels(ctx)
    assert ctx.last_norm_exact_sites() == 0
    assert runs.size > 1000


def test_long_contig_host_and_device_decoders(ctx, long_contig):
    """chrL of LN 2^31 - 1 behind a CSI: normcounts_region's runs are the same on both decoders, and each stretch's
    runs are the oracle's runs of the unshifted reads, moved by the stretch's offset; the last run ends at 2^31 - 1"""
    path, loci, ref, _table, _sets, offs = long_contig
    p = gtmodel.make_params(**gtmodel.DEFAULT_CALL_ARGS)
    out = {}
    for decode in ("device", "host"):
        ctx.set_params(p)
        ctx.set_site_sets()
        out[decode] = normcounts.normcounts_region(ctx, path, "chrL", ref, loci, None, decode=decode, callable_track=True)
        plain = normcounts.normcounts_region(ctx, path, "chrL", ref, loci, None, decode=decode)
        for a, b in zip(plain, out[decode][:5]):
            assert np.array_equal(np.asarray(a), np.asarray(b))
    runs = out["device"][5]
    assert np.array_equal(runs, out["host"][5])
    d, local, _ph, k = _base(False, long_contig)
    base = tracked(p, d.batch, bytes(d.ref), d.batch.chunk_table(local))[4]
    assert base.size > 100
    for j, off in enumerate(offs):
        part = runs[(runs["chunk"] >= j * k) & (runs["chunk"] < (j + 1) * k)].copy()
        moved = base.copy()
        moved["chunk"] += j * k
        moved["start"] += off
        moved["end"] += off
        assert np.array_equal(part, moved), (off, _first_diff(part, moved))
    assert runs.size == 3 * base.size
    assert int(runs["end"].max()) <= LONG and int(runs["start"].max()) > 2**31 - N


def test_full_contig(ctx, big):
    """the 64 Mb contig, every chunk: the runs summed per bin are that call's ref_tri / ccs_tri, their total log[13]"""
    d, p, chunks = big
    ctx.set_params(p)
    ctx.set_site_sets()
    ctx.upload(d.batch)
    g, runs = track_on_off(ctx, d.ref, chunks)
    check_runs_shape(runs, chunks)
    r_ref, r_ccs, total = run_sums(runs, tri_bins(d.ref))
    assert np.array_equal(r_ref, g[1]) and np.array_equal(r_ccs, g[0]) and total == int(g[2][13])
    assert set(np.unique(runs["chunk"]).tolist()) == set(range(len(chunks)))
    assert runs.size > 1_000_000 and int(r_ref.sum()) > CONTIG // 2
    # a second call on the context (buffers reused) gives the same runs
    ctx.callable_track(True)
    try:
        ctx.normcounts_chunks(d.ref, chunks[:7])
        again = ctx.normcounts_chunks(d.ref, chunks)
        assert np.array_equal(ctx.last_callable_runs(), runs)
        assert all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(again[:3], g[:3]))
    finally:
        ctx.callable_track(False)
