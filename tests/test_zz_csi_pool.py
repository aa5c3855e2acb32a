"""The drop-in on a BAM indexed with a CSI only: the forked pool of tests/test_zz_pool.py (BAM pre-pass thresholds,
`call` workers) on a CSI-only copy of the three-contig BAM writes what the reference's own `himut call` wrote for it
(tests/golden/cli_call.json).  Runs last (file name) because it spawns processes."""
import os

import pytest

import test_zz_pool as tz
from himut_b200 import bamdec, bamio


def _csi_only(monkeypatch):
    real = bamio.write_batches_bam
    written = []

    def write(path, contigs, *a, **k):
        real(path, contigs, *a, **dict(k, index="csi"))
        written.append(path)
    monkeypatch.setattr(bamio, "write_batches_bam", write)
    return written


def _check_written(written):
    assert written
    for path in written:
        assert os.path.exists(path + ".csi") and not os.path.exists(path + ".bai")
        assert bamdec.NativeBam(path).index_kind == "csi"


@pytest.mark.parametrize("name", ["plain", "phase"])
def test_forked_pool_on_a_csi_only_bam_cpu(tmp_path, monkeypatch, name):
    written = _csi_only(monkeypatch)
    got = tz._run(str(tmp_path), name, real=False)
    _check_written(written)
    tz._check(got, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["plain", "phase"])
def test_forked_pool_on_a_csi_only_bam_gpu(tmp_path, monkeypatch, name):
    written = _csi_only(monkeypatch)
    got = tz._run(str(tmp_path), name, real=True)
    _check_written(written)
    tz._check(got, name)
