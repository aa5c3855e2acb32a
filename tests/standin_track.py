"""Test infrastructure: the oracle stand-in of lib.Context (tests/standin.py) that also answers the callable-base track
(Context.callable_track / last_callable_runs) from tests/track_oracle.py, so the drop-in's track writer is pinned on
the CPU."""
import numpy as np

import standin
import track_oracle
from himut_b200 import abi


class TrackOracleContext(standin.OracleContext):
    def __init__(self):
        super().__init__()
        self.track = False
        self._runs = np.zeros(0, abi.RUN_DTYPE)

    def callable_track(self, on=True):
        self.track = bool(on)

    def normcounts_chunks(self, refseq, table):
        self._runs = np.zeros(0, abi.RUN_DTYPE)
        if not self.track:
            return super().normcounts_chunks(refseq, table)
        self._seen = np.zeros(int(self.batch.qname_id.max()) + 1 if self.batch.n_reads else 1, np.uint8)
        ref = refseq.encode() if isinstance(refseq, str) else refseq
        *res, self._runs = track_oracle.normcounts_chunks_track(self.params, self.batch, ref, table, self.common, self.pon,
                                                                self.phase, qseen=self._seen)
        return tuple(res)

    def last_callable_runs(self):
        return self._runs
