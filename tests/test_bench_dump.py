"""bench.py --dump-outputs: the files depend on the records alone, not on what the result buffers held after each query's n records."""
import os

import numpy as np

import bench

N = np.array([3, 0, 2, 4], np.int32)


def _records(leftover):
    key = np.arange(16, dtype=np.int64).reshape(4, 4) + 100
    score = np.linspace(1, 2, 16, dtype=np.float32).reshape(4, 4)
    tie = np.arange(16, dtype=np.uint8).reshape(4, 4)
    unwritten = np.arange(4)[None, :] >= N[:, None]
    for a in (key, score, tie):          # the library leaves these slots as the allocator handed them over
        a.view(np.uint8).reshape(4, -1)[np.repeat(unwritten, a.itemsize, axis=1)] = leftover
    return dict(doc_key=key, score=score, tie=tie, n=N.copy(), total_candidates=N * 3, status=np.zeros(4, np.int32))


def test_dump_outputs_pads_unwritten_slots(tmp_path):
    for leftover in (0x00, 0xFF):        # 0xFF..FF is a NaN bit pattern in `score`
        bench.dump_outputs(str(tmp_path / str(leftover)), _records(leftover))
    names = sorted(os.listdir(tmp_path / "0"))
    assert names == sorted(os.listdir(tmp_path / "255")) == sorted(k + ".npy" for k in _records(0))
    for f in names:
        a, b = np.load(tmp_path / "0" / f), np.load(tmp_path / "255" / f)
        assert a.dtype == b.dtype and a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    key, score = np.load(tmp_path / "255" / "doc_key.npy"), np.load(tmp_path / "255" / "score.npy")
    written = np.arange(4)[None, :] < N[:, None]
    assert np.array_equal(key[written], (np.arange(16).reshape(4, 4) + 100)[written])
    assert (key[~written] == -1).all() and (score[~written] == 0).all()
