"""CPU-side checks of the many-reference sharded path's host pieces: the record layout muse_merge_partials_many merges."""
import numpy as np

import muse_b200 as mb


def test_multi_records_layout():
    sc = np.array([[0.9, 0.8, 0.0], [0.0, 0.0, 0.0], [0.7, 0.0, 0.0]])
    lg = np.array([[3, -4, 0], [0, 0, 0], [-1, 0, 0]], dtype=np.int64)
    ix = np.array([[1000012, 5, 0], [0, 0, 0], [77, 0, 0]], dtype=np.int64)
    rec = mb.multi_records(sc, lg, ix, np.array([2, -1, 1]))
    assert rec.dtype == mb.PARTIAL_DTYPE and rec.shape == (3, 3) and rec.itemsize == 32
    np.testing.assert_array_equal(rec["flags"], [[0, 0, 1], [1, 1, 1], [0, 1, 1]])     # std-zero row: all padding
    np.testing.assert_array_equal(rec["series_idx"][0, :2], [1000012, 5])
    np.testing.assert_array_equal(rec["group_key"][0, :2], [1000012, 5])
    np.testing.assert_array_equal(rec["lag"][0, :2], [3, -4])
    np.testing.assert_array_equal(rec["score"][2, :1], [0.7])
    # the host merge reads the same records: the valid ones of row 0 and row 2 together, best first
    s, l, i = mb.merge_partials(np.concatenate([rec[0], rec[2]]), 10, 3, 0.0)
    np.testing.assert_array_equal(i, [1000012, 5, 77])
    np.testing.assert_array_equal(l, [3, -4, -1])
