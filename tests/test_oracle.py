"""The oracle against every expectation the reference's own tests hold for the
Batch.Run path (tests/golden/reference_kats.json, transcribed from the Go tests).
CPU only."""
import math

import numpy as np
import pytest

from oracle import muse_oracle as mo


def test_next_pow_of2(kats):
    # xcorr_test.go:20-38
    for val, want in kats["next_pow_of2"]["cases"]:
        assert mo.next_pow_of2(val) == want
    for N, n in [(480, 512), (1440, 2048), (10080, 16384), (12, 16), (8, 8), (5, 8)]:
        assert mo.next_pow_of2(float(N)) == n


def test_z_normalize(kats):
    # xcorr_test.go:40-61 -- sum of squares == N-1 (sample std)
    k = kats["z_normalize"]
    for ts in k["cases"]:
        z = mo.z_normalize(np.array(ts, dtype=np.float64))
        assert abs(float(np.sum(z * z)) - (len(ts) - 1)) <= k["tol"]
    assert mo.z_normalize(np.full(7, 3.0)) is None


def test_zero_pad(kats):
    # xcorr_test.go:63-85
    for c in kats["zero_pad"]["cases"]:
        got = mo.zero_pad(np.array(c["x"], dtype=np.float64), c["n"])
        assert got.tolist() == [float(v) for v in c["expected"]]


def _check_cc(cc, lag, mv, c, tol):
    if c["cc"] is None:
        assert cc is None
    else:
        assert cc is not None and np.max(np.abs(cc - np.array(c["cc"], dtype=np.float64))) <= tol
    assert lag == c["lag"]
    if c["sign"] > 0:
        assert mv > 0
    elif c["sign"] < 0:
        assert mv < 0
    else:
        assert mv == 0


def test_x_corr(kats):
    # xcorr_test.go:86-202
    k = kats["x_corr"]
    for c in k["cases"]:
        cc, lag, mv = mo.x_corr(c["x"], c["y"], len(c["x"]), c["normalize"])
        _check_cc(cc, lag, mv, c, k["tol"])


def test_x_corr_with_x(kats):
    # xcorr_test.go:204-286 (n = 5, not a power of two)
    k = kats["x_corr_with_x"]
    for c in k["cases"]:
        n = len(c["x"])
        x = mo.z_normalize(np.array(c["x"], dtype=np.float64))
        x = x * (1.0 / (len(x) - 1))
        X = np.fft.rfft(mo.zero_pad(x, n))
        cc, lag, mv = mo.x_corr_with_x(X, c["y"], n)
        _check_cc(cc, lag, mv, c, k["tol"])


def _mk(entries):
    return [mo.Series(e["y"], mo.Labels(e["labels"])) for e in entries]


def _compare_scores(scores, expected, tol):
    # muse_test.go:11-39 compareScores, with the F4 tie-lag allowance
    assert len(scores) == len(expected)
    for got, want in zip(scores, expected):
        assert got.Lag in want.get("tie_lags", [want["lag"]])
        assert abs(got.PercentScore - want["score"]) <= tol
        assert got.Labels.labels == want["labels"]


@pytest.mark.parametrize("name", ["batch_run_simple", "batch_run_multi_dimensional"])
def test_batch_run_kats(kats, name):
    # muse_batch_test.go:9-82
    k = kats[name]
    ref = mo.Series(k["ref"]["y"], mo.Labels(k["ref"]["labels"]))
    g = mo.Group("targets")
    g.Add(*_mk(k["comp"]))
    r = k["results"]
    b = mo.Batch(ref, g, mo.Results(r["max_lag"], r["top_n"], r["threshold"], r["sign_filter"]),
                 k["concurrency"])
    b.Run(list(k["group_by"]))
    scores, _ = b.Results.Fetch()
    _compare_scores(scores, k["expected"], k["score_tol"])


def test_batch_run_fp64_values(kats):
    # SURVEY section 8c: six-digit fp64 values of the two KATs
    k = kats["batch_run_simple"]
    s, l = mo.score_series_batch(k["ref"]["y"], np.array([e["y"] for e in k["comp"]], dtype=float))
    np.testing.assert_allclose(s, [1.0, 0.928571, 0.732941, 0.753576, 0.0], rtol=0, atol=6e-7)
    assert l[0] == 0 and l[1] == 0 and l[2] == 2 and l[3] in (-3, -2) and l[4] == 0
    k = kats["batch_run_multi_dimensional"]
    s, l = mo.score_series_batch(k["ref"]["y"], np.array([e["y"] for e in k["comp"]], dtype=float))
    np.testing.assert_allclose(s, [1.0, 0.169031, 0.976187, 0.247841, 0.759257, 0.718865],
                               rtol=0, atol=6e-7)


def test_batch_run_with_larger_group(kats):
    # muse_batch_test.go:83-102
    k = kats["batch_run_with_larger_group"]
    ref = mo.Series(k["ref"]["y"], mo.Labels(k["ref"]["labels"]))
    g = mo.Group("targets")
    g.Add(*_mk(k["comp"]))
    with pytest.raises(ValueError):
        mo.Batch(ref, g, mo.Results(10, 20, 0, mo.SIGN_FILTER_ANY), 1)


def test_batch_rejects_constant_reference():
    # muse_batch.go:38-41
    g = mo.Group("t")
    g.Add(mo.Series([1.0, 2.0, 3.0, 4.0], mo.Labels({"a": "b"})))
    with pytest.raises(ValueError):
        mo.Batch(mo.Series([2.0, 2.0, 2.0, 2.0]), g, mo.Results(1, 1, 0, 0), 1)


def test_muse_run_kats(kats):
    # muse_test.go:41-142
    k = kats["muse_run_simple"]
    for key, sf in (("expected_any", mo.SIGN_FILTER_ANY), ("expected_pos", mo.SIGN_FILTER_POS),
                    ("expected_neg", mo.SIGN_FILTER_NEG)):
        ref = mo.Series(k["ref"]["y"], mo.Labels(k["ref"]["labels"]))
        m = mo.Muse(ref, mo.Results(k["results"]["max_lag"], k["results"]["top_n"],
                                    k["results"]["threshold"], sf))
        for s in _mk(k["comp"]):
            m.Run([s])
        scores, _ = m.Results.Fetch()
        _compare_scores(scores, k[key], k["score_tol"])
    # TestRunNoInput
    m = mo.Muse(mo.Series(k["ref"]["y"], mo.Labels(k["ref"]["labels"])), mo.Results(10, 20, 0, 0))
    assert m.Run([]) is None
    scores, mean = m.Results.Fetch()
    assert scores == [] and math.isnan(mean)


def test_group_and_labels(kats):
    # group_test.go:5-113, labels_test.go:5-72, series_test.go:12-100
    k = kats["group_add"]
    g = mo.Group("test")
    for c in k["cases"]:
        s = mo.Series(k["y"], mo.Labels(c["labels"]))
        if c["expect_error"]:
            with pytest.raises(ValueError):
                g.Add(s)
        else:
            g.Add(s)
    k = kats["index_label_values"]
    g = mo.Group("test")
    for l in k["labels"]:
        g.Add(mo.Series(k["y"], mo.Labels(l)))
    for names, want in k["cases"]:
        assert len(g.indexLabelValues(list(names))) == want
    for labels, want in k["filter_cases"]:
        lab = mo.Labels(labels)
        g.indexLabelValues(list(lab.Keys()))
        assert len(g.FilterByLabelValues(lab)) == want
    for c in kats["labels_id"]["cases"]:
        gb = list(c["group_by"]) if c["group_by"] else None
        assert mo.Labels(c["labels"]).ID(gb) == c["expected"]
    k = kats["series"]
    assert mo.Series([0.1, 0.2, 0.3], None).Labels().Keys() == [k["default_label"]]
    for c in k["uid_cases"]:
        assert mo.Series([0.1], mo.Labels(c["labels"])).UID() == c["expected"]
    for c in k["key_cases"]:
        assert mo.Series([0.1], mo.Labels(c["labels"])).Labels().Keys() == c["expected"]
    # group.go:45-51 length mismatch, :33-36 handled by NewSeries default label
    g = mo.Group("len")
    g.Add(mo.Series([1.0, 2.0], mo.Labels({"a": "1"})))
    with pytest.raises(ValueError):
        g.Add(mo.Series([1.0, 2.0, 3.0], mo.Labels({"a": "2"})))


def test_results_heap_semantics():
    # results.go:55-87: cap TopN, strict-greater replace, descending Fetch, NaN mean when empty
    r = mo.Results(5, 3, 0.2, mo.SIGN_FILTER_ANY)
    lab = mo.Labels({"a": "b"})
    for sc, lag in [(0.5, 0), (0.9, 1), (0.1, 0), (0.7, 6), (0.3, -5), (0.6, 2), (0.5, 3)]:
        r.Update(mo.Score(lab, lag, sc))
    r.Update(mo.Score(None, 0, 1.0))                       # nil labels ignored
    out, mean = r.Fetch()
    assert [s.PercentScore for s in out] == [0.9, 0.6, 0.5]
    assert out[2].Lag == 0                                  # equal score does not replace the root
    assert abs(mean - (0.9 + 0.6 + 0.5) / 3) < 1e-15
    out, mean = r.Fetch()
    assert out == [] and math.isnan(mean)


def test_array_form_matches_object_form():
    rng = np.random.default_rng(7)
    N, S = 100, 60
    ref = np.zeros(N)
    ref[40:50] = 1.5
    ref += 0.1 * (rng.random(N) - 0.5)
    Y = 0.1 * (rng.random((S, N)) - 0.5)
    for i in range(0, S, 3):
        w = int(rng.integers(3, 20))
        m = int(rng.integers(30, 70))
        Y[i, m:m + w] += rng.uniform(0.5, 40)
    Y[5] = 2.0                                              # constant -> score 0, lag 0
    graphs = [i // 6 for i in range(S)]
    series = [mo.Series(Y[i], mo.Labels({"graph": "g%d" % graphs[i], "host": "h%d" % (i % 6)}))
              for i in range(S)]
    sc_all, lg_all = mo.score_series_batch(ref, Y)
    for group_by, gids in ((None, None), (["graph"], np.array(graphs))):
        for thr, topn, maxlag in ((0.0, 100, 64), (0.3, 5, 10), (0.0, 7, 3)):
            g = mo.Group("g")
            g.Add(*series)
            b = mo.Batch(mo.Series(ref), g, mo.Results(maxlag, topn, thr, 0), 4)
            b.Run(list(group_by) if group_by else None)
            want, _ = b.Results.Fetch()
            sc, lg, idx = mo.batch_run_arrays(ref, Y, gids, maxlag, topn, thr)
            assert len(want) == len(sc)
            for w, s, l, i in zip(want, sc, lg, idx):
                assert abs(w.PercentScore - s) < 1e-12 and w.Lag == l
                assert w.Labels is series[i].labels
                assert abs(sc_all[i] - s) == 0 and lg_all[i] == l


def test_golden_file_is_what_the_generator_reads_out_of_the_reference():
    """tools/gen_kats.py parses every vector, label and expected score out of the reference's *_test.go literals; the
    committed tests/golden/reference_kats.json must be exactly its output (no hand transcription to slip).  Needs a
    checkout of the reference (go-muse), which is not part of this repository: MUSE_REFERENCE names its directory."""
    import os
    import subprocess
    import sys
    if not os.path.isdir(os.environ.get("MUSE_REFERENCE", "")):
        pytest.skip("MUSE_REFERENCE does not name a checkout of the reference (go-muse)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gen_kats.py"), "--check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
