"""CPU-side checks of the boundary: the C-ABI library builds, loads and exports every
symbol include/muse_b200.h declares; host-side facade logic (labels, group, results)
mirrors the reference's tests.  No compute calls (no GPU here)."""
import json
import os
import re

import pytest

import muse_b200 as mb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "muse_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(muse_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    mb.build()
    L = mb.lib()
    decl = _declared_symbols()
    assert len(decl) >= 25
    for name in decl:
        assert hasattr(L, name), name
    assert sorted(mb.ABI.keys()) == decl       # the ctypes table covers the whole header
    assert b"sm_100a" in L.muse_version()


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(mb.MuseError) as e:
        mb.Context(0)
    assert e.value.code == mb.MUSE_ERR_NO_DEVICE


def test_merge_partials_host_logic():
    import numpy as np
    parts = np.zeros(7, dtype=mb.PARTIAL_DTYPE)
    # two shards report group 5; the higher score wins BEFORE the lag filter (SURVEY F2)
    parts[0] = (5, 0.70, 10, 0, 0)
    parts[1] = (5, 0.90, 2000, 99, 0)      # best of group 5 but lag 99 -> group 5 rejected
    parts[2] = (6, 0.60, 11, -3, 0)
    parts[3] = (7, 0.60, 7, 2, 0)          # ties with group 6 -> lower series index first
    parts[4] = (8, 0.10, 12, 0, 0)         # below threshold
    parts[5] = (9, float("nan"), 13, 0, 0)
    parts[6] = (6, 0.60, 3000, 1, 0)       # same score as idx 11 -> lowest index keeps
    sc, lg, ix = mb.merge_partials(parts, 10, 5, 0.5)
    assert ix.tolist() == [7, 11] and lg.tolist() == [2, -3] and sc.tolist() == [0.6, 0.6]
    sc, lg, ix = mb.merge_partials(parts, 100, 1, 0.0)
    assert ix.tolist() == [2000]


def test_facade_labels_group_results(kats):
    for c in kats["labels_id"]["cases"]:
        gb = list(c["group_by"]) if c["group_by"] else None
        assert mb.NewLabels(c["labels"]).ID(gb) == c["expected"]
    k = kats["series"]
    assert mb.NewSeries([0.1, 0.2, 0.3], None).Labels().Keys() == [k["default_label"]]
    for c in k["uid_cases"]:
        assert mb.NewSeries([0.1], mb.NewLabels(c["labels"])).UID() == c["expected"]
    k = kats["group_add"]
    g = mb.NewGroup("test")
    for c in k["cases"]:
        s = mb.NewSeries(k["y"], mb.NewLabels(c["labels"]))
        if c["expect_error"]:
            with pytest.raises(mb.MuseError):
                g.Add(s)
        else:
            g.Add(s)
    with pytest.raises(mb.MuseError) as e:
        g.Add(mb.NewSeries([1.0, 2.0], mb.NewLabels({"zz": "1"})))
    assert e.value.code == mb.MUSE_ERR_LENGTH_MISMATCH
    k = kats["index_label_values"]
    g = mb.NewGroup("test")
    for l in k["labels"]:
        g.Add(mb.NewSeries(k["y"], mb.NewLabels(l)))
    for labels, want in k["filter_cases"]:
        assert len(g.FilterByLabelValues(mb.NewLabels(labels))) == want
    # results.go:55-87
    r = mb.NewResults(5, 3, 0.2, mb.SignFilter_ANY)
    lab = mb.NewLabels({"a": "b"})
    for sc, lag in [(0.5, 0), (0.9, 1), (0.1, 0), (0.7, 6), (0.3, -5), (0.6, 2), (0.5, 3)]:
        r.Update(mb.Score(lab, lag, sc))
    r.Update(mb.Score(None, 0, 1.0))
    out, mean = r.Fetch()
    assert [s.PercentScore for s in out] == [0.9, 0.6, 0.5] and out[2].Lag == 0
    import math
    out, mean = r.Fetch()
    assert out == [] and math.isnan(mean)


def test_kernel_phases_on_cpu(tmp_path):
    """The per-thread phases of the CUDA kernels, compiled as host code and run for all
    'threads' of a series, against a direct O(n^2) long-double cross correlation."""
    import subprocess
    exe = str(tmp_path / "muse_emulate_kernel")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "go-muse_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "emulate_kernel.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "ALL OK" in out.stdout


def test_big_kernel_phases_on_cpu(tmp_path):
    """score_screen_big_kernel's phases (n = 4096 .. 16384: mirror-paired last pass, split and conj(Y)*X in
    registers, transposed inverse) run thread by thread on the CPU against a double-precision FFT: the bound
    sum |Y||X| / n and the maxima of |cc| inside and outside the lag window."""
    import subprocess
    exe = str(tmp_path / "muse_emulate_big")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "go-muse_b200", "csrc"),
                           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "cpp", "emulate_big.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert out.stdout.count(" ok") == 10 and "FAIL" not in out.stdout


def test_merge_partials_against_a_model():
    """muse_merge_partials against a direct Python model on random shard outputs: group max across shards
    BEFORE the filter (muse_batch.go:87-89, SURVEY F2), ties by lowest global series index, filter
    (results.go:46-52), top-N in descending |score| (results.go:81-85); padding and NaN records ignored."""
    import numpy as np
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 2**32 - 1), st.integers(0, 60), st.integers(1, 12), st.integers(0, 12),
           st.sampled_from([0.0, 0.25, 0.5, 0.75]), st.sampled_from([0, 1, -1]), st.integers(0, 30))
    def check(seed, n, n_groups, max_lag, thr, sign, top_n):
        rng = np.random.default_rng(seed)
        parts = np.zeros(n, dtype=mb.PARTIAL_DTYPE)
        parts["group_key"] = rng.integers(0, n_groups, n)
        parts["score"] = rng.choice([0.0, 0.25, 0.5, 0.75, 1.0, -0.5, -0.75, np.nan], n)
        parts["series_idx"] = rng.permutation(10 * n + 10)[:n]
        parts["lag"] = rng.integers(-15, 16, n)
        parts["flags"] = rng.choice([0, 0, 0, 1], n)
        best = {}
        for p in parts:
            if (p["flags"] & 1) or p["score"] != p["score"]:
                continue
            q = best.get(int(p["group_key"]))
            if q is None or abs(p["score"]) > abs(q["score"]) or \
                    (abs(p["score"]) == abs(q["score"]) and p["series_idx"] < q["series_idx"]):
                best[int(p["group_key"])] = p
        keep = [p for p in best.values()
                if abs(int(p["lag"])) <= max_lag and abs(p["score"]) >= thr and
                (sign == 0 or (p["score"] > 0 and sign == 1) or (p["score"] < 0 and sign == -1))]
        keep.sort(key=lambda p: (-abs(p["score"]), int(p["series_idx"])))
        keep = keep[:top_n]
        sc, lg, ix = mb.merge_partials(parts, max_lag, top_n, thr, sign)
        assert ix.tolist() == [int(p["series_idx"]) for p in keep]
        assert lg.tolist() == [int(p["lag"]) for p in keep]
        assert sc.tolist() == [float(p["score"]) for p in keep]

    check()


def test_score_json_is_what_encoding_json_writes():
    # scores.go:11-15: field order labels / lag / percentScore; *Labels has only unexported fields (labels.go:14-17),
    # so encoding/json writes {} for a non-nil pointer and null for nil
    import json
    import muse_b200 as mb
    s = mb.Score(mb.NewLabels({"graph": "g1", "host": "h1"}), -3, 0.75)
    assert s.MarshalJSON() == '{"labels":{},"lag":-3,"percentScore":0.75}'
    assert mb.Score(None, 0, 1.0).MarshalJSON() == '{"labels":null,"lag":0,"percentScore":1}'      # Go writes 1, not 1.0
    assert mb.Score(None, 2, 2.5e-7).MarshalJSON() == '{"labels":null,"lag":2,"percentScore":2.5e-7}'  # and e-7, not e-07
    assert json.loads(s.MarshalJSON())["percentScore"] == 0.75
    assert s.to_json()["labels"] == {"graph": "g1", "host": "h1"}
    import pytest
    with pytest.raises(ValueError):
        mb.Score(None, 0, float("nan")).MarshalJSON()      # json: unsupported value: NaN


def test_bench_reference_arm_prints_the_contract_line():
    # bench.py --impl reference needs no GPU (the C oracle on the host cores): the JSON line the driver parses
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--series", "3000",
                        "--cpu-sample", "3000", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "series-samples/s" and line["value"] > 0
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_screen_error_survey_keeps_its_margins():
    """profiles/screen_error_survey.json (tools/screen_error_survey.py, measured on a B200): for every FFT length the
    screening kernels serve, the fp32 second stage stays within a quarter of the slack of the fp64 score and no bound
    comes closer than a quarter of the slack to the score it brackets."""
    path = os.path.join(ROOT, "profiles", "screen_error_survey.json")
    d = json.load(open(path))
    slack = d["slack"]
    assert slack == 1e-4
    lens = {r["fft_len"] for r in d["rows"]}
    assert {512, 1024, 2048, 4096, 8192, 16384} <= lens
    assert any(r["N"] & 1 for r in d["rows"])                  # odd lengths are part of the survey
    for r in d["rows"]:
        assert r["fp32_vs_fp64_worst_abs_error"] <= slack / 4, r
        for k in ("spectral_bound_min_margin", "refined_upper_min_margin", "refined_lower_min_margin"):
            assert r[k] >= slack / 4, (k, r)


def test_go_facade_binds_only_declared_symbols():
    """The cgo facade cannot be compiled here (no Go toolchain): at least every C.muse_* function and C.MUSE_* constant it
    names must be one include/muse_b200.h declares, and braces / parentheses must balance in every file."""
    hdr = open(os.path.join(ROOT, "include", "muse_b200.h")).read()
    declared = set(_declared_symbols())
    consts = set(re.findall(r"#define\s+(MUSE_[A-Z0-9_]+)", hdr))
    types = set(re.findall(r"typedef struct (muse_[a-z_]+)", hdr)) | {"muse_partial", "muse_timing"}
    godir = os.path.join(ROOT, "go-muse_b200", "go", "muse")
    used = set()
    for name in sorted(os.listdir(godir)):
        if not name.endswith(".go"):
            continue
        src = open(os.path.join(godir, name)).read()
        code = re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", src, flags=re.S))
        code = re.sub(r'"(\\.|[^"\\])*"', '""', code)
        for a, b in ("{}", "()", "[]"):
            assert code.count(a) == code.count(b), (name, a, code.count(a), code.count(b))
        for sym in re.findall(r"\bC\.(muse_[a-z0-9_]+|MUSE_[A-Z0-9_]+)", code):
            used.add(sym)
            assert sym in declared or sym in consts or sym in types, (name, sym)
    assert {"muse_batch_run", "muse_group_append", "muse_batch_run_exchange_ex", "muse_exchange_open_peers"} <= used
