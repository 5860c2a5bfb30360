"""bench.py prints ONE JSON line with the keys the driver reads; checked here on the reference arm with the small
CPU-runnable workload (config A), no GPU needed."""
import importlib.util
import json
import os
import subprocess
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "A",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "kmeans_iters_per_s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "A",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _bench_module():
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_helpers_sample_rows_and_write_float_arrays(tmp_path):
    import numpy as np
    import scipy.sparse as sp
    import torch
    bench = _bench_module()
    assert np.array_equal(bench.dump_rows(10, 20), np.arange(10))
    r = bench.dump_rows(1000, 37)
    assert np.array_equal(r, bench.dump_rows(1000, 37)) and np.array_equal(r, np.unique(r)) and r.size == 37 and r.max() < 1000
    S = sp.random(300, 50, density=0.05, format="csr", dtype=np.float32, random_state=3)
    S.data[:] = np.arange(1, S.nnz + 1, dtype=np.float32)
    A = types.SimpleNamespace(rowptr=torch.from_numpy(S.indptr.astype(np.int32)), colidx=torch.from_numpy(S.indices.astype(np.int32)),
                              vals=torch.from_numpy(S.data), shape=S.shape, device=torch.device("cpu"))
    g = bench.graph_outputs("g", A)
    assert np.array_equal(g["g"], S[g["g_rows"]].toarray()) and np.array_equal(g["g_row_nnz"], np.diff(S.indptr))
    bench.write_outputs(str(tmp_path / "out"), {**g, "labels": torch.arange(5, dtype=torch.int32), "inertia": 2.5})
    files = {f: np.load(str(tmp_path / "out" / f)) for f in os.listdir(str(tmp_path / "out"))}
    assert sorted(files) == ["g.npy", "g_row_nnz.npy", "g_rows.npy", "inertia.npy", "labels.npy"]
    assert files["g.npy"].dtype == np.float32 and all(a.dtype == np.float64 for f, a in files.items() if f != "g.npy")
    assert np.array_equal(files["labels.npy"], np.arange(5)) and files["inertia.npy"] == 2.5
    with pytest.raises(RuntimeError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_MAX_BYTES // 4 + 1, np.float32)})
    assert not os.path.exists(str(tmp_path / "big"))


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["B", "C"])
def test_dump_outputs_of_the_last_timed_step(tmp_path, workload):
    import numpy as np
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2", "--warmup", "0",
                          "--no-cpu-baseline", "--no-extra-legs", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.strip().splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2
    files = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(a.nbytes for a in files.values()) <= 64 << 20
    if workload == "B":
        assert {"prop", "target", "feature_rows", "labels", "centers", "inertia", "n_iter", "adj_syn", "adj_syn_rows",
                "adj_syn_row_nnz"} == set(files)
        assert float(files["inertia"]) == d["result"]["inertia"] and int(files["n_iter"]) == d["result"]["n_iter"]
        assert files["adj_syn_row_nnz"].sum() == d["result"]["syn_nnz"] and files["labels"].shape == (169343,)
        assert files["target"].shape == (16384, 128) and np.array_equal(files["feature_rows"], np.unique(files["feature_rows"]))
    else:
        assert {"u_emb", "u_emb_rows", "i_emb", "i_emb_rows", "labels_u", "labels_i", "centers_u", "centers_i", "inertia_u",
                "inertia_i", "n_iter_u", "n_iter_i", "condensed", "condensed_rows", "condensed_row_nnz"} == set(files)
        assert float(files["inertia_u"]) + float(files["inertia_i"]) == d["result"]["inertia"]
        assert files["condensed_row_nnz"].sum() == d["result"]["condensed_nnz"]
