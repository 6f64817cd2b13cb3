"""Host-side tooling behind the measurement contract (no GPU): the per-step ncu summary that bench.py reads, its staleness
flag, and the flop / launch bookkeeping the roofline uses."""
import json
import os
import sys

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))


def _row(i, name, metric, unit, value):
    return f'"{i}","1","python","127.0.0.1","{name}","ctx","7","1","1","sec","{metric}","{unit}","{value}"\n'


def test_step_summary_groups_launches_and_records_the_source_hash(tmp_path):
    import summarize_ncu
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Section Name","Metric Name","Metric Unit","Metric Value"\n'
    names = ["void fd::embed_kernel<12>(x)"]
    for _ in range(12):
        names += ["void fd::tc_gemm_kernel<192,3,3,2,1>(a)", "void fd::attention_tc_kernel<0>(a)", "void fd::tc_gemm_kernel<192,3,5,2,1>(a)",
                  "void fd::tc_gemm_kernel<192,3,4,2,1>(a)", "void fd::tc_gemm_kernel<192,3,5,2,1>(a)"]
    names += ["void fd::tc_gemm_kernel<192,3,4,2,1>(a)", "void fd::tail_kernel<12,1>(x)"]
    assert len(names) == 63
    src = tmp_path / "step_metrics.csv"
    with open(src, "w") as f:
        f.write("==PROF== banner line\n" + hdr)
        for i, n in enumerate(names):
            f.write(_row(i, n, "gpu__time_duration.sum", "us", "10.0"))
            f.write(_row(i, n, "dram__bytes_read.sum", "Mbyte", "100"))
            f.write(_row(i, n, "dram__bytes_write.sum", "Mbyte", "50"))
            f.write(_row(i, n, "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "%", "40" if "gemm" in n else "0"))
    (tmp_path / "step_source_sha.txt").write_text("abcdef0123456789\n")
    dst = tmp_path / "out.json"
    summarize_ncu.step(str(src), str(dst))
    d = json.load(open(dst))
    assert d["source_sha"] == "abcdef0123456789" and d["launches"] == 63
    k = d["kernels"]
    assert {c: k[c]["launches"] for c in k} == {"embed": 1, "gemm_qkv": 12, "attention": 12, "gemm_attn_out": 12, "gemm_ffn1": 12,
                                                "gemm_ffn2": 12, "gemm_head": 1, "tail_posterior": 1}
    assert k["gemm_qkv"]["dram_bytes_per_launch"] == 150_000_000 and k["gemm_qkv"]["tensor_pipe_active_pct"] == 40.0
    assert d["dram_bytes_per_reverse_step"] == 63 * 150_000_000


def test_bench_flags_a_stale_ncu_profile(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    import summarize_ncu
    assert bench.source_sha() == summarize_ncu.source_sha()  # one definition of "the CUDA sources", two readers
    prof = bench.load_ncu_profile()
    assert prof is not None and prof["file"].startswith("profiles/") and isinstance(prof["stale"], bool)
    monkeypatch.setattr(bench, "source_sha", lambda: "0" * 16)
    assert bench.load_ncu_profile()["stale"] is True


def test_bench_dump_outputs_writes_float32_and_a_fixed_sample_over_the_limit(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    a = np.arange(40 * 3, dtype=np.float64).reshape(40, 3)
    bench.dump_outputs(str(tmp_path / "all"), {"angles": a})
    got = np.load(tmp_path / "all" / "angles.npy")
    assert got.dtype == np.float32 and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * 3 * 4)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"angles": a})
    s1, s2 = (np.load(tmp_path / d / "angles.npy") for d in ("s1", "s2"))
    assert s1.shape == (10, 3) and np.array_equal(s1, s2)  # within the limit, and the same rows every time
    assert all(row in a.tolist() for row in s1.tolist())


def test_bench_rejects_a_step_count_below_one(monkeypatch):
    import pytest
    sys.path.insert(0, ROOT)
    import bench
    for argv in (["--steps", "0"], ["--warmup", "-1"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse_args()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3", "--dump-outputs", "out"])
    args = bench.parse_args()
    assert args.steps == 3 and args.dump_outputs == "out"


def test_algorithmic_flops_match_survey_table():
    from foldingdiff_b200 import synthetic
    lengths = synthetic.sweep_lengths(512)
    assert sum(lengths) == 44564 and sum(l * l for l in lengths) == 4134764          # SURVEY 8d, config 2
    f = synthetic.algorithmic_flops(synthetic.PRODUCTION, lengths)
    assert abs(f - 1.3895e12) / 1.3895e12 < 1e-3
    assert abs(synthetic.algorithmic_flops(synthetic.PRODUCTION, [128]) - 4.1158e9) / 4.1158e9 < 1e-4


def test_every_tool_script_parses():
    """tools/*.py compile and tools/*.sh pass `bash -n` (they only ever run on the GPU box, where a typo costs a call)."""
    import glob
    import py_compile
    import subprocess
    tools = os.path.join(ROOT, "tools")
    for f in sorted(glob.glob(os.path.join(tools, "*.py"))):
        py_compile.compile(f, doraise=True)
    for f in sorted(glob.glob(os.path.join(tools, "*.sh"))):
        r = subprocess.run(["bash", "-n", f], capture_output=True, text=True)
        assert r.returncode == 0, (f, r.stderr)
