"""bench.py's reference arm runs on the host cores only: its JSON line can be checked without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    return json.loads(lines[0])


def test_reference_arm_line_contract():
    d = _run()
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and base["metric"].startswith(d["metric"]) and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("cfg2") and d["config"]["mics_per_node"] == 4 and d["config"]["n_fft"] == 512
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    # the step time multiplies back to the frames the sample really processed
    frames = cb["value"] * d["ms_per_step"] / 1e3 * d["steps"]
    assert frames > 0 and abs(frames - round(frames / 626) * 626) < 1.0          # whole utterances of 626 frames


def test_reference_arm_other_workload():
    d = _run("--workload", "cfg3")
    assert d["config"]["workload"].startswith("cfg3") and d["config"]["nodes"] == 4


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_dump_outputs_writes_float32_within_budget(tmp_path):
    import numpy as np
    import torch
    b = _bench_module()
    g = torch.Generator().manual_seed(3)
    yf = torch.randn((4, 1, 30, 17), dtype=torch.complex64, generator=g)
    mask = torch.rand((4, 1, 30, 17), generator=g)
    b.dump_outputs(str(tmp_path / "full"), {"yf": yf, "mask": mask})
    assert np.array_equal(np.load(tmp_path / "full" / "yf.npy"), torch.view_as_real(yf).numpy())
    assert np.array_equal(np.load(tmp_path / "full" / "mask.npy"), mask.numpy())
    budget = 6000                                   # bytes; the two arrays hold 2040 * (8 + 4) = 24480
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), {"yf": yf, "mask": mask}, budget=budget)
    a_yf, a_m = np.load(tmp_path / "a" / "yf.npy"), np.load(tmp_path / "a" / "mask.npy")
    assert a_yf.dtype == np.float32 and a_m.dtype == np.float32 and a_yf.shape[-1] == 2
    assert a_yf.nbytes + a_m.nbytes <= budget and a_m.size == a_yf.shape[0] > 0
    assert np.array_equal(a_yf, np.load(tmp_path / "b" / "yf.npy")) and np.array_equal(a_m, np.load(tmp_path / "b" / "mask.npy"))
    # the same positions in every array of the same size: each sampled (re, im) pair sits next to its own mask value
    ref = torch.view_as_real(yf).reshape(-1, 2).numpy()
    pos = [int(np.flatnonzero((ref == row).all(axis=1))[0]) for row in a_yf]
    assert np.array_equal(a_m, mask.reshape(-1).numpy()[pos]) and pos == sorted(pos)


def test_bench_rejects_zero_steps_and_unsupported_dumps(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                  ["--shard", "nodes", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "usage" in r.stderr and not r.stdout, extra


def test_numa_binding_helper_decodes_nvml_mask_and_survives_its_absence():
    b = _bench_module()
    before = os.sched_getaffinity(0)

    def broken(_):
        raise RuntimeError("no NVML")
    b._nvml_handle = broken
    assert b.bind_host_to_gpu(0) is None and os.sched_getaffinity(0) == before
    first = min(before)

    class FakeNvml:
        @staticmethod
        def nvmlDeviceGetCpuAffinity(handle, n_words):
            words = [0] * n_words
            words[first // 64] = 1 << (first % 64)
            return words
    b._nvml_handle = lambda i: (FakeNvml, None)
    try:
        if len(before) > 1:
            assert b.bind_host_to_gpu(0) == 1 and os.sched_getaffinity(0) == {first}
        else:
            assert b.bind_host_to_gpu(0) is None          # mask == allowed set: nothing to do
    finally:
        os.sched_setaffinity(0, before)
