"""CPU: bench.py's bookkeeping -- workload shapes of BASELINE.json configs[1], the algorithmic-bytes table covering
the kernel classes the library can time, and the JSON keys the driver contract names."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_workload_is_baseline_config_1():
    w = bench.make_workload(0)
    assert (w["B"], w["S"], w["P"], w["C"], w["n_class"], w["drop_iter"], w["head"], w["layer"] + 1, w["mode"]) == \
        (35, 336, 21, 20, 21, 4, 9, 8, "blur+crf")
    assert tuple(w["imgs"].shape) == (35, 3, 336, 336) and w["guides"].shape == (35, 336, 336, 3) and w["guides"].dtype == np.uint8
    assert w["gts"].shape == (35, 336, 336) and w["gts"].dtype == np.float32
    assert all(len(c) == 20 for c in w["class_lists"]) and w["dataset_ids"][0] == list(range(1, 21))
    w1 = bench.make_workload(1)
    assert not np.array_equal(w["guides"], w1["guides"])          # ranks get different images (weak scaling)


def test_live_class_distribution():
    w = bench.make_workload(0, classes="live")
    counts = [len(c) for c in w["class_lists"]]
    assert min(counts) >= 1 and max(counts) <= 6 and 1.0 <= np.mean(counts) <= 2.2
    assert all(ids == sorted(ids) and all(1 <= i <= 20 for i in ids) for ids in w["dataset_ids"])
    assert w["name"] == "voc_live_classes_b35_336_drop4_head9_blur+crf"


def test_every_baseline_config_has_a_workload():
    """`--config k` names BASELINE.json configs[k]: shapes per SURVEY 8(d)'s table."""
    import json
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(bench.CONFIGS) == len(base["configs"]) and bench.WORKLOAD is bench.CONFIGS[1]
    want = {0: (1, 336, 21, 336, 20, 21, 1, "blur", 21), 1: (35, 336, 21, 336, 20, 21, 4, "blur+crf", 21),
            2: (35, 336, 21, 336, 150, 151, 4, "blur+crf", 150), 3: (35, 336, 21, 512, 171, 183, 4, "blur+crf", 171),
            4: (35, 448, 28, 448, 80, 91, 4, "blur+crf", 81)}
    for k, cfg in enumerate(bench.CONFIGS):
        assert cfg["id"] == k
        assert (cfg["B"], cfg["S"], cfg["P"], cfg["G"], cfg["C"], cfg["n_class"], cfg["drop_iter"], cfg["mode"], bench.channels_of(cfg)) == want[k]
        assert len(bench.class_names(cfg)) == cfg["C"] == len(bench.class_ids(cfg)) and max(bench.class_ids(cfg)) < cfg["n_class"]
    small = dict(bench.CONFIGS[3], B=2)
    w = bench.make_workload(0, small)
    assert w["gts"].shape == (2, 512, 512) and w["guides"].shape == (2, 512, 512, 3) and tuple(w["imgs"].shape) == (2, 3, 336, 336)
    assert w["dataset_ids"][0][:3] == [1, 2, 3] and w["dataset_ids"][0][79:82] == [90, 92, 93] and w["coco"] is True
    assert w["valid_pixels"] == int(((w["gts"] >= 0) & (w["gts"] < 183)).sum())
    T = max(len(w["tok"].encode(c)) for c in w["captions"])
    assert T <= 500                                               # fits the reference's max_length=500 padding (DRV:317-319)
    args = bench.parse_args(["--config", "4", "--scaling", "strong"])
    assert args.config == 4 and args.gemm == "3xfp16" and args.schedule == "serial" and args.scaling == "strong" and bench.STRONG_IMAGES % 35 == 0


def test_algorithmic_bytes_cover_the_timed_kernel_classes():
    from pnp_ovss_b200 import _lib
    lib = _lib.load()
    w = bench.make_workload(0)
    stats = {"M_s": 14755, "M_b": 3245257}
    n_ids = lib.pnp_profile_num_kernels()
    names = [lib.pnp_profile_kernel_name(i).decode() for i in range(1, n_ids)]
    assert len(set(names)) == n_ids - 1 and all(names) and n_ids <= 32          # the mask of pnp_profile_start is 32 bits
    for n in names:
        b = bench.algorithmic_bytes(n, w, stats, 31)
        assert (b is None) == (n in bench.LATENCY_BOUND), n
        assert bench.algorithmic_bytes(n, w, stats, 31, "3xtf32") is None or bench.algorithmic_bytes(n, w, stats, 31, "3xtf32") >= b
        if b is not None:
            assert b > 0
    # the dominant kernels' figures of DESIGN.md section 3
    assert bench.algorithmic_bytes("crf_blur_axis_bilateral", w, stats, 31) == 2 * (8 * 21 + 8) * 3245257
    assert bench.algorithmic_bytes("softmax_fwd", w, stats, 31) == 8 * 35 * 12 * 31 * 442
    assert bench.algorithmic_bytes("lowrank_unary", w, stats, 31) == 4 * 35 * 20 * 441 + 4 * 35 * 21 * 336 * 336   # SURVEY 8(d) row (d)
    assert bench.MODEL_KERNELS <= set(names)


def test_reference_arm_fills_the_host_cores():
    """The CPU arm processes max(8, cores/2) images per step, every (image, pass) job of the step in one pool.map, so its
    post-processing uses the cores it reports (the round-1 arm ran one image on one core)."""
    assert bench.default_ref_images() >= 8 and bench.default_ref_images() >= (os.cpu_count() or 1) // 2
    assert bench.n_reference_passes(bench.CONFIGS[1]) == 2 and bench.n_reference_passes(bench.CONFIGS[0]) == 1
    assert bench.n_reference_passes(bench.CONFIGS[3]) == 1          # COCO driver: only the accumulated map (DRVC:420)
    import inspect
    from oracle import reference_arm as RA
    assert inspect.getsource(RA.reference_batch_confusion).count("pool.map(") == 1


def test_measured_traffic_is_tied_to_the_kernel_sources(tmp_path, monkeypatch):
    """roofline.traffic comes from an ncu capture; a capture made on other kernel sources is reported stale, not copied."""
    import json
    fp = bench.source_fingerprint()
    assert len(fp) == 16 and fp == bench.source_fingerprint()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    os.makedirs(tmp_path / "profiles")
    os.makedirs(tmp_path / "pnp_ovss_b200" / "csrc")
    (tmp_path / "pnp_ovss_b200" / "csrc" / "k.cu").write_text("__global__ void k() {}\n")
    now = bench.source_fingerprint()
    assert bench.measured_traffic("k")[0] is None
    (tmp_path / "profiles" / "dram_traffic.json").write_text(json.dumps({"source_sha16": now, "workload": "w", "kernels": {"k": 123}}))
    assert bench.measured_traffic("k", "w")[0] == 123 and bench.measured_traffic("other", "w")[0] is None
    assert bench.measured_traffic("k", "another workload")[0] is None
    (tmp_path / "pnp_ovss_b200" / "csrc" / "k.cu").write_text("__global__ void k() { }\n")
    v, why = bench.measured_traffic("k", "w")
    assert v is None and "stale" in why


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` end to end on the host CPU (one image, one step): the JSON line the driver parses."""
    import json
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--ref-images", "1", "--no-alt"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"] == bench.WORKLOAD["name"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert cb["post_jobs_per_step"] == 2 and cb["steps_timed"] == 1 and d["steps_requested"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_writes_the_last_step_as_float64(tmp_path):
    """--dump-outputs: one .npy per array batch_confusion returns, batches stacked, values exact; absent arrays are not written."""
    import torch
    assert bench.parse_args([]).dump_outputs is None
    assert bench.parse_args(["--dump-outputs", str(tmp_path)]).dump_outputs == str(tmp_path)
    h = [torch.arange(9, dtype=torch.int64).view(3, 3) * (k + 1) for k in range(2)]
    chosen = [torch.full((4, 40), k - 1, dtype=torch.int32) for k in range(2)]
    batches = [{"hist_round0": None, "hist_all_drop": h[k], "dropout_chosen": chosen[k]} for k in range(2)]
    bench.dump_outputs(str(tmp_path / "out"), batches, h[0] + h[1])
    assert sorted(os.listdir(tmp_path / "out")) == ["dropout_chosen.npy", "hist_all_drop.npy", "hist_timed_total.npy"]
    got = {n: np.load(tmp_path / "out" / (n + ".npy")) for n in ("dropout_chosen", "hist_all_drop", "hist_timed_total")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["hist_all_drop"], torch.stack(h).numpy()) and np.array_equal(got["hist_timed_total"], (h[0] + h[1]).numpy())
    assert np.array_equal(got["dropout_chosen"], torch.stack(chosen).numpy())


@pytest.mark.gpu
def test_our_arm_times_the_requested_steps_and_dumps_the_last_one(tmp_path):
    """configs[0] (one image, drop_iter 1) end to end through bench.py: --steps sets the timed steps, and the dumped matrix of the
    last step times the step count is the matrix accumulated over the timed region."""
    import json
    import subprocess
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "0", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-e2e", "--no-alt", "--no-parity", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["hist_total"] == d["hist_expected"]
    assert sorted(os.listdir(tmp_path)) == ["hist_round0.npy", "hist_timed_total.npy"]   # drop_iter 1: no DropOut outputs
    h0, total = np.load(tmp_path / "hist_round0.npy"), np.load(tmp_path / "hist_timed_total.npy")
    assert h0.shape == (1, 21, 21) and h0.dtype == np.float64
    assert h0.sum() * 2 == d["hist_expected"] and np.array_equal(h0[0] * 2, total)


def test_our_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: on a box without CUDA the product arm of bench.py stops with a clear message (and exit code != 0)."""
    import subprocess
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
