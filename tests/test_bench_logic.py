"""Host logic of bench.py that needs no GPU."""
import argparse

import numpy as np

import bench


def test_metric_names_follow_the_workload():
    assert "8K VarDCT d1.0" in bench.METRIC["synth8k"]
    assert "d2.0" in bench.METRIC["synth8k_d2"] and "Modular" in bench.METRIC["synthmod4k"]


def test_workloads_are_seeded_and_sized():
    desc, frames, (w, h) = bench.load_workload("synth4k", 5)
    assert (w, h) == (3840, 2160) and len(frames) == 5 and frames[0] == frames[4] and frames[0] != frames[1]
    assert "EPF 2" in desc


def test_fixed_hf_schedule_and_roofline_families():
    assert bench.HF_STREAMS_PER_CTA in (8, 16, 32, 64, 128) and bench.HF_LATENCY_SCHEDULE in (8, 16, 32)
    assert set(bench.CHAIN) & set(bench.KERNELS) and set(bench.ENTROPY) <= set(bench.KERNELS)
    assert bench.algorithmic_bytes("filters_fused", 7680, 4320, 0) == 7680 * 4320 * 24


def test_dump_sample_is_seeded_and_within_budget():
    """--dump-outputs: the same pixels in every run (two builds compare file for file), 96 8K frames within budget."""
    npx = 7680 * 4320
    pos = bench.dump_positions(npx, 3, 96)
    assert np.array_equal(pos, bench.dump_positions(npx, 3, 96))
    assert pos.size * 3 * 4 * 96 <= bench.DUMP_BYTES and pos.size > 40000
    assert np.all(np.diff(pos) > 0) and pos[0] >= 0 and pos[-1] < npx
    assert np.array_equal(bench.dump_positions(640 * 480, 4, 2), np.arange(640 * 480))


def test_gpu_local_cpus_without_a_gpu_is_empty(monkeypatch):
    import torch

    def no_device(*_):  # what torch does on a machine without a CUDA device, also where the suite runs on a GPU
        raise RuntimeError("no CUDA device")
    monkeypatch.setattr(torch.cuda, "get_device_properties", no_device)
    assert bench.gpu_local_cpus(0) == []
