"""The byte / FLOP models behind bench.py's `roofline` objects, pinned to SURVEY.md section 8(d) (no GPU needed)."""
import bench


def test_ar_step_bytes_matches_survey_8d():
    # SURVEY 8d: W = 152,206,336 weight elements; KV = 24,576 elements per cached token (read) + one token written
    w_elems = 152_206_336
    # batch 1, bf16, L = 647: 304.4 MB + 31.8 MB = 336.2 MB
    b1 = bench.ar_step_bytes(1, 647, 2)
    assert abs(b1 - (w_elems * 2 + 24_576 * 2 * 648)) / b1 < 2e-3   # + fp32 biases / LayerNorm affine (0.7 MB)
    assert 335e6 < b1 < 338e6
    # batch 64, bf16, L = 647: 304.4 + 2,036 MB
    b64 = bench.ar_step_bytes(64, 647, 2)
    assert 2.33e9 < b64 < 2.35e9
    # fp32 parity mode doubles the matrices and the cache
    assert abs(bench.ar_step_bytes(1, 647, 4) / b1 - 2.0) < 0.01


def test_nar_pass_flops_matches_survey_8d():
    # SURVEY 8d, config 2: B=32, L=1500 -> 14.50 (projections) + 3.54 (attention) + 0.075 (head) = 18.1 TFLOP / pass
    f = bench.nar_pass_flops(32, 1500, 1125)
    assert abs(f - 18.1e12) / 18.1e12 < 0.01
    # the bench shape (64 x 1025 rows, 753 target frames): projections dominate
    fb = bench.nar_pass_flops(64, 1025, 753)
    proj = 2 * 64 * 1025 * 12 * 12 * 1024 * 1024
    assert 0.80 < proj / fb < 0.90


def test_dump_codes_pads_ragged_utterances(tmp_path):
    import numpy as np
    import torch
    codes = [torch.arange(24).view(3, 8), torch.full((1, 8), 1024)]
    bench.dump_codes(str(tmp_path / "out"), codes)
    got = np.load(tmp_path / "out" / "codes.npy")
    assert got.dtype == np.float32 and got.shape == (2, 3, 8)
    assert (got[0] == np.arange(24).reshape(3, 8)).all()
    assert (got[1, 0] == 1024).all() and (got[1, 1:] == -1).all()


def test_dump_codes_samples_utterances_above_the_size_cap(tmp_path):
    import numpy as np
    import torch
    codes = [torch.full((5, 8), b) for b in range(10)]
    for run in ("a", "b"):
        bench.dump_codes(str(tmp_path / run), codes, max_bytes=3 * 5 * 8 * 4 + 10)
    got = np.load(tmp_path / "a" / "codes.npy")
    assert got.shape == (3, 5, 8) and got.nbytes <= 3 * 5 * 8 * 4
    rows = got[:, 0, 0].tolist()
    assert rows == sorted(rows) and len(set(rows)) == 3                 # distinct utterances, in batch order
    assert all((got[i] == rows[i]).all() for i in range(3))             # whole utterances, not mixed rows
    assert np.array_equal(got, np.load(tmp_path / "b" / "codes.npy"))   # the same sample every time


def test_bench_workload_constants_are_baseline_config1():
    assert (bench.D_MODEL, bench.N_HEAD, bench.N_LAYER, bench.N_Q) == (1024, 16, 12, 8)
    assert (bench.S_TEXT, bench.T_PROMPT) == (47, 225)
    assert bench.FRAMES == 16 * bench.S_TEXT + 1   # valle.py:1047 stop rule with weights that never emit EOS
