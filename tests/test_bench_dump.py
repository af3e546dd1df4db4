"""bench.py --dump-outputs: the stored sample of the headline output is fixed from run to run, float32 / float64 only, and
small enough to keep next to a benchmark result at every rank count the benchmark runs at.  CPU only."""
import numpy as np
import torch


def test_headline_outputs_are_a_fixed_sample_in_budget():
    import bench
    out = torch.rand(3, 300, 280, 3)
    ref_sums = torch.rand(1, 7, dtype=torch.float64)
    a = bench.headline_outputs(out, ref_sums, 0, 1)
    b = bench.headline_outputs(out.clone(), ref_sums, 0, 1)
    assert set(a) == {"rank0_pixels", "rank0_first_frame_top_left", "rank0_last_frame_bottom_right", "rank0_ref_sums"}
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert a["rank0_pixels"].shape == (bench.DUMP_PIXELS, 3)
    assert np.isin(a["rank0_pixels"][:, 0], out[..., 0].numpy()).all()                 # sampled from the output, not made up
    assert np.array_equal(a["rank0_first_frame_top_left"], out[0, :256, :256].numpy())
    assert np.array_equal(a["rank0_last_frame_bottom_right"], out[2, -256:, -256:].numpy())
    assert np.array_equal(a["rank0_ref_sums"], ref_sums.numpy())
    assert not np.array_equal(bench.headline_outputs(out, ref_sums, 1, 2)["rank1_pixels"], a["rank0_pixels"][: bench.DUMP_PIXELS // 2])
    for world in (1, 2, 4, 8):                                                           # every rank's files together
        per_rank = sum(v.nbytes for v in bench.headline_outputs(out, ref_sums, world - 1, world).values())
        assert world * per_rank <= 64 << 20, world
