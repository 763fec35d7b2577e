"""Float sums of rtc_render_u8_multi while frames of rtc_frame_begin are in flight (-m gpu).

The 8-bit calls write the float total over the head entry's own accumulation buffer; a frame slot's buffers belong to
its frame alone.  So a sum asked for between rtc_frame_begin and rtc_frame_end leaves the queued frames as they are,
and is itself the sum a render of its own gives."""
import numpy as np
import pytest

from conftest import scene_path

pytestmark = pytest.mark.gpu


def test_sums_while_frames_are_in_flight(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(256, 192, 16)
    frame_seeds, sum_seeds = (60, 61), (70, 71)
    want_frames = [s.Render(seed=seed) for seed in frame_seeds]
    want_imgs = [s.Render(seed=seed) for seed in sum_seeds]
    want_sums = [s.RenderSum(seed=seed, sample_count=16) for seed in sum_seeds]
    got_frames = [np.zeros_like(want_frames[0]) for _ in frame_seeds]
    for slot, seed in enumerate(frame_seeds):
        s.frame_begin(seed=seed, slot=slot)
    got = [s.RenderMulti(devices, seed=seed, want_sum=True) for devices, seed in (([0], sum_seeds[0]), ([0, 0], sum_seeds[1]))]
    for slot in range(2):
        s.frame_end(slot, got_frames[slot])
    s.close()
    for a, b in zip(want_frames, got_frames):
        assert (np.abs(a.astype(int) - b.astype(int)) <= 1).mean() > 0.999
    for (img, total), want_img, want_sum in zip(got, want_imgs, want_sums):
        ok = np.isfinite(want_sum) & np.isfinite(total)
        assert ok.mean() > 0.999
        assert np.allclose(total[ok], want_sum[ok], rtol=1e-4, atol=1e-5), np.abs(total[ok] - want_sum[ok]).max()
        assert (np.abs(img.astype(int) - want_img.astype(int)) <= 1).mean() > 0.999
