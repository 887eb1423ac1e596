"""The display tensors over a clip of consecutive frames: ``silent_display_sequence`` and ``LineEndDisplayer.run_clip`` /
``callback_clip`` against the per-step path they replace (``silent_display_tensors``, ``run_frames_display``,
``callback``), bit for bit, NaN masks included. The host-side checks run without a GPU."""
import ctypes

import numpy as np
import pytest

from conftest import synthetic_frame

torch = pytest.importorskip("torch")

FAKE = ctypes.c_void_p(16)   # never dereferenced: every check below fails before the first CUDA call


def _args(**kw):
    a = dict(gray=FAKE, steps=2, n=3, h=37, w=53, rh=3, rw=3, half_h=22, half_w=32, energy=FAKE, exh=1.0, exc=1.0, mode=1,
             normer=127.5, centerer=127.5, cent=FAKE, cent2=FAKE, fired=FAKE, update=FAKE, scratch=FAKE, nbytes=1 << 30,
             stream=None)
    a.update(kw)
    return list(a.values())


def test_display_sequence_host_checks_without_gpu(built_lib):
    L = built_lib
    for bad in ("gray", "energy", "cent", "cent2", "fired", "update", "scratch"):
        assert L.silent_display_sequence(*_args(**{bad: None})) == -1, bad
        assert b"null argument" in L.silent_last_error()
    for bad in (dict(steps=0), dict(n=0), dict(h=-1), dict(w=0), dict(rh=0), dict(rw=0), dict(half_h=0), dict(half_w=0)):
        assert L.silent_display_sequence(*_args(**bad)) == -1, bad
        assert b"bad shape" in L.silent_last_error()
    need = L.silent_display_sequence_scratch_bytes(2, 3, 37, 53, 3, 3)
    assert L.silent_display_sequence(*_args(nbytes=need - 1)) == -1
    assert b"scratch" in L.silent_last_error()
    for mode in (0, 4):
        assert L.silent_display_sequence(*_args(mode=mode, nbytes=need)) == -1
        assert L.silent_last_error() == b"You must choose a type of recovery"


def test_display_sequence_scratch_bytes(built_lib):
    from pysilent_b200 import _ops
    L = built_lib
    for steps, n, h, w, r in ((1, 1, 192, 288, 3), (7, 18, 100, 149, 3), (2, 5, 37, 53, 4), (64, 6, 192, 288, 3)):
        oh, ow = -(-h // r), -(-w // r)
        want = (steps * n + n) * oh * ow * 4   # importance of every step + the fallback's one-step bias buffer
        assert L.silent_display_sequence_scratch_bytes(steps, n, h, w, r, r) == want
        assert _ops.display_sequence_scratch_bytes(steps, n, h, w, r, r) == want
    assert L.silent_display_sequence_scratch_bytes(0, 1, 4, 4, 3, 3) == 0
    assert L.silent_display_sequence_scratch_bytes(1, 1, 4, 4, 0, 3) == 0


@pytest.mark.parametrize("shape", [(288, 192), (288, 192, 3), (1, 2, 3, 288, 192, 3)])
def test_clip_entry_points_reject_wrong_rank_before_gpu(shape):
    from pysilent_b200 import LineEndDisplayer
    disp = LineEndDisplayer()
    with pytest.raises(ValueError, match="run_clip"):
        disp.run_clip(torch.zeros(shape, dtype=torch.uint8))
    with pytest.raises(ValueError, match="callback_clip"):
        disp.callback_clip(np.zeros(shape, np.uint8))
    with pytest.raises(ValueError):
        disp.run_clip(torch.zeros((0, 48, 64, 3), dtype=torch.uint8))


# ---- on the GPU ----------------------------------------------------------------------------------------------------------

def assert_bits(actual, expected, what):
    a = actual.detach().cpu().numpy() if isinstance(actual, torch.Tensor) else np.asarray(actual)
    e = expected.detach().cpu().numpy() if isinstance(expected, torch.Tensor) else np.asarray(expected)
    assert a.shape == e.shape, (what, a.shape, e.shape)
    nan_a, nan_e = np.isnan(a), np.isnan(e)
    assert np.array_equal(nan_a, nan_e), "%s: NaN masks differ (%d vs %d)" % (what, nan_a.sum(), nan_e.sum())
    same = (a == e) | nan_e
    assert same.all(), "%s: %d of %d values differ" % (what, (~same).sum(), same.size)


@pytest.fixture
def cuda(built_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return built_lib


def _clip_gray(rs, steps, n, h, w, region):
    gray = rs.uniform(0, 255, size=(steps, n, h, w, 1)).astype(np.float32)
    gray[rs.uniform(size=gray.shape) < 0.4] = 0.0
    gray[:, 0, : 3 * region, : 5 * region] = 0.0            # empty blocks: centroid 0 / 0 = NaN, importance 0
    gray[rs.uniform(size=gray.shape) < 0.002] = np.nan       # NaN propagates through importance and the non-max
    if steps > 1:
        gray[1] = 0.0                                        # an all-zero step
    return torch.from_numpy(gray.reshape(steps * n, h, w, 1)).cuda()


def _half(h, w):
    return tuple(int(v) for v in (np.asarray((h, w), np.float32) / np.float32(np.e ** .5)).astype(np.int32))


def _sequence_against_steps(gray, steps, region, energy0, modes):
    """display_sequence of the clip against `steps` display_tensors calls, for every (recovery, exhaustion,
    excitation) in `modes`."""
    from pysilent_b200 import _ops
    total, h, w, _ = gray.shape
    n = total // steps
    hh, hw = _half(h, w)
    for mode, exh, exc in modes:
        e_seq, e_ref = energy0.clone(), energy0.clone()
        got = _ops.display_sequence(gray, e_seq, steps, region, region, hh, hw, exh, exc, mode)
        want = [[] for _ in range(4)]
        for t in range(steps):
            outs = _ops.display_tensors(gray[t * n:(t + 1) * n], e_ref, region, region, hh, hw, exh, exc, mode)
            for i in range(4):
                want[i].append(outs[i])
        what = "T=%d n=%d %dx%d/%d mode %d (%g, %g)" % (steps, n, h, w, region, mode, exh, exc)
        for i in range(4):
            assert_bits(got[i], torch.cat(want[i]), "%s output %d" % (what, i))
        assert_bits(e_seq, e_ref, what + " final energy")
    return got


MODES = [(mode, exh, exc) for mode in (1, 2, 3) for exh, exc in ((1.0, 1.0), (2.0, 8.0))]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5, 18])
@pytest.mark.parametrize("steps", [1, 2, 7])
@pytest.mark.parametrize("h,w,region", [(192, 288, 3), (100, 149, 3), (37, 53, 4), (64, 96, 2)])
def test_display_sequence_matches_display_tensors_loop(cuda, h, w, region, steps, n):
    rs = np.random.RandomState(h * 31 + w * 7 + steps * 3 + n)
    gray = _clip_gray(rs, steps, n, h, w, region)
    oh, ow = -(-h // region), -(-w // region)
    energy0 = torch.from_numpy(rs.uniform(-2, 8, size=(n, oh, ow, 1)).astype(np.float32)).cuda()
    energy0[0] = 8.0
    got = _sequence_against_steps(gray, steps, region, energy0, MODES)
    assert np.isnan(got[0].cpu().numpy()).any()


def _launches(lib, fn):
    torch.cuda.synchronize()
    before = lib.silent_launch_count()
    fn()
    torch.cuda.synchronize()
    return lib.silent_launch_count() - before


@pytest.mark.gpu
def test_display_sequence_fallback_on_a_grid_no_cluster_holds(cuda):
    """A 400 x 400 block grid: a band of 25 rows on 16 CTAs is 10000 cells, beyond what a CTA holds, so the clip goes
    step by step through the two boosting launches of silent_display_tensors."""
    from pysilent_b200 import _ops
    rs = np.random.RandomState(3)
    steps, n, h, w = 3, 2, 400, 400
    gray = _clip_gray(rs, steps, n, h, w, 1)
    energy0 = torch.full((n, h, w, 1), 8.0, device="cuda")
    _sequence_against_steps(gray, steps, 1, energy0, [(1, 1.0, 1.0), (3, 2.0, 8.0)])
    hh, hw = _half(h, w)
    for t in (1, 7):
        g = gray[:n].repeat(t, 1, 1, 1)
        e = energy0.clone()
        assert _launches(cuda, lambda: _ops.display_sequence(g, e, t, 1, 1, hh, hw, 1, 1, 1)) == 1 + 2 * t


@pytest.mark.gpu
def test_display_sequence_cluster_path_is_two_launches(cuda):
    from pysilent_b200 import _ops
    rs = np.random.RandomState(4)
    n, h, w = 6, 192, 288
    for steps in (1, 16):
        gray = _clip_gray(rs, steps, n, h, w, 3)
        e = torch.full((n, 64, 96, 1), 8.0, device="cuda")
        assert _launches(cuda, lambda: _ops.display_sequence(gray, e, steps, 3, 3, 116, 174, 1, 1, 1)) == 2


def _frames(seed, count, h=480, w=640):
    return np.stack([synthetic_frame(seed, i, h, w) for i in range(count)])


def _compare_six(got, want, what):
    assert len(got) == len(want) == 6
    for i in range(6):
        assert_bits(got[i], want[i], "%s tensor %d" % (what, i))


@pytest.mark.gpu
def test_run_clip_matches_successive_run_frames_display(cuda):
    from pysilent_b200 import LineEndDisplayer
    frames = torch.from_numpy(_frames(11, 5)).cuda()
    clip, step = LineEndDisplayer(zoom_ratio=1.3), LineEndDisplayer(zoom_ratio=1.3)
    got = clip.run_clip(frames)
    want = [step.run_frames_display(frames[t]) for t in range(5)]
    _compare_six(got, [torch.cat([w[i] for w in want]) for i in range(6)], "run_clip T=5")
    assert_bits(clip.energy_values, step.energy_values, "run_clip T=5 energy")


@pytest.mark.gpu
def test_run_clip_interleaves_with_callback(cuda):
    """callback x 2, run_clip(T = 3), callback continue one boosting state, like six callbacks."""
    from pysilent_b200 import LineEndDisplayer
    frames = _frames(12, 6)
    a, b = LineEndDisplayer(zoom_ratio=1.3), LineEndDisplayer(zoom_ratio=1.3)
    want = [[np.stack(lv) for lv in b.callback(frames[t])[1:]] for t in range(6)]
    got = [[np.stack(lv) for lv in a.callback(frames[t])[1:]] for t in range(2)]
    clip = [t.cpu().numpy() for t in a.run_clip(torch.from_numpy(frames[2:5]).cuda())]
    L = clip[0].shape[0] // 3
    got += [[clip[i][t * L:(t + 1) * L] for i in range(6)] for t in range(3)]
    got.append([np.stack(lv) for lv in a.callback(frames[5])[1:]])
    for t in range(6):
        _compare_six(got[t], want[t], "interleaved step %d" % t)
    assert_bits(a.energy_values, b.energy_values, "interleaved energy")


@pytest.mark.gpu
def test_run_clip_against_c_oracle(cuda, c_oracle, default_filters):
    from pysilent_b200 import LineEndDisplayer
    frames = _frames(13, 3)
    disp = LineEndDisplayer(zoom_ratio=1.3)
    got = [t.cpu().numpy() for t in disp.run_clip(torch.from_numpy(frames).cuda())]
    energy = None
    for t in range(3):
        pyr = c_oracle.from_image(frames[t:t + 1], 3, (288, 192), 1.3)
        ref = c_oracle.line_end_stack(pyr, default_filters)
        L = pyr.shape[0]
        if energy is None:
            energy = np.full((L, 64, 96, 1), 8, np.float32)
        want, energy = c_oracle.display_tensors(ref["orient"], ref["padded"], ref["gray"], energy)
        for i in range(6):
            assert_bits(got[i][t * L:(t + 1) * L], want[i], "oracle step %d tensor %d" % (t, i))
    assert_bits(disp.energy_values, energy, "oracle energy")


@pytest.mark.gpu
def test_run_clip_time_major_cameras(cuda):
    from pysilent_b200 import LineEndDisplayer
    frames = torch.from_numpy(_frames(14, 6).reshape(3, 2, 480, 640, 3)).cuda()
    clip, step = LineEndDisplayer(zoom_ratio=1.3), LineEndDisplayer(zoom_ratio=1.3)
    got = clip.run_clip(frames)
    want = [step.run_frames_display(frames[t]) for t in range(3)]
    _compare_six(got, [torch.cat([w[i] for w in want]) for i in range(6)], "run_clip T=3 S=2")
    assert_bits(clip.energy_values, step.energy_values, "run_clip T=3 S=2 energy")


@pytest.mark.gpu
def test_run_clip_orientation_bank(cuda):
    from pysilent_b200 import LineEndDisplayer
    frames = torch.from_numpy(_frames(15, 3)).cuda()
    clip, step = LineEndDisplayer(zoom_ratio=1.3, orientations=16), LineEndDisplayer(zoom_ratio=1.3, orientations=16)
    got = clip.run_clip(frames)
    assert got[0].shape[-1] == 16
    want = [step.run_frames_display(frames[t]) for t in range(3)]
    _compare_six(got, [torch.cat([w[i] for w in want]) for i in range(6)], "run_clip orientations=16")
    assert_bits(clip.energy_values, step.energy_values, "run_clip orientations=16 energy")


@pytest.mark.gpu
def test_callback_clip_matches_callbacks(cuda):
    from pysilent_b200 import LineEndDisplayer
    frames = _frames(16, 4)
    a, b = LineEndDisplayer(zoom_ratio=1.3), LineEndDisplayer(zoom_ratio=1.3)
    got = a.callback_clip(frames)
    assert len(got) == 4
    for t in range(4):
        want = b.callback(frames[t])
        assert len(got[t]) == 7 and np.array_equal(got[t][0], frames[t])
        for x in range(6):
            assert len(got[t][1 + x]) == len(want[1 + x])
            for y in range(len(want[1 + x])):
                assert_bits(got[t][1 + x][y], want[1 + x][y], "callback_clip step %d tensor %d level %d" % (t, x, y))
    assert_bits(a.energy_values, b.energy_values, "callback_clip energy")


@pytest.mark.gpu
def test_run_clip_is_deterministic(cuda):
    from pysilent_b200 import LineEndDisplayer
    frames = torch.from_numpy(_frames(17, 4)).cuda()
    a, b = LineEndDisplayer(zoom_ratio=1.3), LineEndDisplayer(zoom_ratio=1.3)
    _compare_six(a.run_clip(frames), b.run_clip(frames), "two identical clips")
    assert_bits(a.energy_values, b.energy_values, "two identical clips energy")
