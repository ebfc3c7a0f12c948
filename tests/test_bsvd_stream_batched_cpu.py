"""Host-only view of a BSVD stream's layout (ss4k_debug_bsvd_stream_layout): lags and ring lengths for pushes of up to
max_frames frames.  A liveness simulation of the stream's steps checks that no ring slot is overwritten while a later
step still reads it, for every push-size sequence; one-frame streams keep the rings they always had."""
import ctypes
import json
import random

import pytest

from ss4k_b200 import _lib as L


def _layout(max_frames, act_mode=L.ACT_F16, in_fmt=L.FMT_F32_NCHW, h=32, w=136):
    lib = L.load()
    cfg = L.PlanCfg()
    cfg.struct_size = ctypes.sizeof(L.PlanCfg)
    cfg.arch, cfg.n, cfg.h, cfg.w = L.ARCH_BSVD, 1, h, w
    cfg.act_mode, cfg.in_fmt, cfg.out_fmt, cfg.use_graph = act_mode, in_fmt, L.FMT_F32_NCHW, 1
    out = ctypes.c_void_p()
    L.check(lib.ss4k_debug_bsvd_stream_layout(ctypes.byref(cfg), max_frames, ctypes.byref(out)))
    try:
        return json.loads(ctypes.string_at(out).decode())
    finally:
        lib.ss4k_free(out)


def _one_frame_rings(lay):
    """The ring lengths of one-frame streams: producer lag to last reader's lag, + 3, rounded up to a power of two >= 4;
    a low-half twin takes its tensor's length."""
    last = {}
    for st in lay["steps"]:
        for b in st["reads"]:
            last[b] = max(last.get(b, 0), st["lag"])
    rings = []
    for i, b in enumerate(lay["bufs"]):
        need, r = max(0, last.get(i, 0) - b["lag"]) + 3, 4
        while r < need:
            r *= 2
        rings.append(r)
    for st in lay["steps"]:   # [hi, lo] pairs of split precision
        for ids in (st["writes"], st["reads"]):
            for a, b in zip(ids[0::2], ids[1::2]):
                if lay["bufs"][b]["name"] == lay["bufs"][a]["name"] + "_lo":
                    rings[b] = rings[a]
    return rings


def _simulate(lay, pushes, clip_len=None):
    """Run the stream's steps over the push sizes (then the one-frame flush steps when clip_len is given) and record,
    for every ring slot, the frame whose data it holds.  Every read of frame f must find frame f in its slot."""
    rings = [b["ring"] for b in lay["bufs"]]
    holder = [dict() for _ in rings]
    T = clip_len
    t = 0

    def step(n, flush):
        for st in lay["steps"]:
            lo, hi = t - st["lag"], t - st["lag"] + n
            if st["kind"] == 0:
                if flush:
                    continue
                frames = range(lo, hi)
            else:
                frames = range(max(lo, 0), min(hi, T) if T is not None else hi)
            for f in frames:
                for b in st["reads"]:
                    assert holder[b].get(f % rings[b]) == f, (lay["bufs"][b]["name"], f, holder[b].get(f % rings[b]))
            for f in frames:
                for b in st["writes"]:
                    holder[b][f % rings[b]] = f
                    if st["tshift"]:   # channel slices of frame f stored into the slots of frames f-1 and f+1
                        for g in (f - 1, f + 1):
                            if g >= 0 and (T is None or g < T):
                                slot = g % rings[b]
                                assert holder[b].get(slot, g) == g or holder[b][slot] < g - 1, (lay["bufs"][b]["name"], g)
                                holder[b][slot] = g

    for n in pushes:
        step(n, False)
        t += n
    if T is not None:
        while t < T + lay["shift_num"]:
            step(1, True)
            t += 1


@pytest.mark.parametrize("act_mode", [L.ACT_F16, L.ACT_F16_SPLIT])
def test_one_frame_rings_unchanged(act_mode):
    lay = _layout(1, act_mode)
    assert lay["shift_num"] == 16
    assert [b["ring"] for b in lay["bufs"]] == _one_frame_rings(lay)
    assert lay["period"] == max(b["ring"] for b in lay["bufs"])


@pytest.mark.parametrize("act_mode", [L.ACT_F16, L.ACT_F16_SPLIT])
def test_rings_grow_by_max_frames(act_mode):
    base = [b["ring"] for b in _layout(1, act_mode)["bufs"]]
    for m in range(1, 9):
        lay = _layout(m, act_mode)
        for r0, b in zip(base, lay["bufs"]):
            r = b["ring"]
            assert r & (r - 1) == 0 and r >= r0 and r >= m + 2
        assert all(lay["period"] % b["ring"] == 0 for b in lay["bufs"])


@pytest.mark.parametrize("act_mode", [L.ACT_F16, L.ACT_F16_SPLIT])
def test_liveness_random_push_sizes(act_mode):
    rng = random.Random(1234)
    for m in range(1, 9):
        lay = _layout(m, act_mode)
        for trial in range(6):
            pushes = [rng.randint(1, m) for _ in range(rng.randint(1, 40))]
            clip = sum(pushes) if trial % 2 == 0 else None
            _simulate(lay, pushes, clip)


def test_liveness_fails_with_short_rings():
    """The simulation detects rings too short for the pushes: a stream laid out for one frame per push, pushed 8 at a time."""
    lay = _layout(1)
    with pytest.raises(AssertionError):
        _simulate(lay, [8] * 10)


def test_layout_rejects_bad_arguments():
    lib = L.load()
    cfg = L.PlanCfg()
    cfg.struct_size = ctypes.sizeof(L.PlanCfg)
    cfg.arch, cfg.n, cfg.h, cfg.w = L.ARCH_BSVD, 1, 32, 136
    out = ctypes.c_void_p()
    assert lib.ss4k_debug_bsvd_stream_layout(ctypes.byref(cfg), 0, ctypes.byref(out)) != L.OK
    cfg.arch = L.ARCH_SRVGG
    assert lib.ss4k_debug_bsvd_stream_layout(ctypes.byref(cfg), 1, ctypes.byref(out)) != L.OK
