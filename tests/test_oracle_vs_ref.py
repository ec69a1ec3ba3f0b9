"""The oracle against the reference itself (the unmodified fsphil/hacktv sources, run through
oracle/ref_harness.c): bit-exact, incl. inputs and options the golden fixtures of
test_oracle_golden.py do not cover. What the reference emitted is stored in tests/golden/vs_ref.json
(sha256 and size of every stream) and tests/golden/vs_ref.npz (an evenly spaced sample of each;
short streams, such as the WSS lines taken apart below, whole). tests/golden/make_golden_vs_ref.py
makes both by running these tests against the reference binaries built by `make -C oracle ref`."""
import hashlib
import json
import os

import numpy as np
import pytest

import orc

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD_JSON = os.path.join(HERE, "golden", "vs_ref.json")
GOLD_NPZ = os.path.join(HERE, "golden", "vs_ref.npz")
SAMPLE = 2048           # values of each stream kept: they say which values differ when the digest does

# tests/golden/make_golden_vs_ref.py sets this to a dict: the comparisons below then run the reference
# binaries, check against their output and record it under each key
RECORD = None
_gold = None


def _key(*parts):
    return " ".join(str(p) for p in parts)


def _digest(a):
    a = np.ascontiguousarray(a)
    stride = -(-a.size // SAMPLE)
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(), "size": int(a.size), "sample": a.ravel()[::stride].copy()}


def _stored(key):
    global _gold
    if _gold is None:
        with open(GOLD_JSON) as f:
            meta = json.load(f)
        z = np.load(GOLD_NPZ)
        _gold = {k: dict(v, sample=z[k]) for k, v in meta.items()}
    return _gold[key]


def _reference(key, args, kw, view):
    want = orc.run_ref(*args, **kw)
    if view is not None:
        want = view(want)
    RECORD[key] = _digest(want)
    return want


def assert_reference(got, key, *args, view=None, **kw):
    """got equals what orc.run_ref(*args, **kw) emits (through `view`), stored under `key`."""
    if RECORD is not None:
        want = _reference(key, args, kw, view)
        assert np.array_equal(got, want), f"{key}: {np.count_nonzero(got != want)} values differ"
        return
    g, d = _stored(key), _digest(got)
    assert d["size"] == g["size"], f"{key}: {d['size']} values, the reference emitted {g['size']}"
    bad = np.count_nonzero(d["sample"] != g["sample"])
    assert bad == 0, f"{key}: {bad} of {g['sample'].size} sampled values differ"
    assert d["sha256"] == g["sha256"], f"{key}: the sampled values agree, others differ"


def reference_values(key, *args, view=None, **kw):
    """What orc.run_ref(*args, **kw) emits (through `view`): short streams, stored whole under `key`."""
    if RECORD is not None:
        return _reference(key, args, kw, view)
    g = _stored(key)
    assert g["sample"].size == g["size"], f"{key} is not stored whole"
    return g["sample"]


CASES = [
    ("pal", 16000000, 700, False, ()),
    ("i", 16000000, 700, True, ()),
    ("i", 16000000, 700, True, ("--nonicam",)),
    ("i", 16000000, 700, True, ("--noaudio", "--nocolour")),
    ("m", 13500000, 600, True, ()),
    ("l", 16000000, 700, True, ()),
    ("l", 16000000, 700, False, ()),
    ("i", 20000000, 400, True, ()),
    ("secam", 16000000, 700, False, ()),
    ("ntsc", 13500000, 600, False, ()),
    ("b", 16000000, 400, True, ()),
    ("pal-m", 13500000, 400, True, ()),
    ("d", 16000000, 400, True, ()),
    ("i", 16000000, 700, True, ("--offset", "2000000")),
    ("i", 16000000, 400, True, ("--swap-iq",)),
    ("pal", 16000000, 400, True, ()),
    # FM video (SURVEY.md section 8f rank 2): the pre-emphasis table differs per sample rate
    ("pal-fm", 20000000, 700, True, ()),
    ("pal-fm", 20250000, 400, True, ()),
    ("pal-fm", 14000000, 400, True, ("--noaudio",)),
    ("pal-fm", 28000000, 300, True, ()),
    ("pal-fm", 20000000, 700, False, ()),
    ("ntsc-fm", 18000000, 600, True, ()),
    ("ntsc-fm", 20250000, 400, True, ()),
    ("secam-fm", 20250000, 400, True, ()),
    ("pal-fm", 20000000, 400, True, ("--offset", "-3000000", "--swap-iq")),
]


def _conf(H, mode, filt, extra):
    kw = dict(vfilter=filt)
    it = iter(extra)
    for e in it:
        if e == "--nonicam": kw["nonicam"] = True
        elif e == "--noaudio": kw["noaudio"] = True
        elif e == "--nocolour": kw["nocolour"] = True
        elif e == "--swap-iq": kw["swap_iq"] = True
        elif e == "--offset": kw["offset"] = int(next(it))
    return H.mode_config(mode, **kw)


@pytest.mark.parametrize("mode,rate,nlines,filt,extra", CASES)
def test_oracle_equals_reference(built, mode, rate, nlines, filt, extra):
    o = orc.Oracle(_conf(built, mode, filt, extra), rate)
    o.open_test_source()
    got = o.render(nlines)
    o.close()
    assert_reference(got, _key("test", mode, rate, nlines, filt, *extra), mode, rate, nlines, vfilter=filt, extra=extra)


PASSTHRU_CASES = [
    ("pal", 16000000, False, (), 40),                    # real output: I only reaches the sink
    ("i", 16000000, True, ("--offset", "1250000"), 40),  # the README's two-channel recipe (second stage)
    ("l", 16000000, True, (), 40),
    ("i", 16000000, False, ("--noaudio",), 40),
    ("m", 13500000, True, (), 12),                       # external stream ends early, mid-line
]


@pytest.mark.parametrize("mode,rate,filt,extra,ext_lines", PASSTHRU_CASES)
def test_passthru_alignment(built, tmp_path, mode, rate, filt, extra, ext_lines):
    """ref _vid_passthru_process video.c:3517-3541: line alignment (the external stream's first
    line is spent on the filter's fill line), int16 wrap, whole lines only at its end."""
    rng = np.random.default_rng(11)
    o = orc.Oracle(_conf(built, mode, filt, extra), rate)
    W = o.width
    ext = rng.integers(-32768, 32767, size=(ext_lines * W + W // 3, 2), dtype=np.int16)
    o.open_test_source()
    o.set_passthru(ext)
    got = o.render(30)
    o.close()
    fn = tmp_path / "ext.iq"
    ext.tofile(fn)
    assert_reference(got, _key("passthru", mode, rate, filt, ext_lines, *extra), mode, rate, 30, vfilter=filt,
                     extra=tuple(extra) + ("--passthru", str(fn)))
    o = orc.Oracle(_conf(built, mode, filt, extra), rate)
    o.open_test_source()
    plain = o.render(30)
    o.close()
    assert_reference(plain, _key("plain", mode, rate, 30, filt, *extra), mode, rate, 30, vfilter=filt, extra=extra)
    assert not np.array_equal(plain, got)


def wss_overlay(built, mode, rate, wss="16:9"):
    """What the reference's WSS stage does to line 23 (wss.c:154-193): part of the line set to black, then the
    bit waveform added. Recovered from the reference itself: unfiltered, no sound, no colour (the SECAM stage
    runs after WSS and would filter it), with and without --wss."""
    conf = built.mode_config(mode, noaudio=True)
    t = built.Tables(conf, rate)
    W, half = int(t.get("geometry")[0]), int(t.get("geometry")[1])
    black = int(t.get("levels")[1])
    t.close()
    per = 2 if conf.output_type == 0 else 1

    def line23(x):
        return x.reshape(30, W, per)[22, :, 0]
    plain = reference_values(_key("line23", mode, rate), mode, rate, 30, extra=("--noaudio", "--nocolour"),
                             view=line23).astype(np.int32)
    with_wss = reference_values(_key("line23 wss", mode, rate, wss), mode, rate, 30,
                                extra=("--noaudio", "--nocolour", "--wss", wss), view=line23).astype(np.int32)
    blank_to = int(round(rate * 42.5e-6))
    base = plain.copy()
    base[half:blank_to] = black
    return (with_wss - base).astype(np.int16), (half, blank_to, black)


@pytest.mark.parametrize("mode,rate,filt,extra", [("i", 16000000, True, ()), ("pal", 16000000, False, ()),
                                                  ("l", 16000000, True, ()), ("secam", 16000000, False, ())])
def test_vbi_overlay_is_where_the_reference_puts_wss(built, mode, rate, filt, extra):
    """The overlay hook (after the raster, before SECAM / filter / sound) carries the reference's own WSS
    waveform to exactly the reference's --wss output, in modes other than the one it was recovered from."""
    add, rep = wss_overlay(built, mode, rate)
    assert np.count_nonzero(add) > 100
    o = orc.Oracle(_conf(built, mode, filt, extra), rate)
    o.open_test_source()
    o.add_vbi_line(23, add, rep)
    got = o.render(700)
    o.close()
    assert_reference(got, _key("wss", mode, rate, 700, filt, *extra), mode, rate, 700, vfilter=filt,
                     extra=tuple(extra) + ("--wss", "16:9"))


def test_oracle_equals_reference_on_random_input(built):
    rng = np.random.default_rng(7)
    conf = built.mode_config("i", vfilter=True)
    o = orc.Oracle(conf, 16000000)
    frames = rng.integers(0, 1 << 24, size=(2, o.active_lines, o.active_width), dtype=np.uint32)
    audio = rng.integers(-32768, 32767, size=(30000, 2), dtype=np.int16)
    o.set_source(frames, audio)
    got = o.render(1400)
    o.close()
    assert_reference(got, "random i 16000000 1400", "i", 16000000, 1400, vfilter=True, frames=frames, audio=audio,
                     audio_block=4000)


def test_unpatched_heap_differs_only_near_line_ends(built):
    """The stock allocator lets the chroma FIR read past its buffer (SURVEY.md §8c): the
    masked comparison - everything further than 32 samples from a line boundary - is exact
    (against the oracle, which equals the zero-heap build everywhere: test_oracle_equals_reference)."""
    def masked(x):
        return x.reshape(700, 1024, 2)[:, 32:-32]
    o = orc.Oracle(built.mode_config("i", vfilter=True), 16000000)
    o.open_test_source()
    got = masked(o.render(700))
    o.close()
    assert_reference(got, "rawheap masked i 16000000 700 True", "i", 16000000, 700, vfilter=True, rawheap=True,
                     view=masked)


# --pixelrate (SURVEY.md section 8f rank 4): raster at the pixel rate, the reference's polyphase resampler
# (video.c:3627-3651, fir.c:393-428) to the sample rate in front of the video filter. The oracle restates the
# rate pairs that keep the line width constant; the CUDA path does not take them yet (htv_init refuses).
PIXELRATE_CASES = [
    ("pal", 16000000, 13500000, 700, False, ()),                 # 864 -> 1024 samples per line, I/D = 32/27
    ("i", 16000000, 13500000, 700, True, ()),                    # + VSB filter, FM + NICAM two lines ahead
    ("i", 16000000, 13500000, 400, False, ()),                   # resampler alone: one line ahead
    ("i", 16000000, 13500000, 400, True, ("--offset", "2000000")),
    ("i", 20000000, 13500000, 400, True, ()),                    # 40/27
    ("i", 13500000, 16000000, 400, True, ()),                    # resampling down, 27/32
    ("i", 16000000, 14000000, 300, True, ()),                    # 8/7
    ("m", 13500000, 9000000, 400, True, ()),                     # NTSC, 3/2
    ("l", 16000000, 13500000, 700, True, ()),                    # SECAM: the FIRs' reads past the line end find the blanking level
    ("l", 13500000, 16000000, 300, True, ()),
    ("secam", 16000000, 13500000, 400, False, ()),
    ("d", 20000000, 13500000, 300, True, ()),
]


@pytest.mark.parametrize("mode,rate,prate,nlines,filt,extra", PIXELRATE_CASES)
def test_pixelrate_resampler_equals_reference(built, mode, rate, prate, nlines, filt, extra):
    o = orc.Oracle(_conf(built, mode, filt, extra), rate, prate)
    o.open_test_source()
    got = o.render(nlines)
    o.close()
    assert_reference(got, _key("pixelrate", mode, rate, prate, nlines, filt, *extra), mode, rate, nlines, vfilter=filt,
                     extra=tuple(extra) + ("--pixelrate", str(prate)))


def test_pixelrate_later_window_and_random_input(built):
    """A window two frames in (phase of the polyphase filter, NICAM frame counter) and random pictures + audio."""
    conf = built.mode_config("i", vfilter=True)
    o = orc.Oracle(conf, 16000000, 13500000)
    o.open_test_source()
    got = o.render(1700)[1400 * 2048:]
    o.close()
    assert_reference(got, "pixelrate skip 1400 i 16000000 13500000 300 True", "i", 16000000, 300, skip=1400,
                     vfilter=True, extra=("--pixelrate", "13500000"))
    rng = np.random.default_rng(5)
    o = orc.Oracle(conf, 16000000, 13500000)
    frames = rng.integers(0, 1 << 24, size=(2, o.active_lines, o.active_width), dtype=np.uint32)
    audio = rng.integers(-32768, 32767, size=(30000, 2), dtype=np.int16)
    o.set_source(frames, audio)
    got = o.render(900)
    o.close()
    assert_reference(got, "pixelrate random i 16000000 13500000 900 True", "i", 16000000, 900, vfilter=True,
                     frames=frames, audio=audio, audio_block=4000, extra=("--pixelrate", "13500000"))


def test_pixelrate_with_passthru_and_wss(built, tmp_path):
    """Two fill lines in front of the stream (resampler + filter): the passthru stage spends two external
    lines on them; the VBI stages sit in front of the resampler."""
    rng = np.random.default_rng(3)
    conf = built.mode_config("i", vfilter=True)
    o = orc.Oracle(conf, 16000000, 13500000)
    ext = rng.integers(-32768, 32767, size=(40 * o.width + 100, 2), dtype=np.int16)
    o.open_test_source()
    o.set_passthru(ext)
    got = o.render(30)
    o.close()
    fn = tmp_path / "ext.iq"
    ext.tofile(fn)
    assert_reference(got, "pixelrate passthru i 16000000 13500000 30 True", "i", 16000000, 30, vfilter=True,
                     extra=("--pixelrate", "13500000", "--passthru", str(fn)))

    add, rep = wss_overlay(built, "pal", 13500000)               # the waveform at the pixel rate
    o = orc.Oracle(built.mode_config("pal"), 16000000, 13500000)
    o.open_test_source()
    o.add_vbi_line(23, add, rep)
    got = o.render(100)
    o.close()
    assert_reference(got, "pixelrate wss pal 16000000 13500000 100 False", "pal", 16000000, 100,
                     extra=("--pixelrate", "13500000", "--wss", "16:9"))


def test_pixelrate_pairs_the_oracle_does_not_restate(built):
    with pytest.raises(RuntimeError):
        orc.Oracle(built.mode_config("i", vfilter=True), 16000000, 13400000)    # line width would vary
    with pytest.raises(RuntimeError):
        orc.Oracle(built.mode_config("pal-fm", vfilter=True), 20000000, 13500000)
