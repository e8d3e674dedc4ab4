"""Host-side FLAC codec (include/vfx_hostio.h, libvfx_hostio.so) behind the file API.

The reference's acceptance test is FLAC in / FLAC out through librosa.load and soundfile.write
(test/test.py:48-57,85-89; voicefixer/base.py:47-49; tools/wav.py:37).  The decoder is pinned by
(a) a libFLAC-encoded excerpt of the reference's own test input with the PCM of its sibling .wav
(tests/golden/flac_libflac_excerpt.npz, made by tests/golden/make_flac_golden.py), (b) frames of
every .flac the reference ships, against the header and MD5 signatures libFLAC stored in STREAMINFO
(tests/golden/flac_reference_excerpts.npz, same script), and (c) hashlib for the MD5 itself.  The
encoder is pinned by the decoder."""
import hashlib
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_hostio_library_exports_every_declared_symbol():
    from voicefixer_b200 import _hostio
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vfx_hostio.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(vfx_[a-z_0-9]+)\s*\(", hdr))
    lib = _hostio.load()
    assert declared and all(hasattr(lib, n) for n in declared)
    assert declared == set(_hostio.SIGNATURES)


def test_hostio_header_is_valid_c99_and_struct_layout_matches(tmp_path):
    import ctypes, shutil, subprocess
    from voicefixer_b200 import _hostio
    src = tmp_path / "t.c"
    src.write_text('#include <stdio.h>\n#include "vfx_hostio.h"\nint main(void){printf("%zu %zu %zu",sizeof(vfx_flac_info),'
                   '__builtin_offsetof(vfx_flac_info,md5),__builtin_offsetof(vfx_flac_info,audio_offset));return 0;}\n')
    exe = tmp_path / "t"
    subprocess.run([shutil.which("gcc"), "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, off_md5, off_audio = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert size == ctypes.sizeof(_hostio.FlacInfo)
    assert off_md5 == _hostio.FlacInfo.md5.offset and off_audio == _hostio.FlacInfo.audio_offset.offset


def test_md5_matches_hashlib():
    import ctypes
    from voicefixer_b200 import _hostio
    lib = _hostio.load()
    rng = np.random.default_rng(3)
    for n in (0, 1, 55, 56, 57, 63, 64, 65, 119, 120, 1000, 70001):
        data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        out = (ctypes.c_uint8 * 16)()
        lib.vfx_md5(data, n, out)
        assert bytes(out) == hashlib.md5(data).digest(), n


def test_decode_libflac_excerpt_golden():
    """LPC subframes + Rice partitions written by libFLAC, checked against the sibling WAV's PCM."""
    from voicefixer_b200 import _hostio
    g = np.load(os.path.join(ROOT, "tests", "golden", "flac_libflac_excerpt.npz"))
    data = g["flac"].tobytes()
    info = _hostio.flac_info(data)
    assert (info.sample_rate, info.channels, info.bits_per_sample, info.total_samples) == (44100, 1, 16, g["pcm"].shape[0])
    assert bytes(info.md5) == hashlib.md5(g["pcm"].astype("<i2").tobytes()).digest()
    pcm, sr, bps = _hostio.flac_decode(data)
    assert sr == 44100 and bps == 16 and np.array_equal(pcm[:, 0], g["pcm"])


def test_decode_detects_corruption():
    from voicefixer_b200 import _hostio
    g = np.load(os.path.join(ROOT, "tests", "golden", "flac_libflac_excerpt.npz"))
    good = bytearray(g["flac"].tobytes())
    for pos, what in ((len(good) // 2, "CRC-16"), (42 + 2, "CRC-8"), (len(good) - 1, "CRC-16")):
        bad = bytearray(good)
        bad[pos] ^= 0x10
        with pytest.raises(RuntimeError, match=what):
            _hostio.flac_decode(bytes(bad))
    with pytest.raises(RuntimeError, match="stream ends after|truncated|bitstream ended|CRC"):
        _hostio.flac_decode(bytes(good[: len(good) - 700]))
    bad = bytearray(good)
    bad[30] ^= 0xFF                                               # inside the MD5 signature
    with pytest.raises(RuntimeError, match="MD5"):
        _hostio.flac_decode(bytes(bad))
    with pytest.raises(RuntimeError, match="fLaC"):
        _hostio.flac_decode(b"RIFF" + bytes(100))


SIGNALS = {
    "noise": lambda rng, n, ch: rng.integers(-32768, 32768, (n, ch)),
    "tone": lambda rng, n, ch: (12000 * np.sin(2 * np.pi * 220 * np.arange(n)[:, None] / 44100) + rng.normal(0, 20, (n, ch))).astype(np.int64),
    "silence": lambda rng, n, ch: np.zeros((n, ch), dtype=np.int64),
    "dc": lambda rng, n, ch: np.full((n, ch), -7, dtype=np.int64),
    "rails": lambda rng, n, ch: np.where(rng.random((n, ch)) < 0.5, -32768, 32767),
    "quiet": lambda rng, n, ch: rng.integers(-3, 4, (n, ch)),
}


@pytest.mark.parametrize("n", [0, 1, 4, 5, 255, 256, 257, 4095, 4096, 4097, 3 * 4096 + 17])
@pytest.mark.parametrize("ch", [1, 2])
def test_encode_decode_roundtrip_is_bit_exact(n, ch):
    """Empty, ragged last block, every subframe choice (constant / verbatim / fixed 0-4), stereo."""
    from voicefixer_b200 import _hostio
    rng = np.random.default_rng(n * 2 + ch)
    for name, make in SIGNALS.items():
        x = make(rng, n, ch).astype(np.int16)
        data = _hostio.flac_encode_int16(x, 44100 if name != "quiet" else 12345)
        info = _hostio.flac_info(data)
        assert info.total_samples == n and info.channels == ch and info.bits_per_sample == 16
        assert bytes(info.md5) == hashlib.md5(x.astype("<i2").tobytes()).digest()
        y, sr, bps = _hostio.flac_decode(data)
        assert y.shape == (n, ch) and np.array_equal(y, x), name
        if n >= 4096 and name in ("tone", "silence", "quiet"):
            assert len(data) < 0.6 * x.nbytes                      # it does compress


def test_long_stream_frame_numbers_use_multibyte_coding():
    """> 2048 frames: the UTF-8 style frame number takes 1, 2 and 3 bytes along the stream."""
    from voicefixer_b200 import _hostio
    x = (np.arange(4096 * 2100) % 251 - 125).astype(np.int16)
    y, _, _ = _hostio.flac_decode(_hostio.flac_encode_int16(x, 44100))
    assert np.array_equal(y[:, 0], x)


def test_wavio_flac_follows_the_file_extension(tmp_path):
    """save_wave -> .flac has tools/wav.py:9-37 semantics (x 2^15, int16 truncation); load_mono reads it back
    like librosa.load (float32 in [-1, 1), mono mix), and a .wav of the same frames loads identically."""
    from voicefixer_b200 import wavio
    rng = np.random.default_rng(0)
    x = (0.3 * rng.standard_normal((1, 30000))).clip(-1, 1).astype(np.float32)
    wavio.save_wave(x, str(tmp_path / "a.flac"), 44100)
    wavio.save_wave(x, str(tmp_path / "a.wav"), 44100)
    assert (tmp_path / "a.flac").read_bytes()[:4] == b"fLaC"
    yf, yw = wavio.load_mono(str(tmp_path / "a.flac")), wavio.load_mono(str(tmp_path / "a.wav"))
    assert yf.dtype == np.float32 and np.array_equal(yf, yw)
    assert np.array_equal((yf * 32768).astype(np.int16), (x[0] * 2 ** 15).astype(np.short))
    stereo = np.stack([x[0], -0.5 * x[0]], axis=1)                   # [samples, 2] -> two channels
    wavio.save_wave(stereo, str(tmp_path / "s.flac"), 22050)
    r = wavio.read_wave(str(tmp_path / "s.flac"), 22050)
    assert r.shape == (30000, 2)
    m = wavio.load_mono(str(tmp_path / "s.flac"), 44100)             # resampled mono mix, like librosa.load(sr=44100)
    assert m.shape == (60000,)


def test_decode_every_reference_flac_against_its_libflac_md5(tmp_path):
    """Every distinct FLAC file the reference ships (inputs, targets, outputs), as tests/golden/make_flac_golden.py
    stored it: the metadata chain libFLAC wrote (header fields, the sample counts BASELINE.md quotes, an MD5
    signature), and the file's first, middle and last frames with frame CRCs and the MD5 of those frames' audio,
    taken from a full decode that matched libFLAC's signature; original.flac's frames == original.wav's samples."""
    from voicefixer_b200 import _hostio, wavio
    g = np.load(os.path.join(ROOT, "tests", "golden", "flac_reference_excerpts.npz"))
    files = [str(f) for f in g["files"]]
    assert len(files) >= 6
    expect = {"original.flac": 132300, "p360_001_mic1.flac": 96076, "oracle.flac": 97902, "output_mode_0.flac": 132300,
              "output_mode_1.flac": 132096, "output_mode_2.flac": 132300}
    for i, f in enumerate(files):
        info = _hostio.flac_info(g[f"header{i}"].tobytes())
        n, bs = expect[os.path.basename(f)], info.max_blocksize
        assert (info.sample_rate, info.channels, info.bits_per_sample, info.total_samples) == (44100, 1, 16, n), f
        assert any(info.md5), f
        data = g[f"excerpt{i}"].tobytes()
        pcm, sr, bps = _hostio.flac_decode(data)                     # raises on CRC / MD5 mismatch
        want = sum(min(bs, n - k * bs) for k in g[f"frames{i}"])
        assert g[f"frames{i}"][-1] == (n - 1) // bs                  # the ragged last block is among them
        assert (sr, bps, pcm.shape) == (44100, 16, (want, 1)), f
        assert hashlib.md5(pcm.astype("<i2").tobytes()).digest() == bytes(_hostio.flac_info(data).md5)
        if os.path.basename(f) == "original.flac":
            (tmp_path / "original.flac").write_bytes(data)
            got = wavio.load_mono(str(tmp_path / "original.flac"))
            assert np.array_equal(got, g["original_wav"].astype(np.float32) / 32768.0)


# ------------------------------------------------------------------ decoder paths no available file reaches
def _decode(data):
    from voicefixer_b200 import _hostio
    pcm, sr, bps = _hostio.flac_decode(data)
    return pcm, sr, bps


def test_decode_stereo_decorrelation_modes():
    """left/side (8), side/right (9), mid/side (10): the side channel carries bps + 1 bits."""
    import flac_writer as W
    rng = np.random.default_rng(1)
    n = 192
    left = rng.integers(-32768, 32768, n).tolist()
    right = rng.integers(-32768, 32768, n).tolist()
    left[0], right[0], left[1], right[1] = 32767, -32768, -32768, 32767            # extreme side values
    side = [l - r for l, r in zip(left, right)]
    mid = [(l + r) >> 1 for l, r in zip(left, right)]
    inter = [v for lr in zip(left, right) for v in lr]
    plans = {8: (left, 16, side, 17), 9: (side, 17, right, 16), 10: (mid, 16, side, 17), 1: (left, 16, right, 16)}
    for ch_code, (c0, b0, c1, b1) in plans.items():
        fr = W.frame(0, n, ch_code, 16, [lambda b, c0=c0, b0=b0: W.sub_verbatim(b, c0, b0),
                                         lambda b, c1=c1, b1=b1: W.sub_verbatim(b, c1, b1)])
        pcm, sr, bps = _decode(W.stream([fr], 44100, 2, 16, n, inter))
        assert np.array_equal(pcm[:, 0], left) and np.array_equal(pcm[:, 1], right), ch_code


@pytest.mark.parametrize("bps", [8, 12, 20, 24])
def test_decode_other_bit_depths_and_scaling(bps, tmp_path):
    import flac_writer as W
    from voicefixer_b200 import wavio
    rng = np.random.default_rng(bps)
    lo, hi = -(1 << (bps - 1)), (1 << (bps - 1))
    x = rng.integers(lo, hi, 256).tolist()
    x[0], x[1] = lo, hi - 1
    fr = W.frame(0, 256, 0, bps, [lambda b: W.sub_verbatim(b, x, bps)], ss_from_info=(bps == 12))
    data = W.stream([fr], 48000, 1, bps, 256, x)
    pcm, sr, got_bps = _decode(data)
    assert (sr, got_bps) == (48000, bps) and np.array_equal(pcm[:, 0], x)
    (tmp_path / "d.flac").write_bytes(data)
    y = wavio.read_wave(str(tmp_path / "d.flac"), 48000)                           # float32 in [-1, 1)
    assert y.shape == (256, 1) and y[0, 0] == -1.0 and abs(y[1, 0] - (hi - 1) / hi) < 1e-7


def test_decode_subframe_types_partitions_and_escape_codes():
    """CONSTANT, wasted bits, FIXED 0-4 with partitioned Rice (4- and 5-bit parameters) and escape partitions
    (raw n-bit residuals, n = 0 included), LPC with explicit precision / shift."""
    import flac_writer as W
    rng = np.random.default_rng(7)
    n = 256
    t = np.arange(n)
    smooth = (9000 * np.sin(2 * np.pi * t / 57.0) + 30 * rng.standard_normal(n)).astype(int).tolist()
    cases = []
    cases.append(("constant", lambda b: W.sub_constant(b, [-1234] * n, 16), [-1234] * n))
    w = (rng.integers(-2000, 2000, n) * 8).tolist()
    cases.append(("wasted3", lambda b: W.sub_verbatim(b, w, 16, wasted=3), w))
    for order in range(5):
        cases.append((f"fixed{order}", lambda b, o=order: W.sub_fixed(b, smooth, 16, o, 2, [9, 8, 10, 9]), smooth))
    cases.append(("rice2", lambda b: W.sub_fixed(b, smooth, 16, 1, 1, [17, 3], method=1), smooth))
    cases.append(("escape", lambda b: W.sub_fixed(b, smooth, 16, 2, 2, [8, ("esc", 14), 9, ("esc", 13)]), smooth))
    ramp = [3 * i - 100 for i in range(n)]                                         # order-2 residual is all zero
    cases.append(("escape0", lambda b: W.sub_fixed(b, ramp, 16, 2, 1, [("esc", 0), ("esc", 0)]), ramp))
    cases.append(("lpc", lambda b: W.sub_lpc(b, smooth, 16, [117, -60, 5], 8, 6, 3, [7] * 8), smooth))
    cases.append(("lpc32", lambda b: W.sub_lpc(b, smooth, 16, [1] * 32, 3, 5, 0, [15], method=1), smooth))
    for name, sub, expect in cases:
        pcm, _, _ = _decode(W.stream([W.frame(0, n, 0, 16, [sub])], 44100, 1, 16, n, expect))
        assert np.array_equal(pcm[:, 0], expect), name


def test_decode_frame_header_variants():
    """Blocksize codes (table, 8-bit, 16-bit), sample-rate codes (table, kHz byte, Hz, tens of Hz), fixed and variable
    blocking with multi-byte frame / sample numbers, unknown total_samples, unset MD5, trailing bytes after the audio."""
    import flac_writer as W
    rng = np.random.default_rng(11)

    def verb(x):
        return [lambda b: W.sub_verbatim(b, x, 16)]

    blocks = [(192, {}), (576, {}), (256, {}), (100, dict(bs_explicit=8)), (1000, dict(bs_explicit=16)), (17, dict(bs_explicit=8))]
    xs = [rng.integers(-500, 500, n).tolist() for n, _ in blocks]
    total = sum(n for n, _ in blocks)
    flat = [v for x in xs for v in x]
    # variable blocking: the header number is the first sample of the frame (here offset so it needs 2-5 bytes)
    frames, pos = [], 0
    for (n, kw), x in zip(blocks, xs):
        frames.append(W.frame(pos, n, 0, 16, verb(x), variable=True, sr_code=9, **kw))
        pos += n
    pcm, sr, _ = _decode(W.stream(frames, 44100, 1, 16, total, flat))
    assert sr == 44100 and np.array_equal(pcm[:, 0], flat)
    for number in (0x7F, 0x80, 0x7FF, 0x800, 0xFFFF, 0x10000, 0x1FFFFF, 0x200000, 0x3FFFFFF, 0x4000000, 0x7FFFFFFF):
        fr = W.frame(number, 192, 0, 16, verb(xs[0]))
        assert np.array_equal(_decode(W.stream([fr], 44100, 1, 16, 192, xs[0]))[0][:, 0], xs[0]), hex(number)
    big = W.frame((1 << 35) + 5, 192, 0, 16, verb(xs[0]), variable=True)            # 36-bit sample number, 7 bytes
    assert np.array_equal(_decode(W.stream([big], 44100, 1, 16, 192, xs[0]))[0][:, 0], xs[0])
    for sr, code, extra in ((32000, 12, bytes([32])), (12345, 13, (12345).to_bytes(2, "big")), (22050, 14, (2205).to_bytes(2, "big")),
                            (96000, 11, b""), (8000, 4, b"")):
        fr = W.frame(0, 192, 0, 16, verb(xs[0]), sr_code=code, sr_extra=extra)
        pcm, got_sr, _ = _decode(W.stream([fr], sr, 1, 16, 192, xs[0]))
        assert got_sr == sr and np.array_equal(pcm[:, 0], xs[0])
    # unknown length + no signature + junk after the last frame (e.g. an ID3v1 tag)
    frames = [W.frame(i, 192, 0, 16, verb(xs[0])) for i in range(3)]
    pcm, _, _ = _decode(W.stream(frames, 44100, 1, 16, 0, None) + b"TAG" + bytes(125))
    assert pcm.shape == (576, 1) and np.array_equal(pcm[:192, 0], xs[0]) and np.array_equal(pcm[384:, 0], xs[0])


def test_decode_rejects_reserved_fields():
    import flac_writer as W
    from voicefixer_b200 import _hostio
    x = list(range(192))

    def one(mutate):
        b = W.Bits()
        mutate(b)
        return b

    bad_type = lambda b: (b.put(0, 1), b.put(2, 6), b.put(0, 1), [b.signed(v, 16) for v in x])          # reserved subframe type
    with pytest.raises(RuntimeError, match="reserved subframe type"):
        _hostio.flac_decode(W.stream([W.frame(0, 192, 0, 16, [bad_type])], 44100, 1, 16, 192, x))
    bad_method = lambda b: (b.put(0, 1), b.put(8, 6), b.put(0, 1), b.put(2, 2), b.put(0, 4))            # residual method 2
    with pytest.raises(RuntimeError, match="reserved residual coding method"):
        _hostio.flac_decode(W.stream([W.frame(0, 192, 0, 16, [bad_method])], 44100, 1, 16, 192, x))
    with pytest.raises(RuntimeError, match="channel"):                                                      # 2 channels in a mono stream
        fr = W.frame(0, 192, 1, 16, [lambda b: W.sub_verbatim(b, x, 16)] * 2)
        _hostio.flac_decode(W.stream([fr], 44100, 1, 16, 192, x))


def test_flac_roundtrip_property_random_walks():
    """Property test (hypothesis): any int16 signal of any length / channel count / rate survives encode -> decode
    bit-exactly, the STREAMINFO signature matches hashlib, and truncating the stream anywhere is detected."""
    from hypothesis import given, settings, strategies as st
    from voicefixer_b200 import _hostio

    @settings(max_examples=60, deadline=None)
    @given(st.integers(0, 9000), st.integers(1, 3), st.integers(0, 2 ** 31 - 1), st.sampled_from([1, 7, 300, 5000, 40000]),
           st.sampled_from([8000, 22050, 44100, 48000, 12345]))
    def check(n, ch, seed, step, sr):
        rng = np.random.default_rng(seed)
        x = np.clip(np.cumsum(rng.integers(-step, step + 1, (n, ch)), axis=0), -32768, 32767).astype(np.int16)
        data = _hostio.flac_encode_int16(x, sr)
        y, got_sr, bps = _hostio.flac_decode(data)
        assert got_sr == sr and bps == 16 and y.shape == (n, ch) and np.array_equal(y, x)
        assert bytes(_hostio.flac_info(data).md5) == hashlib.md5(x.astype("<i2").tobytes()).digest()
        if n > 0:
            cut = 42 + int(rng.integers(0, len(data) - 42))
            with pytest.raises(RuntimeError):
                _hostio.flac_decode(data[:cut])

    check()


def test_decoder_survives_random_corruption():
    """Bit flips and truncation of valid streams either decode or raise RuntimeError -- never crash the process
    (tools/fuzz_flac.c is the long-running version under ASan / UBSan, including CRC-repaired corruptions)."""
    from voicefixer_b200 import _hostio
    rng = np.random.default_rng(99)
    g = np.load(os.path.join(ROOT, "tests", "golden", "flac_libflac_excerpt.npz"))
    seeds = [g["flac"].tobytes(), _hostio.flac_encode_int16(rng.integers(-3000, 3000, (6000, 2)).astype(np.int16), 44100)]
    outcomes = {"ok": 0, "rejected": 0}
    for it in range(400):
        data = bytearray(seeds[it % 2])
        for _ in range(int(rng.integers(1, 5))):
            data[int(rng.integers(0, len(data)))] ^= 1 << int(rng.integers(0, 8))
        if it % 4 == 0:
            data = data[: int(rng.integers(0, len(data)))]
        try:
            _hostio.flac_decode(bytes(data))
            outcomes["ok"] += 1
        except RuntimeError:
            outcomes["rejected"] += 1
    assert outcomes["rejected"] > 300
