"""Builds the FLAC fixtures of tests/test_hostio.py, cut from the libFLAC-encoded files the reference ships under
test/utterance, so that the tests need no reference checkout:

    python tests/golden/make_flac_golden.py <reference checkout>

flac_libflac_excerpt.npz: a short stream (LPC subframes) cut from test/utterance/original/original.flac (the input of
the reference's test/test.py:48-57), plus the PCM it must decode to, from its sibling original.wav, which holds the
same 132300 samples as plain PCM -- an independent decode.

flac_reference_excerpts.npz: every distinct .flac under test/utterance (inputs, outputs, targets), each as its
metadata chain exactly as shipped (STREAMINFO with libFLAC's MD5 signature of the whole file) and as a stream of its
first, middle and last frames.  The frames' audio comes from a full decode of the file that matched that signature
(and, for original.flac, original.wav); the excerpt's STREAMINFO carries its sample count and MD5.

FLAC frames are self-contained, so STREAMINFO + some of the frames are a valid stream once total_samples and the
MD5 signature in STREAMINFO are rewritten for the excerpt.
"""
import glob
import hashlib
import os
import sys
import wave

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
NFRAMES = 2
OUT = os.path.join(HERE, "flac_libflac_excerpt.npz")
OUT_ALL = os.path.join(HERE, "flac_reference_excerpts.npz")


def crc8(b):
    c = 0
    for x in b:
        c ^= x
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
    return c


def frame_offset(data, start, number):
    """Offset of the fixed-blocksize frame with the given frame number (< 128): sync, number byte, header CRC-8."""
    i = start
    while True:
        i = data.index(b"\xff\xf8", i)
        bs_code, sr_code = data[i + 2] >> 4, data[i + 2] & 15
        n = 5 + {6: 1, 7: 2}.get(bs_code, 0) + {12: 1, 13: 2, 14: 2}.get(sr_code, 0)
        if data[i + 4] == number and crc8(data[i:i + n]) == data[i + n]:
            return i
        i += 1


def audio_offset(data):
    """Offset of the first frame: the end of the metadata chain."""
    off, last = 4, False
    while not last:
        last, ln = bool(data[off] >> 7), int.from_bytes(data[off + 1:off + 4], "big")
        off += 4 + ln
    return off


def with_streaminfo(data, nsamp, pcm):
    """data's metadata chain with total_samples and the MD5 signature rewritten for nsamp samples of int16 pcm."""
    head = bytearray(data[:audio_offset(data)])
    info = head[8:42]
    info[13] = (info[13] & 0xF0) | ((nsamp >> 32) & 0x0F)
    info[14:18] = (nsamp & 0xFFFFFFFF).to_bytes(4, "big")
    info[18:34] = hashlib.md5(pcm.astype("<i2").tobytes()).digest()
    head[8:42] = info
    return bytes(head)


def libflac_excerpt(orig):
    data = open(os.path.join(orig, "original.flac"), "rb").read()
    assert data[:4] == b"fLaC" and data[4] & 0x7F == 0 and data[5:8] == b"\x00\x00\x22"
    off = audio_offset(data)
    first, end = frame_offset(data, off, 0), frame_offset(data, off, NFRAMES)
    assert first == off
    blocksize = int.from_bytes(data[8:10], "big")
    nsamp = NFRAMES * blocksize
    with wave.open(os.path.join(orig, "original.wav"), "rb") as w:
        pcm = np.frombuffer(w.readframes(nsamp), dtype="<i2").copy()
    info = bytearray(data[8:42])
    info[13] = (info[13] & 0xF0) | ((nsamp >> 32) & 0x0F)
    info[14:18] = (nsamp & 0xFFFFFFFF).to_bytes(4, "big")
    info[18:34] = hashlib.md5(pcm.astype("<i2").tobytes()).digest()
    stream = b"fLaC" + bytes([0x80, 0, 0, 34]) + bytes(info) + data[first:end]
    np.savez_compressed(OUT, flac=np.frombuffer(stream, dtype=np.uint8), pcm=pcm,
                        source="test/utterance/original/original.flac frames 0..%d" % (NFRAMES - 1))
    print(OUT, len(stream), "bytes,", nsamp, "samples")


def reference_excerpts(utt):
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from voicefixer_b200 import _hostio, build
    build.build_hostio()
    with wave.open(os.path.join(utt, "original", "original.wav"), "rb") as w:
        wav = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
    fixture, files, digests = {}, [], set()
    for path in sorted(glob.glob(os.path.join(utt, "*", "*.flac"))):
        data = open(path, "rb").read()
        if hashlib.sha256(data).digest() in digests:              # outputs and targets are mostly the same files
            continue
        digests.add(hashlib.sha256(data).digest())
        info = _hostio.flac_info(data)
        full, _, _ = _hostio.flac_decode(data)                     # raises unless it matches libFLAC's MD5 signature
        assert hashlib.md5(full.astype("<i2").tobytes()).digest() == bytes(info.md5)
        name = os.path.relpath(path, utt)
        if name == os.path.join("original", "original.flac"):
            assert np.array_equal(full[:, 0], wav)
        bs, n = int(info.max_blocksize), int(info.total_samples)
        assert info.min_blocksize == bs and info.channels == 1
        nframes = -(-n // bs)
        frames = [0, nframes // 2, nframes - 1]
        off = audio_offset(data)
        starts = [frame_offset(data, off, k) for k in range(nframes)] + [len(data)]
        pcm = np.concatenate([full[k * bs:(k + 1) * bs, 0] for k in frames]).astype(np.int16)
        i = len(files)
        files.append(name)
        fixture[f"header{i}"] = np.frombuffer(data[:off], dtype=np.uint8)
        fixture[f"excerpt{i}"] = np.frombuffer(with_streaminfo(data, len(pcm), pcm)
                                               + b"".join(data[starts[k]:starts[k + 1]] for k in frames), dtype=np.uint8)
        fixture[f"frames{i}"] = np.array(frames)
        if name == os.path.join("original", "original.flac"):
            fixture["original_wav"] = pcm
    fixture["files"] = np.array(files)
    np.savez_compressed(OUT_ALL, **fixture)
    print(OUT_ALL, os.path.getsize(OUT_ALL), "bytes,", len(files), "files")


def main(ref):
    utt = os.path.join(ref, "test", "utterance")
    libflac_excerpt(os.path.join(utt, "original"))
    reference_excerpts(utt)


if __name__ == "__main__":
    main(sys.argv[1])
