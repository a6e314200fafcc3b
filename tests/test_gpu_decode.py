"""GPU parity tests for the decode path (through the C ABI, host buffers): decoded PCM must be
bit-exact (a) to the original PCM for frames produced by the compiled reference encoder, by the
oracle and by our own encoder, and (b) to the oracle decoder on hand-made frames that exercise
paths the reference encoder never emits (escape partitions)."""
import numpy as np
import pytest

import oraclelib
import refdata
import reflib
import signals

pytestmark = pytest.mark.gpu


def _offsets(frames):
    offs = np.zeros(len(frames) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(f) for f in frames])
    return np.frombuffer(b"".join(frames), dtype=np.uint8).copy(), offs


def _gpu_decode(frames, ch, bps, rate, bs, total):
    import flac_b200
    dec = flac_b200.Decoder(ch, bps, rate, bs)
    try:
        stream, offs = _offsets(frames)
        return dec.decode(stream, offs, total_samples=total)
    finally:
        dec.close()


def _encoded_frames(x, bps, rate, level, bs=0, source="oracle"):
    enc = oraclelib.Encoder(oraclelib.preset(x.shape[1], bps, rate, level, bs))
    frames = enc.encode_stream(x)
    if source == "reference":  # the reference's frames (tests/refdata.py): the oracle's, checked to be exactly those
        return refdata.encode(x, bps, rate=rate, level=level, blocksize=bs, opts=reflib.RefEncOpts(streamable_subset=0)).frames(witness=frames)
    return frames


@pytest.mark.parametrize("level", range(9))
def test_levels_stereo16(level):
    x = signals.music_like(4096 * 5 + 321, 2, 16, 44100, seed=1)
    frames = _encoded_frames(x, 16, 44100, level, source="reference")
    bs = 1152 if level < 3 else 4096
    y = _gpu_decode(frames, 2, 16, 44100, bs, x.shape[0])
    assert np.array_equal(x, y)


@pytest.mark.parametrize("level", [0, 5, 8])
@pytest.mark.parametrize("ch,bps,rate", [(1, 16, 44100), (2, 24, 96000), (8, 24, 192000), (3, 20, 48000), (2, 8, 22050), (1, 12, 8000)])
def test_depths_and_channel_counts(level, ch, bps, rate):
    x = signals.music_like(4096 * 2 + 77, ch, bps, rate, seed=11 + ch)
    frames = _encoded_frames(x, bps, rate, level, source="reference")
    bs = 1152 if level < 3 else 4096
    y = _gpu_decode(frames, ch, bps, rate, bs, x.shape[0])
    assert np.array_equal(x, y)


@pytest.mark.parametrize("bs", [16, 33, 192, 1000, 4608, 8192, 16384])
def test_blocksizes(bs):
    x = signals.music_like(3 * bs + bs // 3, 2, 16, 44100, seed=3)
    frames = _encoded_frames(x, 16, 44100, 8, bs)
    assert np.array_equal(x, _gpu_decode(frames, 2, 16, 44100, bs, x.shape[0]))


STRESS = {
    "white_noise_fs": lambda: signals.white_noise(4096 * 2, 2, 16, seed=5),
    "white_noise_24": lambda: signals.white_noise(4096 * 2, 2, 24, seed=6),
    "silence": lambda: signals.silence(4096 * 2 + 5, 2),
    "dc_mono_neg": lambda: signals.dc(5000, 1, -32768),
    "wasted3": lambda: signals.wasted_bits(4096 * 2, 2, 16, 3),
    "fsd": lambda: signals.full_scale_deflection(4096 * 2, 2, 16, 7),
    "sine24": lambda: signals.sine(4096 * 2, 2, 24, 96000, freq=997.0),
    "left_only": lambda: np.ascontiguousarray(np.stack([signals.music_like(9000, 1, 16, seed=4)[:, 0], np.zeros(9000, np.int32)], axis=1)),
}


@pytest.mark.parametrize("name", sorted(STRESS))
@pytest.mark.parametrize("level", [1, 8])
def test_stress_inputs(name, level):
    x = STRESS[name]()
    bps = 24 if name.endswith("24") else 16
    frames = _encoded_frames(x, bps, 44100, level)
    bs = 1152 if level < 3 else 4096
    assert np.array_equal(x, _gpu_decode(frames, x.shape[1], bps, 44100, bs, x.shape[0]))


def test_high_order_and_exhaustive():
    x = signals.music_like(4096 * 2, 2, 16, 44100, seed=2)
    enc = oraclelib.Encoder(oraclelib.preset(2, 16, 44100, 8, max_lpc_order=32, do_exhaustive_model_search=0))
    frames = enc.encode_stream(x)
    assert np.array_equal(x, _gpu_decode(frames, 2, 16, 44100, 4096, x.shape[0]))


class _BW:
    def __init__(self):
        self.bits = []

    def put(self, v, n):
        for i in range(n - 1, -1, -1):
            self.bits.append((v >> i) & 1)

    def bytes(self):
        b = self.bits + [0] * (-len(self.bits) % 8)
        return bytes(int("".join(map(str, b[i:i + 8])), 2) for i in range(0, len(b), 8))


def _handmade_escape_frame(samples, bps=16, frame_number=0):
    """Mono frame, FIXED order 1, partition order 1: partition 0 Rice k=3, partition 1 ESCAPED
    with raw 7-bit residuals (stream_decoder.c:3334-3350). Built bit by bit."""
    L = oraclelib.lib()
    bs = len(samples)
    assert bs == 32
    w = _BW()
    w.put(0x3ffe, 14); w.put(0, 1); w.put(0, 1)
    w.put(6, 4)            # blocksize: 8-bit (bs-1) follows
    w.put(9, 4)            # 44.1 kHz
    w.put(0, 4)            # mono
    w.put(4, 3)            # 16 bit
    w.put(0, 1)
    w.put(frame_number, 8)
    w.put(bs - 1, 8)
    hdr = np.frombuffer(w.bytes(), dtype=np.uint8).copy()
    w.put(L.fo_crc8(hdr.ctypes.data, hdr.size), 8)
    w.put(0x10 | (1 << 1), 8)                    # FIXED order 1, no wasted bits
    w.put(samples[0] & 0xffff, bps)              # warm-up
    res = [samples[i] - samples[i - 1] for i in range(1, bs)]
    w.put(0, 2); w.put(1, 4)                     # RICE, partition order 1
    w.put(3, 4)                                  # partition 0: k = 3, 15 residuals
    for r in res[:15]:
        u = (r << 1) ^ (r >> 31) if r >= 0 else ((-r) << 1) - 1
        w.put(0, u >> 3); w.put(1, 1); w.put(u & 7, 3)
    w.put(15, 4); w.put(7, 5)                    # partition 1: escape, 7 raw bits
    for r in res[15:]:
        assert -64 <= r < 64
        w.put(r & 0x7f, 7)
    body = np.frombuffer(w.bytes(), dtype=np.uint8).copy()
    crc = L.fo_crc16(body.ctypes.data, body.size)
    return body.tobytes() + bytes([crc >> 8, crc & 0xff])


def test_escape_partition_handmade_frame():
    rng = np.random.default_rng(3)
    steps = rng.integers(-20, 21, size=32)
    samples = [int(v) for v in np.cumsum(steps)]
    fr = _handmade_escape_frame(samples)
    want = oraclelib.decode_frames(fr, 1, 16, 44100, 32)
    assert [int(v) for v in want[:, 0]] == samples
    got = _gpu_decode([fr], 1, 16, 44100, 32, 32)
    assert np.array_equal(got, want)


def test_corruption_is_detected():
    import flac_b200
    x = signals.music_like(4096 * 4, 2, 16, 44100, seed=9)
    frames = _encoded_frames(x, 16, 44100, 5)
    bad = bytearray(frames[2])
    bad[len(bad) // 2] ^= 0x10
    frames2 = list(frames)
    frames2[2] = bytes(bad)
    dec = flac_b200.Decoder(2, 16, 44100, 4096)
    stream, offs = _offsets(frames2)
    with pytest.raises(flac_b200.FlacB200Error):
        dec.decode(stream, offs)
    # the undamaged frames still decode when looked at one by one
    s0, o0 = _offsets(frames2[:2])
    assert np.array_equal(dec.decode(s0, o0), x[:8192])
    dec.close()


def test_encode_decode_round_trip_full_size():
    """cfg5-sized property: 100 000 stereo frames encoded (-8) and decoded on the GPU give back the input."""
    import flac_b200
    nblocks = 100000
    base = signals.music_like(4096 * 40, 2, 16, 44100, seed=5)
    x = np.ascontiguousarray(np.tile(base, (nblocks // 40, 1)))
    x[::5, 1] ^= 1
    enc = flac_b200.Encoder(flac_b200.preset(2, 16, 44100, 8), max_blocks_per_launch=4096)
    stream, offs = enc.encode(x)
    enc.close()
    dec = flac_b200.Decoder(2, 16, 44100, 4096)
    y = dec.decode(stream, offs)
    dec.close()
    assert y.shape == x.shape and np.array_equal(x, y)


def test_gpu_front_end_index_with_junk_around_frames():
    """fb200_decoder_index_host + fb200_decode_indexed_host: frames are found with no caller-supplied offsets, junk in front of,
    between and behind them (ID3v1-style tag) costs nothing, every frame's true length comes out of the parse."""
    import flac_b200
    x = signals.music_like(4096 * 6 + 1000, 2, 16, 44100, seed=13)
    frames = _encoded_frames(x, 16, 44100, 8)
    junk0, junk1, tag = b"\x00\x01\x02" * 11, b"\xff\xf8junk-that-looks-like-sync\xff\xf9" * 3, b"TAG" + b"\x55" * 125
    blob, starts = bytearray(junk0), []
    for i, f in enumerate(frames):
        starts.append(len(blob))
        blob += f
        if i == 2:
            blob += junk1
    blob += tag
    dec = flac_b200.Decoder(2, 16, 44100, 4096)
    try:
        cand = dec.index(np.frombuffer(bytes(blob), dtype=np.uint8))
        assert set(starts) <= set(int(c) for c in cand), "a true frame start is missing from the candidates"
        pcm, st, fb = dec.decode_indexed(cand, 2 * 4096 * 2 * 3)
        good = {int(c): i for i, c in enumerate(cand) if (st[i] & 0xff) == 0}
        assert sorted(good) == starts, f"accepted {sorted(good)} expected {starts}"
        y = np.concatenate([pcm[good[s] * 4096: good[s] * 4096 + (int(st[good[s]]) >> 8)] for s in starts])
        assert np.array_equal(y, x)
        assert [int(fb[good[s]]) for s in starts] == [len(f) for f in frames]
    finally:
        dec.close()


def test_subframe_info_matches_the_encoders_plan():
    """FLAC__Frame.subframes[] material: type / order / precision / shift / partition order / coefficients / warm-up reported by the
    decode kernels equal what the encoder decided (its plans) for every subframe of every frame."""
    import flac_b200
    x = signals.music_like(4096 * 4, 2, 16, 44100, seed=31)
    enc = flac_b200.Encoder(flac_b200.preset(2, 16, 44100, 8))
    stream, offs = enc.encode(x)
    plans, ca = enc.debug_plans(4)
    enc.close()
    dec = flac_b200.Decoder(2, 16, 44100, 4096)
    try:
        dec.enable_subframe_info(True)
        y = dec.decode(stream, offs)
        assert np.array_equal(x, y)
        info = dec.subframe_info(4)
        for f in range(4):
            a = int(ca[f])
            sel = [(0 if a in (0, 1) else (3 if a == 2 else 2)), (1 if a in (0, 2) else 3)]
            for c in range(2):
                p, i = plans[f * 4 + sel[c]], info[f * 2 + c]
                want_type = {0: 0, 1: 1, 2: 2, 3: 3}[p.type]
                assert i.type == want_type and i.wasted_bits == p.wasted
                if p.type >= 2:
                    assert i.order == p.order and i.partition_order == p.porder and i.entropy_method == p.method
                if p.type == 3:
                    assert i.qlp_coeff_precision == p.precision and i.quantization_level == p.shift
                    assert list(i.qlp_coeff[:p.order]) == list(p.qlp[:p.order])
    finally:
        dec.close()


def test_truncated_and_lying_frames_never_read_past_their_end():
    """A frame whose header claims more data than the buffer holds (valid CRC-8, truncated body) is reported, not decoded;
    the neighbours decode. (Bit reader returns zeros past the frame end: no out-of-bounds read.)"""
    import flac_b200
    x = signals.music_like(4096 * 3, 2, 16, 44100, seed=23)
    frames = _encoded_frames(x, 16, 44100, 5)
    cut = frames[1][: len(frames[1]) // 3]
    stream, offs = _offsets([frames[0], cut, frames[2]])
    dec = flac_b200.Decoder(2, 16, 44100, 4096)
    try:
        with pytest.raises(flac_b200.FlacB200Error):
            dec.decode(stream, offs)
        st = dec.frame_status(3)
        assert (st[0] & 0xff) == 0 and (st[1] & 0xff) != 0 and (st[2] & 0xff) == 0
    finally:
        dec.close()


@pytest.mark.parametrize("ch,bps,nbytes", [(2, 16, 2), (2, 24, 3), (1, 12, 2), (8, 24, 3), (2, 16, 3), (3, 20, 3)])
def test_packed_output_and_chunked_host_path(ch, bps, nbytes):
    """fb200_decode_host_packed: the samples arrive as packed little-endian 16-/24-bit PCM; the host path decodes in chunks of
    frames (>= 1024 per chunk: 2500 frames make three), and the per-frame records line up across chunks."""
    import flac_b200
    bs = 256
    x = signals.music_like(bs * 2500 + 77, ch, bps, 44100, seed=41)
    enc = flac_b200.Encoder(flac_b200.preset(ch, bps, 44100, 5, bs))
    stream, offs = enc.encode(x)
    enc.close()
    dec = flac_b200.Decoder(ch, bps, 44100, bs)
    try:
        dec.enable_subframe_info(True)
        packed, ns = dec.decode_packed(stream, offs, nbytes)
        assert ns == x.shape[0]
        assert np.array_equal(packed, flac_b200.pack_pcm(x, nbytes))
        nfr = offs.size - 1
        st = dec.frame_status(nfr)
        assert np.all((st & 0xff) == 0) and int(st[0] >> 8) == bs and int(st[-1] >> 8) == 77
        info = dec.subframe_info(nfr)
        ref = flac_b200.Decoder(ch, bps, 44100, bs)
        try:
            ref.enable_subframe_info(True)
            # frames 2400.. decoded on their own: their records must equal the tail of the chunked call's
            y = ref.decode(stream[int(offs[2400]):], offs[2400:] - offs[2400])
            assert np.array_equal(y, x[2400 * bs:])
            tail = ref.subframe_info(nfr - 2400)
            for a, b in zip(info[2400 * ch:], tail):
                assert (a.type, a.order, a.wasted_bits, a.partition_order) == (b.type, b.order, b.wasted_bits, b.partition_order)
        finally:
            ref.close()
        assert np.array_equal(dec.decode(stream, offs), x)
    finally:
        dec.close()
