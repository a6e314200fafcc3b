"""GPU parity tests proper: the CUDA encode path (through the C ABI, host buffers) against
 (1) the CPU restatement oracle/flac_oracle.c, and
 (2) the compiled reference libFLAC (oracle/_ref/*.so), through its answers stored in
     tests/golden/reference.json.gz (tests/refdata.py),
frame by frame, bit-exact."""
import numpy as np
import pytest

import oraclelib
import refdata
import reflib
import signals

pytestmark = pytest.mark.gpu


def _gpu_frames(x, bps, rate, level, bs=0, **over):
    import flac_b200
    enc = flac_b200.Encoder(flac_b200.preset(x.shape[1], bps, rate, level, bs, **over))
    try:
        return enc.encode_frames(x)
    finally:
        enc.close()


def _oracle_frames(x, bps, rate, level, bs=0, **over):
    enc = oraclelib.Encoder(oraclelib.preset(x.shape[1], bps, rate, level, bs, **over))
    return enc.encode_stream(x)


def _assert_same(got, want, what):
    assert len(got) == len(want), f"{what}: frame count {len(got)} != {len(want)}"
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, f"{what}: {len(bad)}/{len(want)} frames differ, first {bad[:5]}"


def _assert_reference(got, ref, what):
    """got: frames; ref: the reference's answer (refdata.Encoding)."""
    assert len(got) == len(ref), f"{what}: frame count {len(got)} != {len(ref)}"
    bad = ref.mismatches(got)
    assert not bad, f"{what}: {len(bad)}/{len(ref)} frames differ, first {bad[:5]}"


@pytest.mark.parametrize("level", range(9))
def test_levels_16bit_stereo_vs_oracle_and_reference(level):
    x = signals.music_like(4096 * 10 + 777, 2, 16, 44100, seed=1)
    got = _gpu_frames(x, 16, 44100, level)
    _assert_same(got, _oracle_frames(x, 16, 44100, level), "oracle")
    for variant in ("strict", "default"):
        _assert_reference(got, refdata.encode(x, 16, rate=44100, level=level, variant=variant), f"reference[{variant}]")


@pytest.mark.parametrize("level", [0, 3, 5, 8])
@pytest.mark.parametrize("ch,bps,rate", [(1, 16, 44100), (2, 24, 96000), (8, 24, 192000), (3, 20, 48000), (2, 8, 22050), (1, 12, 8000)])
def test_depths_and_channel_counts(level, ch, bps, rate):
    x = signals.music_like(4096 * 3 + 123, ch, bps, rate, seed=11 + ch)
    got = _gpu_frames(x, bps, rate, level)
    _assert_same(got, _oracle_frames(x, bps, rate, level), "oracle")
    _assert_reference(got, refdata.encode(x, bps, rate=rate, level=level), "reference[default]")


@pytest.mark.parametrize("bs", [16, 17, 32, 33, 192, 256, 576, 1000, 1024, 1152, 2048, 2304, 3072, 4608, 5120, 6144, 8192, 9216])
@pytest.mark.parametrize("level", [2, 5, 8])
def test_blocksizes(bs, level):
    x = signals.music_like(max(3 * bs + bs // 3, 600), 2, 16, 44100, seed=3)
    got = _gpu_frames(x, 16, 44100, level, bs)
    _assert_same(got, _oracle_frames(x, 16, 44100, level, bs), "oracle")


STRESS = {
    "white_noise_fs": lambda: signals.white_noise(4096 * 3, 2, 16, seed=5),
    "white_noise_24": lambda: signals.white_noise(4096 * 3, 2, 24, seed=6),
    "silence": lambda: signals.silence(4096 * 3 + 5, 2),
    "dc": lambda: signals.dc(4096 * 3, 2, 1234),
    "dc_mono_neg": lambda: signals.dc(5000, 1, -32768),
    "wasted3": lambda: signals.wasted_bits(4096 * 3, 2, 16, 3),
    "fsd": lambda: signals.full_scale_deflection(4096 * 2, 2, 16, 7),
    "noisy_sine": lambda: signals.noisy_sine(4096 * 3, 2, 16),
    "quiet_noise": lambda: signals.white_noise(4096 * 2, 2, 16, seed=9, scale=0.0002),
    "two_tone": lambda: signals.sine(4096 * 4, 1, 16, 44100, freq=1000.0, freq2=1001.3),
    "sine24": lambda: signals.sine(4096 * 3, 2, 24, 96000, freq=997.0),
    "left_only": lambda: np.ascontiguousarray(np.stack([signals.music_like(9000, 1, 16, seed=4)[:, 0], np.zeros(9000, np.int32)], axis=1)),
    "identical_lr": lambda: np.ascontiguousarray(np.repeat(signals.music_like(9000, 1, 16, seed=4), 2, axis=1)),
}


@pytest.mark.parametrize("name", sorted(STRESS))
@pytest.mark.parametrize("level", [1, 5, 8])
def test_stress_inputs(name, level):
    x = STRESS[name]()
    bps = 24 if name.endswith("24") else 16
    got = _gpu_frames(x, bps, 44100, level)
    _assert_same(got, _oracle_frames(x, bps, 44100, level), "oracle")
    _assert_reference(got, refdata.encode(x, bps, rate=44100, level=level, variant="strict"), "reference[strict]")


def test_option_matrix():
    x = signals.music_like(4096 * 3 + 99, 2, 16, 44100, seed=2)
    cases = [
        (dict(do_exhaustive_model_search=1), dict(do_exhaustive_model_search=1), 5),
        (dict(do_exhaustive_model_search=1), dict(do_exhaustive_model_search=1), 8),
        (dict(do_mid_side_stereo=0), dict(do_mid_side=0), 8),
        (dict(loose_mid_side_stereo=1), dict(loose_mid_side=1), 8),
        (dict(max_lpc_order=32), dict(max_lpc_order=32), 8),
        (dict(qlp_coeff_precision=9), dict(qlp_coeff_precision=9), 5),
        (dict(min_residual_partition_order=2, max_residual_partition_order=8), dict(min_residual_partition_order=2, max_residual_partition_order=8), 5),
        (dict(disable_constant_subframes=1), dict(disable_constant_subframes=1), 5),
        (dict(disable_fixed_subframes=1), dict(disable_fixed_subframes=1), 5),
        (dict(disable_verbatim_subframes=1), dict(disable_verbatim_subframes=1), 0),
    ]
    for gpu_kw, or_kw, level in cases:
        got = _gpu_frames(x, 16, 44100, level, **gpu_kw)
        _assert_same(got, _oracle_frames(x, 16, 44100, level, **or_kw), str(gpu_kw))


def test_multi_launch_chunking_and_frame_numbers():
    """More blocks than one launch holds + a non-zero first frame number (UTF-8 header widths)."""
    import flac_b200
    x = signals.music_like(1152 * 23 + 5, 2, 16, 44100, seed=8)
    enc = flac_b200.Encoder(flac_b200.preset(2, 16, 44100, 2), max_blocks_per_launch=4)
    stream, offs = enc.encode(x, first_frame_number=0)
    want = _oracle_frames(x, 16, 44100, 2)
    got = [stream[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(len(offs) - 1)]
    _assert_same(got, want, "chunked")
    # large frame numbers: compare single frames against the oracle at that number
    o = oraclelib.Encoder(oraclelib.preset(2, 16, 44100, 2))
    for first in (127, 128, 2047, 2048, 65535, 65536, 0x1FFFFF, 0x200000, 0x3FFFFFF, 0x4000000, 0x7FFFFFF0):
        g = enc.encode_frames(x[:1152 * 2], first_frame_number=first)
        for j in range(2):
            assert g[j] == o.encode_frame(x[1152 * j:1152 * (j + 1)], first + j), f"frame number {first + j}"
    enc.close()


def test_reference_decoder_accepts_gpu_stream():
    """flac -t equivalent: the reference decoder decodes our frames (behind a reference-made
    stream header) to the original PCM with no errors."""
    for ch, bps, level in ((2, 16, 8), (2, 24, 8), (1, 16, 5), (8, 24, 5)):
        x = signals.music_like(4096 * 3 + 50, ch, bps, 48000, seed=31)
        header = refdata.encode(x, bps, rate=48000, level=level, header=True).header
        mine = b"".join(_gpu_frames(x, bps, 48000, level))
        y = refdata.decode(header + mine, x.shape[0], ch)
        assert y.info[3] == 0 and y.matches(x)


def test_big_batch_property_round_trip():
    """BASELINE cfg2-sized property check (10 000 blocks stereo 16-bit -5): every frame decodes
    (oracle decoder on a sample of frames, CRC-16 verified) back to the input."""
    import flac_b200
    nblocks = 10000
    base = signals.music_like(4096 * 50, 2, 16, 44100, seed=1)
    x = np.ascontiguousarray(np.tile(base, (nblocks // 50, 1)))
    x[::7, 0] ^= 1  # break the periodicity a little
    enc = flac_b200.Encoder(flac_b200.preset(2, 16, 44100, 5), max_blocks_per_launch=4096)
    stream, offs = enc.encode(x)
    assert len(offs) == nblocks + 1
    rng = np.random.default_rng(0)
    for i in rng.choice(nblocks, 200, replace=False):
        fr = stream[int(offs[i]):int(offs[i + 1])].tobytes()
        y = oraclelib.decode_frames(fr, 2, 16, 44100, 4096)
        assert np.array_equal(y, x[i * 4096:(i + 1) * 4096]), f"frame {i}"
    enc.close()


@pytest.mark.parametrize("level,ch,bps", [(8, 2, 16), (5, 2, 24), (5, 1, 16), (2, 2, 16), (8, 2, 24)])
def test_general_kernels_equal_fast_kernels(monkeypatch, level, ch, bps):
    """FB200_FORCE_GENERAL_KERNELS=1 runs the general kernels (any blocksize) on a blocksize the fast kernels
    (k_autoc3 / k_search4 / k_emit3) normally take: both must give the oracle's frames."""
    monkeypatch.setenv("FB200_FORCE_GENERAL_KERNELS", "1")
    x = signals.music_like(4096 * 3 + 55, ch, bps, 44100, seed=17)
    got = _gpu_frames(x, bps, 44100, level)
    _assert_same(got, _oracle_frames(x, bps, 44100, level), "general kernels")


@pytest.mark.parametrize("bps", [16, 12, 24, 20])
@pytest.mark.parametrize("mlo", [13, 16, 17, 20, 24, 32])
def test_search4_orders_13_to_32(bps, mlo):
    """k_search4's 32-tap instantiation (max_lpc_order 13..32) is the default for every regular blocksize.
    Round 1 kept orders > 12 on the previous kernel generation because a first version of k_search4 mis-evaluated
    orders > 16; that version handled the warm-up samples with a masked first tile (group-relative order mask for
    MAXORD > G), which commit ef78d8c replaced by one unmasked pass + a warm-up correction. This matrix
    (tools/probe_search4_32.py is the longer form: 108 configurations, 0 of 432 frames differ) pins it."""
    for bs, ex in ((4096, 0), (4608, 0), (1024, 0), (2304, 0), (4096, 1)):
        if ex and mlo > 17:
            continue
        over = dict(max_lpc_order=mlo)
        if ex:
            over["do_exhaustive_model_search"] = 1
        x = signals.music_like(bs * 2 + 99, 2, bps, 44100, seed=2 + mlo % 5)
        got = _gpu_frames(x, bps, 44100, 8, bs, **over)
        _assert_same(got, _oracle_frames(x, bps, 44100, 8, bs, **over), f"bps {bps} max_lpc_order {mlo} bs {bs} exhaustive {ex}")


@pytest.mark.parametrize("bps,nbytes,ch", [(16, 2, 2), (12, 2, 2), (24, 3, 2), (20, 3, 1), (16, 3, 2), (16, 2, 1)])
def test_packed_pcm_entry_point(bps, nbytes, ch):
    """fb200_encode_host_packed (16-/24-bit little-endian PCM, widened on the device) == the int32 entry point == oracle."""
    import flac_b200
    n = 4096 * 5 + 1234 + (1 if nbytes == 3 else 0)  # odd byte offsets for the short last block too
    x = signals.music_like(n, ch, bps, 44100, seed=21)
    enc = flac_b200.Encoder(flac_b200.preset(ch, bps, 44100, 5), max_blocks_per_launch=2)
    try:
        stream, offs = enc.encode_packed(flac_b200.pack_pcm(x, nbytes), nbytes, n)
        got = [stream[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(len(offs) - 1)]
    finally:
        enc.close()
    _assert_same(got, _oracle_frames(x, bps, 44100, 5), f"packed {nbytes} bytes/sample")


def test_packed_pcm_out_of_range_sample_fails():
    import flac_b200
    x = signals.music_like(4096 * 2, 2, 16, 44100, seed=3)  # 16-bit samples into a 12-bit stream
    enc = flac_b200.Encoder(flac_b200.preset(2, 12, 44100, 5))
    try:
        with pytest.raises(flac_b200.FlacB200Error) as ei:
            enc.encode_packed(flac_b200.pack_pcm(x, 2), 2, x.shape[0])
        assert ei.value.code == -3
    finally:
        enc.close()


@pytest.mark.parametrize("ch,bps,level", [(2, 16, 5), (8, 24, 8), (1, 16, 8)])
def test_file_blocks_restarts_frame_numbers(ch, bps, level):
    """Many-file batches: with set_file_blocks(n) every run of n blocks is numbered like its own stream
    (reference: one encoder per file, frame_number from 0, stream_encoder.c:3772)."""
    import flac_b200
    per_file, files = 6, 3
    x = signals.music_like(4096 * per_file * files, ch, bps, 44100, seed=5)
    enc = flac_b200.Encoder(flac_b200.preset(ch, bps, 44100, level), max_blocks_per_launch=7)
    try:
        enc.set_file_blocks(per_file)
        got = enc.encode_frames(x)
    finally:
        enc.close()
    want = []
    for f in range(files):
        want += _oracle_frames(x[f * per_file * 4096:(f + 1) * per_file * 4096], bps, 44100, level)
    _assert_same(got, want, "file-major frame numbering")


@pytest.mark.parametrize("ch,bps,level,bs", [(2, 16, 5, 0), (2, 16, 8, 0), (2, 16, 0, 0), (2, 16, 1, 0), (1, 16, 5, 0), (3, 20, 5, 0),
                                            (8, 24, 8, 0), (2, 24, 5, 0), (2, 16, 5, 1000), (2, 16, 2, 4608)])
def test_limit_min_bitrate(ch, bps, level, bs):
    """stream_encoder.c:3874-3879: a frame must not consist of constant subframes only -- blocks of digital silence, of a DC
    level, with one constant and one live channel, and ordinary audio, against the oracle and the compiled reference."""
    blk = bs or 4096
    x = signals.music_like(blk * 8 + 311, ch, bps, 44100, seed=23)
    x[blk:2 * blk] = 0                       # silence: every channel constant
    x[2 * blk:3 * blk] = 37                  # DC: constant, non-zero (mid constant, side zero)
    x[3 * blk:4 * blk, 0] = -5               # first channel constant, the others live
    x[4 * blk:5 * blk, ch - 1] = 9           # last channel constant, the others live
    x[6 * blk:7 * blk] = np.arange(ch)[None, :] * 3   # every channel its own constant
    got = _gpu_frames(x, bps, 44100, level, bs, limit_min_bitrate=1)
    _assert_same(got, _oracle_frames(x, bps, 44100, level, bs, limit_min_bitrate=1), "oracle")
    plain = _gpu_frames(x, bps, 44100, level, bs)
    if level != 1:  # loose mid-side: the constant frames are coded mid/side only, outside the independent-channel loop
        assert plain != got, "limit_min_bitrate changed nothing"
    ref = refdata.encode(x, bps, rate=44100, level=level, blocksize=bs, opts=reflib.RefEncOpts(limit_min_bitrate=1))
    _assert_reference(got, ref, "reference[default]")


@pytest.mark.parametrize("ch,bps,level,bs,exhaustive", [(2, 16, 5, 0, 0), (2, 16, 8, 0, 0), (2, 24, 5, 0, 0), (1, 16, 3, 0, 0), (2, 16, 5, 1152, 1),
                                                       (8, 24, 8, 0, 0), (2, 16, 5, 1000, 0), (2, 20, 8, 4608, 0)])
def test_qlp_coeff_precision_search(ch, bps, level, bs, exhaustive):
    """flac -p (stream_encoder.c:4230-4243): every order is quantised at precisions 5 .. 15, in the reference's evaluation order."""
    x = signals.music_like((bs or 4096) * 3 + 311, ch, bps, 44100, seed=29)
    kw = dict(do_qlp_coeff_prec_search=1, do_exhaustive_model_search=exhaustive)
    got = _gpu_frames(x, bps, 44100, level, bs, **kw)
    _assert_same(got, _oracle_frames(x, bps, 44100, level, bs, **kw), "oracle")
    assert got != _gpu_frames(x, bps, 44100, level, bs, do_exhaustive_model_search=exhaustive), "precision search changed nothing"
    opts = reflib.RefEncOpts(prec_search=1, exhaustive=exhaustive if exhaustive else -1)
    _assert_reference(got, refdata.encode(x, bps, rate=44100, level=level, blocksize=bs, opts=opts, variant="strict"), "reference[strict]")
