"""Pins oracle/flac_oracle.c (the CPU restatement) against the compiled, unmodified
reference libFLAC (oracle/_ref/*.so, built by oracle/Makefile), through its answers stored
in tests/golden/reference.json.gz (tests/refdata.py).

The reference's own tests do not pin encoder bytes (SURVEY.md §0.6: only round trips and
size monotonicity, test/test_streams.sh:52-79), so encoder parity is pinned by running the
reference side by side, frame by frame. Decoder parity is pinned by round trips.

Gates (SURVEY.md §7.3-1):
  G1  100 % frame parity vs the source-order-FP build (libFLAC_ref_strict.so) on every input.
  G2  100 % frame parity vs the shipped-flags build (libFLAC_ref.so) on noise-bearing inputs.
  G3  noise-free tonal stress inputs: mismatch rate vs the shipped-flags build is reported
      (the reference does not reproduce those bytes across its own dispatch paths).
"""
import numpy as np
import pytest

import oraclelib
import refdata
import reflib
import signals


def _frames_equal(x, bps, rate, level, bs=0, variant="strict", opts=None, **cfg_over):
    ref = refdata.encode(x, bps, rate=rate, level=level, blocksize=bs, variant=variant, opts=opts)
    enc = oraclelib.Encoder(oraclelib.preset(x.shape[1], bps, rate, level, bs, **cfg_over))
    got = enc.encode_stream(x)
    bad = ref.mismatches(got)
    return bad, ref, got


@pytest.mark.parametrize("level", range(9))
def test_all_levels_16bit_stereo_both_builds(level):
    x = signals.music_like(4096 * 6 + 777, 2, 16, 44100, seed=1)
    for variant in ("strict", "default"):
        bad, _, _ = _frames_equal(x, 16, 44100, level, variant=variant)
        assert bad == [], f"{variant}: mismatching frames {bad}"


@pytest.mark.parametrize("level", [0, 3, 5, 8])
@pytest.mark.parametrize("ch,bps,rate", [(1, 16, 44100), (2, 24, 96000), (8, 24, 192000), (3, 20, 48000), (2, 8, 22050), (1, 12, 8000)])
def test_depths_and_channel_counts(level, ch, bps, rate):
    n = 4096 * 3 + 123
    x = signals.music_like(n, ch, bps, rate, seed=11 + ch)
    for variant in ("strict", "default"):
        bad, _, _ = _frames_equal(x, bps, rate, level, variant=variant)
        assert bad == [], f"{variant}: mismatching frames {bad}"


@pytest.mark.parametrize("bs", [16, 17, 32, 33, 192, 256, 576, 1000, 1152, 2304, 4608, 8192, 16384])
@pytest.mark.parametrize("level", [2, 5, 8])
def test_blocksizes(bs, level):
    x = signals.music_like(max(3 * bs + bs // 3, 600), 2, 16, 44100, seed=3)
    opts = reflib.RefEncOpts(streamable_subset=0)
    bad, _, _ = _frames_equal(x, 16, 44100, level, bs=bs, opts=opts)
    assert bad == []


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
    "left_only": lambda: np.ascontiguousarray(np.stack([signals.music_like(9000, 1, 16, seed=4)[:, 0], np.zeros(9000, np.int32)], axis=1)),
    "identical_lr": lambda: np.ascontiguousarray(np.repeat(signals.music_like(9000, 1, 16, seed=4), 2, axis=1)),
}


@pytest.mark.parametrize("name", sorted(STRESS))
@pytest.mark.parametrize("level", [1, 5, 8])
def test_stress_inputs(name, level):
    x = STRESS[name]()
    bps = 24 if name.endswith("24") else 16
    for variant in ("strict", "default"):
        bad, _, _ = _frames_equal(x, bps, 44100, level, variant=variant)
        assert bad == [], f"{variant}: mismatching frames {bad}"


def test_option_matrix():
    x = signals.music_like(4096 * 3 + 99, 2, 16, 44100, seed=2)
    cases = [
        (dict(exhaustive=1), dict(do_exhaustive_model_search=1), 5),
        (dict(exhaustive=1), dict(do_exhaustive_model_search=1), 8),
        (dict(mid_side=0), dict(do_mid_side=0), 8),
        (dict(loose_mid_side=1), dict(loose_mid_side=1), 8),
        (dict(max_lpc_order=32, streamable_subset=0), dict(max_lpc_order=32), 8),
        (dict(qlp_precision=9), dict(qlp_coeff_precision=9), 5),
        (dict(min_part_order=2, max_part_order=8), dict(min_residual_partition_order=2, max_residual_partition_order=8), 5),
        (dict(limit_min_bitrate=1), dict(limit_min_bitrate=1), 5),
        (dict(prec_search=1), dict(do_qlp_coeff_prec_search=1), 5),
        (dict(prec_search=1), dict(do_qlp_coeff_prec_search=1), 8),
    ]
    for ref_kw, cfg_kw, level in cases:
        bad, _, _ = _frames_equal(x, 16, 44100, level, opts=reflib.RefEncOpts(**ref_kw), **cfg_kw)
        assert bad == [], f"{ref_kw}: {bad}"
    # limit_min_bitrate acts on constant frames
    z = signals.silence(4096 * 2, 2)
    bad, _, _ = _frames_equal(z, 16, 44100, 5, opts=reflib.RefEncOpts(limit_min_bitrate=1), limit_min_bitrate=1)
    assert bad == []


def test_tonal_stress_reported_not_gated():
    """G3: pure tones make the LPC normal equations near-singular; the shipped-flags build
    reassociates its FP sums, so only the source-order build is gated."""
    x = signals.sine(4096 * 6, 1, 16, 44100, freq=1000.0, freq2=1001.3)
    bad_strict, _, _ = _frames_equal(x, 16, 44100, 8, variant="strict")
    assert bad_strict == []
    bad_default, ref_frames, _ = _frames_equal(x, 16, 44100, 8, variant="default")
    print(f"two-tone -8: {len(bad_default)}/{len(ref_frames)} frames differ from the shipped-flags build")


@pytest.mark.parametrize("level", [0, 5, 8])
@pytest.mark.parametrize("ch,bps", [(1, 16), (2, 16), (2, 24), (8, 24)])
def test_decoder_round_trip(level, ch, bps):
    """Decoder pin: reference-encoded frames -> oracle decoder == original PCM, and
    oracle-encoded frames -> reference decoder (through a reference-made header) round trip."""
    x = signals.music_like(4096 * 2 + 500, ch, bps, 48000, seed=21)
    ref = refdata.encode(x, bps, rate=48000, level=level, header=True)
    mine = oraclelib.Encoder(oraclelib.preset(ch, bps, 48000, level)).encode_stream(x)
    y = oraclelib.decode_frames(b"".join(ref.frames(witness=mine)), ch, bps, 48000, x.shape[0])
    assert np.array_equal(x, y)
    z = refdata.decode(ref.header + b"".join(mine), x.shape[0], ch)
    assert z.info[3] == 0 and z.matches(x)


def test_decoder_stress_round_trip():
    for name in sorted(STRESS):
        x = STRESS[name]()
        bps = 24 if name.endswith("24") else 16
        ref = refdata.encode(x, bps, level=8)
        witness = oraclelib.Encoder(oraclelib.preset(x.shape[1], bps, 44100, 8)).encode_stream(x)
        y = oraclelib.decode_frames(b"".join(ref.frames(witness)), x.shape[1], bps, 44100, x.shape[0])
        assert np.array_equal(x, y), name


def test_crc_known_answers():
    """CRC KATs: CRC-8 poly 0x07 and CRC-16 poly 0x8005, init 0, no reflection
    (/root/reference/src/libFLAC/crc.c:39-76, 78-342). Check value for '123456789'."""
    L = oraclelib.lib()
    msg = np.frombuffer(b"123456789", dtype=np.uint8).copy()
    assert L.fo_crc8(msg.ctypes.data, 9) == 0xF4      # CRC-8/SMBUS
    assert L.fo_crc16(msg.ctypes.data, 9) == 0xFEE8   # CRC-16/UMTS (BUYPASS)
