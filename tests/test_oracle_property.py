"""Property check (CPU): for randomly drawn configurations the oracle's frames equal the compiled reference's
(source-order FP build), frame for frame. Deterministic (derandomized hypothesis), bounded to a few seconds.
The reference's frames are its answers stored in tests/golden/reference.json.gz (tests/refdata.py)."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, seed, settings, strategies as st

import oraclelib
import refdata
import reflib
import signals

APODS = [None, "tukey(0.5)", "subdivide_tukey(3)", "hann", "welch;gauss(0.3)", "partial_tukey(2/0.2);punchout_tukey(2)", "rectangle;triangle", "tukey(0.1);connes"]
SIGNALS = ["music_like", "white_noise", "noisy_sine", "wasted_bits"]
# Fixed example sets: the ones derandomized Hypothesis drew for the first version of each test. The stored
# reference answers cover exactly these, and editing a test must not change what it draws.
SEED_RANDOM_CONFIGURATIONS = 0xf773a649452f823b1c0d266cfb7fe5db2051d6e1db4b0c32a9078bf52850b37fcc40444b4de9f5501c5443c9b1104464
SEED_PRECISION_SEARCH = 0x293c74b5dfda01fdbd48f4ca3703c5935d67052e77590cf3955c83a6082dcccba37af45d1b7a51265c7f2b8d32179303


def _signal(kind, n, ch, bps, seed):
    if kind == "music_like":
        return signals.music_like(n, ch, bps, 44100, seed=seed)
    if kind == "white_noise":
        return signals.white_noise(n, ch, bps, seed=seed, scale=0.05)
    if kind == "noisy_sine":
        return signals.noisy_sine(n, ch, bps)
    return signals.wasted_bits(n, ch, bps, 2)


@seed(SEED_RANDOM_CONFIGURATIONS)
@settings(max_examples=400, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
@given(ch=st.integers(1, 2), bps=st.sampled_from([8, 12, 16, 20, 24]), level=st.integers(0, 8),
       bs=st.sampled_from([0, 192, 576, 1000, 1152, 2048, 4096, 4608]), kind=st.sampled_from(SIGNALS), seed=st.integers(1, 50),
       apod=st.sampled_from(APODS), exhaustive=st.booleans(), max_order=st.sampled_from([None, 4, 10, 16, 32]),
       precision=st.sampled_from([None, 7, 11, 14]), po=st.sampled_from([None, (0, 3), (2, 2), (0, 8)]), loose=st.booleans())
def test_oracle_equals_reference_on_random_configurations(ch, bps, level, bs, kind, seed, apod, exhaustive, max_order, precision, po, loose):
    bsz = bs or (1152 if level < 3 else 4096)
    n = bsz * 2 + 37
    x = _signal(kind, n, ch, bps, seed)
    okw, rkw = {}, {}
    if apod:
        okw["apodization"] = rkw["apodization"] = apod
    if exhaustive and (max_order or 8) <= 10:  # keep the exhaustive search small
        okw["do_exhaustive_model_search"] = 1; rkw["exhaustive"] = 1
    if max_order is not None:
        okw["max_lpc_order"] = max_order; rkw["max_lpc_order"] = max_order
    if precision is not None:
        okw["qlp_coeff_precision"] = precision; rkw["qlp_precision"] = precision
    if po is not None:
        okw["min_residual_partition_order"], okw["max_residual_partition_order"] = po
        rkw["min_part_order"], rkw["max_part_order"] = po
    if loose and ch == 2:
        okw["do_mid_side"] = 1; okw["loose_mid_side"] = 1
        rkw["mid_side"] = 1; rkw["loose_mid_side"] = 1
    try:
        enc = oraclelib.Encoder(oraclelib.preset(ch, bps, 44100, level, bs, **okw))
    except ValueError:
        return  # outside the oracle's declared scope
    got = enc.encode_stream(x)
    try:
        ref = refdata.encode(x, bps, rate=44100, level=level, blocksize=bs, variant="strict", opts=reflib.RefEncOpts(streamable_subset=0, **rkw))
    except RuntimeError:
        return  # the reference rejects this combination at init (e.g. precision too high for the sample width)
    bad = ref.mismatches(got)
    assert not bad, f"frames {bad} differ"


@seed(SEED_PRECISION_SEARCH)
@settings(max_examples=120, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
@given(ch=st.sampled_from([1, 2, 2, 3, 5, 8]), bps=st.sampled_from([8, 16, 20, 24]), level=st.integers(0, 8), bs=st.sampled_from([0, 576, 1000, 4096]),
       seed=st.integers(1, 50), prec_search=st.booleans(), min_bitrate=st.booleans(), silence=st.sampled_from(["none", "all", "first", "last", "dc"]))
def test_oracle_equals_reference_with_precision_search_and_limit_min_bitrate(ch, bps, level, bs, seed, prec_search, min_bitrate, silence):
    """flac -p (stream_encoder.c:4230-4243) and limit_min_bitrate (:3874-3879), on inputs whose second block is (partly) constant."""
    bsz = bs or (1152 if level < 3 else 4096)
    x = signals.music_like(bsz * 3 + 19, ch, bps, 44100, seed=seed)
    blk = slice(bsz, 2 * bsz)
    if silence == "all":
        x[blk] = 0
    elif silence == "dc":
        x[blk] = 5
    elif silence == "first":
        x[blk, 0] = -3
    elif silence == "last":
        x[blk, ch - 1] = 7
    okw, rkw = {}, {}
    if prec_search:
        okw["do_qlp_coeff_prec_search"] = 1; rkw["prec_search"] = 1
    if min_bitrate:
        okw["limit_min_bitrate"] = 1; rkw["limit_min_bitrate"] = 1
    enc = oraclelib.Encoder(oraclelib.preset(ch, bps, 44100, level, bs, **okw))
    got = enc.encode_stream(x)
    # disable_isa=16: the reference's C / SSE dispatch. Its AVX2 routine for the fixed-order guess drops the last (n - 4) % 4 samples of
    # a block (fixed_intrin_avx2.c:138 "Ignore the remainder"), which only shows on short last blocks -- see the test below.
    ref = refdata.encode(x, bps, rate=44100, level=level, blocksize=bs, variant="strict",
                         opts=reflib.RefEncOpts(streamable_subset=0, disable_isa=16, **rkw))
    bad = ref.mismatches(got)
    assert not bad, f"frames {bad} differ"


def test_reference_dispatch_paths_disagree_on_a_short_last_block():
    """The reference is not self-consistent across its own CPU dispatch: FLAC__fixed_compute_best_predictor_wide_intrin_avx2
    (fixed_intrin_avx2.c:57-138) reads lane j from offset (j * n) / 4 but seeds its difference history from j * (n / 4),
    and never sums the last n % 4 samples (n = blocksize - 4); the C routine (fixed.c:292-353) sums every sample. Regular
    blocksizes make n a multiple of 4, where both agree, so only a stream's short last block can see it; there the guessed
    fixed order may differ (20-/24-bit input: 32 of 360 random last blocks at -1 / -2 / -5; 16-bit input: 0 of 180).
    The oracle's default -- and the CUDA engine -- follow the C routine; fo_config.x86_avx2_fixed_guess restates the AVX2
    routine as written, which pins the explanation: with it the oracle equals the reference as dispatched on an AVX2 host."""
    x = signals.music_like(1152 * 3 + 19, 2, 24, 44100, seed=1)
    got = oraclelib.Encoder(oraclelib.preset(2, 24, 44100, 2)).encode_stream(x)
    c_path = refdata.encode(x, 24, rate=44100, level=2, variant="strict", opts=reflib.RefEncOpts(streamable_subset=0, disable_isa=16))
    assert c_path.mismatches(got) == []
    # the reference as dispatched on the host it was recorded on
    host_path = refdata.encode(x, 24, rate=44100, level=2, variant="strict", opts=reflib.RefEncOpts(streamable_subset=0))
    assert host_path.mismatches(got) in ([], [len(got) - 1])  # full blocks never differ
    if host_path.mismatches(got) == []:
        pytest.skip("the reference was recorded on a host that does not dispatch to the AVX2 routine")
    rng = np.random.default_rng(5)
    for bps, level in [(24, 2), (24, 1), (20, 2), (24, 5), (16, 2)]:
        for t in range(12):
            tail = int(rng.integers(17, 3000)) | 1  # (tail - 4) % 4 != 0
            bsz = 1152 if level < 3 else 4096
            y = signals.music_like(bsz + tail, 2, bps, 44100, seed=300 + t)
            q = oraclelib.Encoder(oraclelib.preset(2, bps, 44100, level, x86_avx2_fixed_guess=1)).encode_stream(y)
            ref = refdata.encode(y, bps, rate=44100, level=level, variant="strict", opts=reflib.RefEncOpts(streamable_subset=0))
            assert ref.mismatches(q) == [], (bps, level, tail)
