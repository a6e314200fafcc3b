"""The drop-in boundary, checked with the reference's OWN client code.

CPU: the unmodified examples/c/{decode,encode}/file/main.c link against libflac_b200.so (every libFLAC symbol they take from
the library is exported); the structs a client reads through the callbacks (FLAC__Frame, FLAC__StreamMetadata, ...) have the
reference's layout. Both compare with what the reference's sources give, stored in tests/golden/dropin.json by
tests/golden/make_dropin_golden.py.
GPU: the prebuilt example binaries (oracle/_ref/examples, built by `make -C oracle examples` where the reference's sources
are) run against libflac_b200.so and produce what the same binaries produce with the compiled reference."""
import json
import os
import shutil
import subprocess
import sys
import wave

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
EXDIR = os.path.join(ROOT, "oracle", "_ref", "examples")
GOLDEN = os.path.join(ROOT, "tests", "golden", "dropin.json")
# the reference's units the encode client is linked with besides the library (oracle/Makefile, target `examples`)
METADATA_UNITS = ("metadata_object", "format", "memory", "bitwriter", "stream_encoder_framing", "crc", "bitmath")

LAYOUT_PROBE = r"""
#include <stddef.h>
#include <stdio.h>
%s
#define P(T) printf(#T " %%zu\n", sizeof(T))
#define O(T, f) printf(#T "." #f " %%zu\n", offsetof(T, f))
int main(void) {
	P(FLAC__Frame); P(FLAC__FrameHeader); P(FLAC__Subframe); P(FLAC__Subframe_LPC); P(FLAC__Subframe_Fixed); P(FLAC__FrameFooter);
	P(FLAC__EntropyCodingMethod); P(FLAC__EntropyCodingMethod_PartitionedRice); P(FLAC__EntropyCodingMethod_PartitionedRiceContents);
	P(FLAC__StreamMetadata); P(FLAC__StreamMetadata_StreamInfo); P(FLAC__StreamMetadata_SeekPoint); P(FLAC__StreamMetadata_VorbisComment);
	O(FLAC__Frame, header); O(FLAC__Frame, subframes); O(FLAC__Frame, footer);
	O(FLAC__FrameHeader, blocksize); O(FLAC__FrameHeader, sample_rate); O(FLAC__FrameHeader, channels); O(FLAC__FrameHeader, channel_assignment);
	O(FLAC__FrameHeader, bits_per_sample); O(FLAC__FrameHeader, number_type); O(FLAC__FrameHeader, number); O(FLAC__FrameHeader, crc);
	O(FLAC__Subframe, type); O(FLAC__Subframe, data); O(FLAC__Subframe, wasted_bits);
	O(FLAC__Subframe_LPC, entropy_coding_method); O(FLAC__Subframe_LPC, order); O(FLAC__Subframe_LPC, qlp_coeff_precision); O(FLAC__Subframe_LPC, quantization_level);
	O(FLAC__Subframe_LPC, qlp_coeff); O(FLAC__Subframe_LPC, warmup); O(FLAC__Subframe_LPC, residual);
	O(FLAC__Subframe_Fixed, entropy_coding_method); O(FLAC__Subframe_Fixed, order); O(FLAC__Subframe_Fixed, warmup); O(FLAC__Subframe_Fixed, residual);
	O(FLAC__StreamMetadata, type); O(FLAC__StreamMetadata, is_last); O(FLAC__StreamMetadata, length); O(FLAC__StreamMetadata, data);
	O(FLAC__StreamMetadata_StreamInfo, total_samples); O(FLAC__StreamMetadata_StreamInfo, md5sum);
	return 0;
}
"""


def _golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


def test_reference_examples_link_against_libflac_b200():
    import flac_b200
    from flac_b200 import build
    build.build()
    lib = flac_b200.lib()
    for client, names in _golden()["clients"].items():
        missing = [n for n in names if not hasattr(lib, n)]
        assert not missing, f"the reference's {client} example client would not link: {missing} not exported"


@pytest.mark.skipif(shutil.which("gcc") is None, reason="gcc not present")
def test_struct_layouts_match_reference_headers(tmp_path):
    src = tmp_path / "layout_ours.c"
    src.write_text(LAYOUT_PROBE % '#include <stdio.h>\n#include "flac_b200_stream.h"')
    exe = tmp_path / "layout_ours"
    r = subprocess.run(["gcc", str(src), "-o", str(exe), f"-I{ROOT}/include"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ours, ref = subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines(), _golden()["layout"]
    assert ours == ref, "struct layout differs from the reference headers:\n" + "\n".join(
        f"{a}   |   {b}" for a, b in zip(ref, ours) if a != b)


def _write_wav(path, x):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(x.shape[1]); w.setsampwidth(2); w.setframerate(44100)
        w.writeframes(x.astype("<i2").tobytes())


def _audio_offset(flac_bytes):
    assert flac_bytes[:4] == b"fLaC"
    pos = 4
    while True:
        last = flac_bytes[pos] & 0x80
        n = int.from_bytes(flac_bytes[pos + 1:pos + 4], "big")
        pos += 4 + n
        if last:
            return pos


@pytest.mark.gpu
def test_reference_example_clients_run_on_libflac_b200(tmp_path):
    """encode: frames byte-identical to the reference-linked binary's; decode: WAV byte-identical."""
    need = [os.path.join(EXDIR, n) for n in ("encode_b200", "decode_b200", "encode_ref", "decode_ref")]
    if not all(os.path.exists(p) for p in need):
        pytest.skip("oracle/_ref/examples not built (make -C oracle examples)")
    sys.path.insert(0, os.path.dirname(__file__))
    import signals
    x = signals.music_like(4096 * 9 + 321, 2, 16, 44100, seed=12)
    wav = tmp_path / "in.wav"
    _write_wav(wav, x)
    outs = {}
    for tag in ("b200", "ref"):
        r = subprocess.run([os.path.join(EXDIR, f"encode_{tag}"), str(wav), str(tmp_path / f"{tag}.flac")], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (tag, r.stdout[-500:], r.stderr[-500:])
        outs[tag] = (tmp_path / f"{tag}.flac").read_bytes()
    a, b = outs["b200"], outs["ref"]
    assert a[_audio_offset(a):] == b[_audio_offset(b):], "audio frames differ between libflac_b200 and the reference under the same client"
    # STREAMINFO (34 bytes after the 4-byte block header at offset 4): everything incl. min/max frame size, total samples and MD5
    assert a[8:8 + 34] == b[8:8 + 34]
    for tag in ("b200", "ref"):
        r = subprocess.run([os.path.join(EXDIR, f"decode_{tag}"), str(tmp_path / "ref.flac"), str(tmp_path / f"{tag}.wav")], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (tag, r.stdout[-500:], r.stderr[-500:])
    assert (tmp_path / "b200.wav").read_bytes() == (tmp_path / "ref.wav").read_bytes()
