"""The reference's object API on top of the engine (include/flac_b200_stream.h), driven the way
src/test_libFLAC/encoders.c / decoders.c drive libFLAC: setters, init_stream with client
callbacks, process, finish -- and compared with the compiled reference byte for byte
(frames, STREAMINFO incl. MD5) / sample for sample."""
import ctypes as C
import os

import numpy as np
import pytest

import oraclelib
import refdata
import signals

pytestmark = pytest.mark.gpu

WRITE = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_ubyte), C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p)
SEEK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_void_p)
TELL = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p)
DREAD = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_ubyte), C.POINTER(C.c_size_t), C.c_void_p)
DWRITE = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.POINTER(C.c_int32)), C.c_void_p)
DMETA = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_void_p)
DERR = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_void_p)


def L():
    import flac_b200
    lib = flac_b200.lib()
    lib.FLAC__stream_encoder_new.restype = C.c_void_p
    lib.FLAC__stream_decoder_new.restype = C.c_void_p
    lib.FLAC__stream_encoder_init_stream.argtypes = [C.c_void_p, WRITE, SEEK, TELL, C.c_void_p, C.c_void_p]
    lib.FLAC__stream_encoder_process_interleaved.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    lib.FLAC__stream_encoder_process.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
    lib.FLAC__stream_decoder_init_stream.argtypes = [C.c_void_p, DREAD, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, DWRITE, DMETA, DERR, C.c_void_p]
    lib.FLAC__stream_decoder_seek_absolute.argtypes = [C.c_void_p, C.c_uint64]
    lib.FLAC__stream_decoder_get_total_samples.restype = C.c_uint64
    for n in ("encoder_delete", "encoder_finish", "encoder_get_state", "decoder_delete", "decoder_finish", "decoder_get_state",
              "decoder_process_until_end_of_stream", "decoder_process_until_end_of_metadata", "decoder_process_single",
              "decoder_get_total_samples", "decoder_get_channels", "decoder_get_bits_per_sample", "decoder_get_sample_rate"):
        getattr(lib, "FLAC__stream_" + n).argtypes = [C.c_void_p]
    return lib


class Sink:
    """In-memory seekable output, like a FILE."""

    def __init__(self):
        self.buf = bytearray()
        self.pos = 0
        self.frames = []

    def write(self, enc, p, n, samples, frame, client):
        data = bytes(p[:n]) if n else b""
        end = self.pos + n
        if end > len(self.buf):
            self.buf.extend(b"\0" * (end - len(self.buf)))
        self.buf[self.pos:end] = data
        self.pos = end
        if samples:
            self.frames.append(data)
        return 0

    def seek(self, enc, off, client):
        self.pos = off
        return 0

    def tell(self, enc, out, client):
        out[0] = self.pos
        return 0


def encode_with_api(x, bps, rate, level, chunk=2048, verify=False, planar=False, batch=None, md5=True, apodization=None):
    lib = L()
    if batch:
        os.environ["FB200_BATCH_BLOCKS"] = str(batch)
    e = C.c_void_p(lib.FLAC__stream_encoder_new())
    lib.FLAC__stream_encoder_set_channels(e, C.c_uint32(x.shape[1]))
    lib.FLAC__stream_encoder_set_bits_per_sample(e, C.c_uint32(bps))
    lib.FLAC__stream_encoder_set_sample_rate(e, C.c_uint32(rate))
    lib.FLAC__stream_encoder_set_compression_level(e, C.c_uint32(level))
    if apodization is not None:  # after the level, like the flac CLI's -A
        lib.FLAC__stream_encoder_set_apodization.argtypes = [C.c_void_p, C.c_char_p]
        assert lib.FLAC__stream_encoder_set_apodization(e, apodization.encode())
    lib.FLAC__stream_encoder_set_verify(e, C.c_int(1 if verify else 0))
    lib.FLAC__stream_encoder_set_do_md5(e, C.c_int(1 if md5 else 0))
    sink = Sink()
    cbs = (WRITE(sink.write), SEEK(sink.seek), TELL(sink.tell))
    st = lib.FLAC__stream_encoder_init_stream(e, cbs[0], cbs[1], cbs[2], None, None)
    assert st == 0, f"init status {st}"
    n = x.shape[0]
    for i in range(0, n, chunk):
        part = np.ascontiguousarray(x[i:i + chunk])
        if planar:
            chans = [np.ascontiguousarray(part[:, c]) for c in range(part.shape[1])]
            arr = (C.c_void_p * len(chans))(*[c.ctypes.data for c in chans])
            assert lib.FLAC__stream_encoder_process(e, arr, part.shape[0])
        else:
            assert lib.FLAC__stream_encoder_process_interleaved(e, part.ctypes.data, part.shape[0])
    assert lib.FLAC__stream_encoder_finish(e), lib.FLAC__stream_encoder_get_state(e)
    assert lib.FLAC__stream_encoder_get_state(e) == 1  # back to UNINITIALIZED
    lib.FLAC__stream_encoder_delete(e)
    os.environ.pop("FB200_BATCH_BLOCKS", None)
    return bytes(sink.buf), sink.frames


@pytest.mark.parametrize("level,ch,bps,rate", [(5, 2, 16, 44100), (8, 2, 16, 44100), (8, 2, 24, 96000), (2, 1, 16, 44100), (5, 8, 24, 192000)])
def test_encoder_api_matches_reference_stream(level, ch, bps, rate):
    x = signals.music_like(4096 * 7 + 1234, ch, bps, rate, seed=3)
    stream, frames = encode_with_api(x, bps, rate, level, batch=3)
    ref = refdata.encode(x, bps, rate=rate, level=level, md5=True)
    assert ref.mismatches(frames) == []
    # STREAMINFO body as update_metadata_ (stream_encoder.c:3139-3300) leaves it: blocksizes, min/max frame
    # size, rate/channels/bps, total samples and the MD5 of the little-endian interleaved input
    import hashlib
    bs = 1152 if level < 3 else 4096
    nbytes = (bps + 7) // 8
    raw = x.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :nbytes].tobytes()
    sizes = ref.sizes
    packed = (rate << 44) | ((ch - 1) << 41) | ((bps - 1) << 36) | x.shape[0]
    want = (bs.to_bytes(2, "big") * 2 + min(sizes).to_bytes(3, "big") + max(sizes).to_bytes(3, "big") + packed.to_bytes(8, "big")
            + hashlib.md5(raw).digest())
    assert stream[:4] == b"fLaC" and stream[4] == 0x00 and stream[5:8] == (34).to_bytes(3, "big")
    assert stream[8:42] == want
    # and the reference decoder accepts the whole file, MD5 checked
    y = refdata.decode(stream, x.shape[0], ch, md5=True)
    assert y.info[3] == 0 and y.matches(x)


def test_encoder_api_planar_process_and_verify():
    x = signals.music_like(4096 * 3 + 10, 2, 16, 44100, seed=4)
    s1, f1 = encode_with_api(x, 16, 44100, 5, planar=True, verify=True)
    s2, f2 = encode_with_api(x, 16, 44100, 5, chunk=777)
    assert f1 == f2 and s1 == s2


def test_encoder_api_rejects_out_of_range_samples():
    lib = L()
    e = C.c_void_p(lib.FLAC__stream_encoder_new())
    sink = Sink()
    cbs = (WRITE(sink.write), SEEK(sink.seek), TELL(sink.tell))
    assert lib.FLAC__stream_encoder_init_stream(e, cbs[0], cbs[1], cbs[2], None, None) == 0
    bad = np.array([[0, 40000]], dtype=np.int32)   # does not fit 16 bits -> CLIENT_ERROR (stream_encoder.c:2543-2548)
    assert not lib.FLAC__stream_encoder_process_interleaved(e, bad.ctypes.data, 1)
    assert lib.FLAC__stream_encoder_get_state(e) == 5
    lib.FLAC__stream_encoder_finish(e)
    lib.FLAC__stream_encoder_delete(e)


def test_encoder_api_file_variant(tmp_path):
    lib = L()
    x = signals.music_like(4096 * 2 + 5, 2, 16, 44100, seed=5)
    path = str(tmp_path / "out.flac").encode()
    e = C.c_void_p(lib.FLAC__stream_encoder_new())
    lib.FLAC__stream_encoder_set_compression_level(e, C.c_uint32(8))
    lib.FLAC__stream_encoder_init_file.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]
    assert lib.FLAC__stream_encoder_init_file(e, path, None, None) == 0
    assert lib.FLAC__stream_encoder_process_interleaved(e, x.ctypes.data, x.shape[0])
    assert lib.FLAC__stream_encoder_finish(e)
    lib.FLAC__stream_encoder_delete(e)
    data = open(path, "rb").read()
    y = refdata.decode(data, x.shape[0], 2, md5=True)
    assert y.info[3] == 0 and y.matches(x)


class DecClient:
    def __init__(self, data):
        self.data = data
        self.pos = 0
        self.blocks = []
        self.meta = []
        self.errors = []
        self.ch = 0

    def read(self, dec, buf, nbytes, client):
        n = min(nbytes[0], len(self.data) - self.pos)
        if n == 0:
            nbytes[0] = 0
            return 1  # END_OF_STREAM
        C.memmove(buf, self.data[self.pos:self.pos + n], n)
        self.pos += n
        nbytes[0] = n
        return 0

    def write(self, dec, frame, buffers, client):
        hdr = C.cast(frame, C.POINTER(C.c_uint32))
        bs, ch = hdr[0], hdr[2]
        self.ch = ch
        blk = np.stack([np.ctypeslib.as_array(buffers[c], shape=(bs,)).copy() for c in range(ch)], axis=1)
        self.blocks.append(blk)
        return 0

    def metadata(self, dec, m, client):
        self.meta.append(C.cast(m, C.POINTER(C.c_uint32))[0])

    def error(self, dec, status, client):
        self.errors.append(status)


def decode_with_api(stream, md5=True, seek_to=None):
    lib = L()
    d = C.c_void_p(lib.FLAC__stream_decoder_new())
    lib.FLAC__stream_decoder_set_md5_checking(d, C.c_int(1 if md5 else 0))
    cl = DecClient(stream)
    cbs = (DREAD(cl.read), DWRITE(cl.write), DMETA(cl.metadata), DERR(cl.error))
    assert lib.FLAC__stream_decoder_init_stream(d, cbs[0], None, None, None, None, cbs[1], cbs[2], cbs[3], None) == 0
    assert lib.FLAC__stream_decoder_process_until_end_of_metadata(d)
    total = lib.FLAC__stream_decoder_get_total_samples(d)
    if seek_to is not None:
        assert lib.FLAC__stream_decoder_seek_absolute(d, seek_to)
    assert lib.FLAC__stream_decoder_process_until_end_of_stream(d)
    assert lib.FLAC__stream_decoder_get_state(d) == 4  # END_OF_STREAM
    ok = lib.FLAC__stream_decoder_finish(d)
    lib.FLAC__stream_decoder_delete(d)
    return np.concatenate(cl.blocks, axis=0), cl, total, ok


@pytest.mark.parametrize("level,ch,bps,rate", [(5, 2, 16, 44100), (8, 2, 24, 96000), (0, 1, 16, 22050), (8, 8, 24, 192000)])
def test_decoder_api_on_reference_streams(level, ch, bps, rate):
    x = signals.music_like(4096 * 5 + 99, ch, bps, rate, seed=6)
    # (a) the reference's stream as captured without a seek callback: STREAMINFO unpatched (total 0, MD5 0); its frames are the
    # oracle's, checked to be exactly the reference's (tests/refdata.py)
    ref = refdata.encode(x, bps, rate=rate, level=level, md5=True, header=True)
    ref_stream = ref.header + b"".join(ref.frames(witness=oraclelib.Encoder(oraclelib.preset(ch, bps, rate, level)).encode_stream(x)))
    y, cl, total, ok = decode_with_api(ref_stream)
    assert total == 0 and ok and cl.errors == [] and cl.meta == [0]
    assert np.array_equal(x, y)
    # (b) a complete file (frames identical to the reference's, STREAMINFO patched at finish): total + MD5 checked
    stream, _ = encode_with_api(x, bps, rate, level)
    y, cl, total, ok = decode_with_api(stream)
    assert total == x.shape[0] and ok and cl.errors == [] and cl.meta == [0]
    assert np.array_equal(x, y)


def test_decoder_api_seek_and_md5_failure():
    x = signals.music_like(4096 * 6, 2, 16, 44100, seed=7)
    stream, _ = encode_with_api(x, 16, 44100, 5)
    y, cl, total, ok = decode_with_api(stream, seek_to=10000)
    assert np.array_equal(y, x[10000:])
    # corrupt the STREAMINFO MD5: finish() must report the mismatch (stream_decoder.c:3620-3632)
    bad = bytearray(stream)
    bad[30] ^= 0xff
    y, cl, total, ok = decode_with_api(bytes(bad))
    assert np.array_equal(x, y) and not ok
