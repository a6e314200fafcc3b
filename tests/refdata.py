"""What the compiled reference libFLAC answered for the exact inputs the tests give it, stored in
tests/golden/reference.json.gz, so that every comparison with the reference runs where the reference is absent.

Each answer is keyed by a digest of the call (input samples or bytes and every parameter). An encode answer
holds every frame's size and the first 64 bits of its SHA-256 (the stream header too where a test needs its
bytes); a decode answer holds the decoded samples' digest and the decoder's report; a window answer holds the
table's digest. A call whose key is not stored fails the test: the reference never saw that input.

To regenerate, build the reference (`make -C oracle ref`) and run the suite with
FLAC_REF_RECORD=<path>: every call then goes to the reference through reflib, and the stored answers together
with the new ones are written to <path> when the run ends (delete tests/golden/reference.json.gz first to drop
answers no test asks for). The GPU tests hand the reference streams the engine produced, so their answers are
recorded on a machine with a GPU.
"""
import atexit
import ctypes as C
import gzip
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference.json.gz")
RECORD = os.environ.get("FLAC_REF_RECORD")

_store = None


def _answers():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(GOLDEN):
            with gzip.open(GOLDEN, "rt") as fh:
                _store = json.load(fh)
        if RECORD:
            atexit.register(_write)
    return _store


def _write():
    """One answer per line, sorted, gzip'ed without a timestamp: the same answers give the same file."""
    text = "{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(_store[k], separators=(',', ':'))}" for k in sorted(_store)) + "\n}\n"
    with open(RECORD, "wb") as fh, gzip.GzipFile(fileobj=fh, mode="wb", mtime=0) as gz:
        gz.write(text.encode())


def digest(data):
    """First 64 bits of the SHA-256 of bytes, or of an array's dtype, shape and contents, as hex."""
    if isinstance(data, np.ndarray):
        data = np.ascontiguousarray(data)
        data = f"{data.dtype.str}{data.shape}".encode() + data.tobytes()
    return hashlib.sha256(bytes(data)).hexdigest()[:16]


def _key(kind, *parts):
    h = hashlib.sha256(kind.encode())
    for p in parts:
        h.update(b"|" + (digest(p) if isinstance(p, (bytes, np.ndarray)) else repr(p)).encode())
    return f"{kind}:{h.hexdigest()[:16]}"


def _answer(key, ask):
    store = _answers()
    if RECORD:
        rec = ask()
        assert store.get(key, rec) == rec, f"{key}: the reference now answers {rec}, stored: {store[key]}"
        store[key] = rec
    assert key in store, f"no stored reference answer for this call ({key} in {GOLDEN}); record it with FLAC_REF_RECORD"
    return store[key]


def _opts_tuple(opts):
    return None if opts is None else tuple(getattr(opts, f) for f, _ in opts._fields_)


class Encoding:
    """The reference encoder's frames for one input: sizes, digests and (when asked for) the stream header."""

    def __init__(self, rec):
        self.sizes = rec["sizes"]
        self.digests = [rec["sha"][i:i + 16] for i in range(0, len(rec["sha"]), 16)]
        self.header = bytes.fromhex(rec["header"]) if "header" in rec else None

    def __len__(self):
        return len(self.sizes)

    def mismatches(self, frames):
        """Indices of the frames that differ from the reference's (frames must be as many)."""
        assert len(frames) == len(self), f"frame count {len(frames)} != the reference's {len(self)}"
        return [i for i, f in enumerate(frames) if len(f) != self.sizes[i] or digest(f) != self.digests[i]]

    def frames(self, witness):
        """The reference's frame bytes, taken from `witness` (another encoder's frames) after checking that
        they are exactly the reference's."""
        bad = self.mismatches(witness)
        assert not bad, f"frames {bad[:5]} of the witness differ from the reference's, so they cannot stand for them"
        return list(witness)


def encode(pcm, bps, rate=44100, level=5, blocksize=0, md5=False, variant="default", opts=None, header=False):
    """The reference encoder's answer for int32 pcm [samples, channels] (reflib.encode's arguments).
    Raises RuntimeError where the reference rejected the configuration."""
    pcm = np.ascontiguousarray(pcm, dtype=np.int32)

    def ask():
        import reflib
        try:
            stream, hdr, frames = reflib.encode(pcm, bps, rate=rate, level=level, blocksize=blocksize, md5=md5, variant=variant, opts=opts)
        except RuntimeError as ex:
            return {"error": str(ex)}
        rec = {"sizes": [len(f) for f in frames], "sha": "".join(digest(f) for f in frames)}
        if header:
            rec["header"] = stream[:hdr].hex()
        return rec

    rec = _answer(_key("encode", pcm, bps, rate, level, blocksize, md5, variant, _opts_tuple(opts), header), ask)
    if "error" in rec:
        raise RuntimeError(rec["error"])
    return Encoding(rec)


class Decoding:
    """The reference decoder's answer: samples decoded, their digest, and (channels, bps, rate, errors)."""

    def __init__(self, rec):
        self.samples, self.pcm, self.info = rec["samples"], rec["pcm"], tuple(rec["info"])

    def matches(self, x):
        """The decoded samples equal int32 x [samples, channels]."""
        return self.samples == x.shape[0] and self.pcm == digest(np.ascontiguousarray(x, dtype=np.int32))


def decode(stream, max_samples, channels, variant="default", md5=False):
    stream = bytes(stream)

    def ask():
        import reflib
        y, info = reflib.decode(stream, max_samples, channels, variant=variant, md5=md5)
        return {"samples": int(y.shape[0]), "pcm": digest(np.ascontiguousarray(y, dtype=np.int32)), "info": [int(v) for v in info]}

    return Decoding(_answer(_key("decode", stream, max_samples, channels, variant, md5), ask))


def _live_window(variant, sym, n, *params):
    """The reference's window function `sym` (FLAC__window_*), called directly: float32 [n]."""
    import reflib
    f = getattr(reflib.lib(variant), sym)
    f.restype = None
    f.argtypes = [C.c_void_p, C.c_int32] + [C.c_float] * len(params)
    out = np.full(n + 8, np.float32(-77.0))
    f(out.ctypes.data, n, *params)
    assert np.all(out[n:] == np.float32(-77.0))
    return out[:n]


def window(variant, sym, n, *params):
    """Digest of the reference's window table, and for the shipped-flags build ("default") the largest absolute
    difference of its table from the source-order build's ("strict")."""
    params = tuple(float(np.float32(p)) for p in params)

    def ask():
        got = _live_window(variant, sym, n, *params)
        rec = {"sha": digest(got)}
        if variant == "default":
            rec["max_abs_diff_vs_strict"] = float(np.abs(got - _live_window("strict", sym, n, *params)).max())
        return rec

    return _answer(_key("window", variant, sym, n, params), ask)
