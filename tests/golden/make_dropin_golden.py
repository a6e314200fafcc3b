"""Generates tests/golden/dropin.json from the reference's sources and the objects `make -C oracle ref` built from them:

    make -C oracle ref REF=<reference source tree>
    python tests/golden/make_dropin_golden.py <reference source tree>

  clients  the libFLAC symbols each of the reference's example programs (examples/c/{decode,encode}/file/main.c)
           takes from the library it is linked against. The encode client is linked together with the reference's
           metadata-object units (oracle/Makefile, target `examples`), so what those define is not asked of the library.
  layout   what tests/test_dropin_examples.py's LAYOUT_PROBE prints (sizeof / offsetof of the structs a client reads
           through the callbacks) when compiled against the reference's headers.
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))

from test_dropin_examples import LAYOUT_PROBE, METADATA_UNITS, ROOT  # noqa: E402


def _nm(args):
    return subprocess.run(["nm"] + args, capture_output=True, text=True, check=True).stdout.splitlines()


def main(ref):
    cflags = ["-O1", "-include", "inttypes.h", f"-I{ref}/include"]
    meta = [os.path.join(ROOT, "oracle", "_ref", "obj_default", u + ".o") for u in METADATA_UNITS]
    provided = {ln.split()[2] for ln in _nm(["--defined-only"] + meta) if len(ln.split()) == 3}
    out = {"clients": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for client, extra in (("decode", []), ("encode", meta)):
            obj = os.path.join(tmp, client + ".o")
            subprocess.run(["gcc", "-c"] + cflags + [f"{ref}/examples/c/{client}/file/main.c", "-o", obj], check=True)
            needed = {ln.split()[-1] for ln in _nm(["-u", obj] + extra) if ln.split() and ln.split()[-1].startswith("FLAC__")}
            out["clients"][client] = sorted(needed - provided)
        src, exe = os.path.join(tmp, "layout.c"), os.path.join(tmp, "layout")
        with open(src, "w") as fh:
            fh.write(LAYOUT_PROBE % '#include "FLAC/all.h"')
        subprocess.run(["gcc", src, "-o", exe, f"-I{ref}/include"], check=True)
        out["layout"] = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines()
    with open(os.path.join(HERE, "dropin.json"), "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
