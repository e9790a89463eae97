"""Writes tests/golden/reference_reader.json from the UNMODIFIED reference's reader (common/seqiter.hpp, through
oracle/_ref/libmm_ref.so, built by oracle/Makefile): its (rc, records, bases, FNV-1a digest) of every file of
tests/test_input_cpu.py's reader comparison, plain and gzip'ed.
Run from the repository root after the build: python tests/golden/make_reference_reader.py"""
import ctypes as C
import gzip
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import refh  # noqa: E402
import test_input_cpu as t  # noqa: E402

R = refh.lib()
R.refh_read_file_digest.argtypes = [C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
wd = tempfile.mkdtemp()
out = {}
for name, data in t.reader_files().items():
    p = t.write(os.path.join(wd, name), data)
    gz = p + ".gz"
    with gzip.open(gz, "wb") as f:
        f.write(data)
    out[name] = [t._digest(R.refh_read_file_digest, p.encode()), t._digest(R.refh_read_file_digest, gz.encode())]
with open(t.READER_GOLDEN, "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
print("wrote", len(out), "files")
