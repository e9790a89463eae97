"""Writes tests/golden/reference_params.json from the UNMODIFIED reference (oracle/_ref/libmm_ref.so, built by
oracle/Makefile): the skch::Parameters its parseandSave fills for every command line tests/test_args_cpu.py gives the
product's parser. Run from the repository root after the build: python tests/golden/make_reference_params.py"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import datasets  # noqa: E402
import refh  # noqa: E402
import test_args_cpu as t  # noqa: E402


def fields(p):
    return {name: getattr(p, name) for name, _ in refh.OrcParams._fields_}


wd = tempfile.mkdtemp()
d = datasets.make_panel_set(wd, tag="args", n_strains=2, chrom_len=40_000)
params = {}
for with_query in (True, False):
    for opts in t.OPTION_SETS:
        R = refh.RefSession(t.cli_args(d, opts, with_query))
        params[t.params_key(opts, with_query)] = fields(R.p)
        R.close()
for size in t.SIZES:
    f = os.path.join(wd, f"big_{size}.fa")
    t.write_sparse_fasta(f, size)
    params[f"size {size}"] = fields(refh.parse_only(t.size_args(f)))
    os.remove(f)
with open(t.GOLDEN, "w") as f:
    json.dump(params, f, indent=0, sort_keys=True)
print("wrote", len(params), "command lines")
