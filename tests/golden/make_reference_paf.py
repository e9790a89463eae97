"""Writes tests/golden/reference_paf.json from the UNMODIFIED
reference CLI, oracle/_ref/mashmap_ref (built by oracle/Makefile): the PAF it prints for every run tests/test_gpu_cli.py
compares the product with. Run from the repository root after the build: python tests/golden/make_reference_paf.py"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import datasets  # noqa: E402
import refh  # noqa: E402
import test_gpu_cli as t  # noqa: E402


def reference(args, out):
    subprocess.run([refh.REF_BIN] + args + ["-o", out], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    with open(out) as f:
        return f.read()


wd = tempfile.mkdtemp()
out = os.path.join(wd, "out.paf")
paf = {}
for which, args in t.CONFIGS:
    d = t.MAKERS[which][1](wd, tag=t.MAKERS[which][0])
    paf[t.config_key(which, args)] = reference(["-r", d["ref"], "-q", d["qry"], "-t", "8"] + args, out)
d = datasets.make_panel_set(wd, tag="clip")
paf["multiple query files"] = reference(["-r", d["ref"], "--ql", t.write_split_queries(wd, d)] + t.MULTI_QUERY_ARGS, out)
with open(t.GOLDEN, "w") as f:
    json.dump(paf, f, indent=0, sort_keys=True)
print("wrote", len(paf), "runs")
