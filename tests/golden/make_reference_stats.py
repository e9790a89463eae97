"""Writes tests/golden/reference_stats.json from the UNMODIFIED reference (oracle/_ref/libmm_ref.so, built by
oracle/Makefile): the statistics tables tests/test_host_cpu.py compares the product's with (minimum hits, the float
Jaccard / mash-distance functions as float32 bit patterns, the automatic sketch size, the sketch cut-offs).
Run from the repository root after the build: python tests/golden/make_reference_stats.py"""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import refh  # noqa: E402
import test_host_cpu as t  # noqa: E402

R = refh.lib()
out = {}
for pi in t.MIN_HITS_PI:
    out[f"min_hits {pi}"] = {str(k): [R.refh_min_hits(s, k, pi) for s in t.MIN_HITS_S] for k in (19, 16)}
f = {"j2md": [], "md2j": [], "lower_bound_d": [], "md_lower_bound": []}
for j in t.stat_inputs():
    for k in t.STAT_K:
        f["j2md"].append(t.f32_bits(R.refh_j2md(float(j), k)))
        f["md2j"].append(t.f32_bits(R.refh_md2j(float(j), k)))
for s, shared in t.lower_bound_inputs():
    d = R.refh_j2md(np.float32(shared / s), 19)
    f["lower_bound_d"].append(t.f32_bits(d))
    f["md_lower_bound"].append(t.f32_bits(R.refh_md_lower_bound(d, s, 19)))
out["float functions"] = f
out["recommended sketch size"] = [R.refh_recommended_sketch_size(19, pi, seg, size) for size, pi, seg in t.SKETCH_SIZE_CASES]
ref = t.write_cutoff_fasta(tempfile.mkdtemp())
for args in t.CUTOFF_ARGS:
    S = refh.RefSession(["-r", ref, "-q", ref] + args)
    p = {n: getattr(S.p, n) for n in ("sketchSize", "kmerSize", "ANIDiff", "ANIDiffConf", "stage1_topANI_filter")}
    out["cutoffs " + " ".join(args)] = {"params": p, "value": S.cutoffs().tolist()}
    S.close()
with open(t.GOLDEN, "w") as fh:
    json.dump(out, fh, separators=(",", ":"), sort_keys=True)
print("wrote", len(out), "tables")
