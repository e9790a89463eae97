"""CPU tests of the host-side product code (no GPU): statistics tables, the host index builder and the
host tail, each against the UNMODIFIED reference through oracle/_ref (when built). The statistics tables of the
reference are stored in tests/golden/reference_stats.json (written by tests/golden/make_reference_stats.py), so those
comparisons need no reference build."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import datasets
import refh
from mashmap_b200 import capi, hostlib, synth

needs_ref = pytest.mark.skipif(not refh.available(), reason="oracle/_ref not built")

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_stats.json")
MIN_HITS_PI = [0.85, 0.90, 0.95, 0.80]
MIN_HITS_S = list(range(1, 420)) + [500, 777, 1000]
STAT_K = (15, 19, 21)
LOWER_BOUND_S = (20, 130, 220, 400)
SKETCH_SIZE_CASES = [(size, pi, seg) for size in (1_200_000, 25_711_390, 100_000_000, 3_050_000_000)
                     for pi, seg in ((0.85, 5000), (0.95, 5000), (0.90, 10000), (0.85, 1000))]
CUTOFF_ARGS = [["-s", "5000", "--pi", "85"], ["-s", "5000", "--pi", "95", "--dense"], ["-s", "2000", "--pi", "90", "-J", "25"],
               ["-s", "5000", "--pi", "85", "--hgFilterAniDiff", "2", "--hgFilterConf", "99"]]


def reference_stats(key):
    """the reference's values for one table of this module (see tests/golden/make_reference_stats.py)"""
    with open(GOLDEN) as f:
        return json.load(f)[key]


def stat_inputs():
    """the Jaccard values the float functions are compared on"""
    rng = np.random.default_rng(3)
    return np.concatenate([rng.random(200).astype(np.float32), np.float32([0, 1, 0.5, 1e-6])])


def lower_bound_inputs():
    """(s, shared) pairs of the mash-distance lower bound"""
    return [(s, shared) for s in LOWER_BOUND_S for shared in range(0, s + 1, max(1, s // 37))]


def f32_bits(x):
    return int(np.float32(x).view(np.uint32))


def write_cutoff_fasta(workdir):
    ref = os.path.join(workdir, "cut_ref.fa")
    synth.write_fasta(ref, ["c0"], synth.random_genome(1, 60_000, seed=8))
    return ref


def test_c_abi_library_loads_and_exports_every_symbol():
    L = capi.lib()
    for sym in capi.EXPORTED_SYMBOLS:
        assert hasattr(L, sym), sym
    # every function declared in include/mashmap_b200.h must be exported
    import os
    import re

    hdr = open(os.path.join(os.path.dirname(capi._HERE), "include", "mashmap_b200.h")).read()
    declared = set(re.findall(r"\b(mm_[a-z_0-9]+)\s*\(", hdr))
    for sym in declared:
        assert hasattr(L, sym), f"{sym} declared in the header but not exported"
    assert declared == set(capi.EXPORTED_SYMBOLS)


def test_nccl_library_loads_and_exports_every_symbol():
    """include/mashmap_b200_nccl.h (multi-GPU entry points) vs libmashmap_nccl.so: loads without a GPU, exports every
    declared function"""
    import os
    import re

    from mashmap_b200 import nccl

    L = nccl.lib()
    hdr = open(os.path.join(os.path.dirname(capi._HERE), "include", "mashmap_b200_nccl.h")).read()
    declared = set(re.findall(r"\b(mm_[a-z_0-9]+)\s*\(", hdr))
    for sym in declared:
        assert hasattr(L, sym), f"{sym} declared in the header but not exported"
    assert declared == set(nccl.EXPORTED_SYMBOLS)


def test_no_cpu_fallback_without_device():
    from conftest import have_gpu

    if have_gpu():
        pytest.skip("GPU present")
    with pytest.raises(capi.MashmapError) as e:
        capi.Context()
    assert e.value.code == capi.MM_ENODEVICE


@pytest.mark.parametrize("pi", MIN_HITS_PI)
def test_min_hits_table_matches_reference(pi):
    ref = reference_stats(f"min_hits {pi}")
    L = hostlib.lib()
    for k in (19, 16):
        for s, want in zip(MIN_HITS_S, ref[str(k)], strict=True):
            assert L.skch_min_hits(s, k, pi) == want, (s, k, pi)


def test_float_stat_functions_bit_equal():
    ref = reference_stats("float functions")
    L = hostlib.lib()
    assert len(ref["j2md"]) == len(ref["md2j"]) == len(stat_inputs()) * len(STAT_K)
    i = 0
    for j in stat_inputs():
        for k in STAT_K:
            assert f32_bits(L.skch_j2md(float(j), k)) == ref["j2md"][i]
            assert f32_bits(L.skch_md2j(float(j), k)) == ref["md2j"][i]
            i += 1
    for (s, shared), d, want in zip(lower_bound_inputs(), ref["lower_bound_d"], ref["md_lower_bound"], strict=True):
        d = float(np.uint32(d).view(np.float32))
        assert f32_bits(L.skch_md_lower_bound(d, s, 19)) == want, (s, shared)


def test_recommended_sketch_size_matches_reference():
    ref = reference_stats("recommended sketch size")
    L = hostlib.lib()
    for (size, pi, seg), want in zip(SKETCH_SIZE_CASES, ref, strict=True):
        assert L.skch_recommended_sketch_size(19, pi, seg, size) == want, (size, pi, seg)


def test_binomial_tail_against_exact_summation():
    """the product's mode-anchored recurrence vs the oracle shim's independent log-gamma form"""
    import math

    L = hostlib.lib()
    for n, p in ((130, 0.0121), (220, 0.2), (1000, 0.03), (20, 0.5)):
        for k in range(0, min(n, 60)):
            exact = sum(math.exp(math.lgamma(n + 1) - math.lgamma(i + 1) - math.lgamma(n - i + 1) + i * math.log(p)
                                 + (n - i) * math.log1p(-p)) for i in range(k + 1, n + 1))
            got = L.skch_binomial_Q(k, p, n)
            assert abs(got - exact) <= 1e-12 + 1e-9 * exact, (n, p, k, got, exact)


@pytest.mark.parametrize("args", CUTOFF_ARGS)
def test_sketch_cutoffs_match_reference(args):
    """the cut-off table for the reference's own Parameters of a 60 kb reference file"""
    ref = reference_stats("cutoffs " + " ".join(args))
    p = ref["params"]
    got = hostlib.sketch_cutoffs(p["sketchSize"], p["kmerSize"], p["ANIDiff"], p["ANIDiffConf"], bool(p["stage1_topANI_filter"]))
    assert np.array_equal(got, ref["value"])


def _cases_for_index():
    rng = np.random.default_rng(17)
    g = synth.random_sequence(60_000, rng)
    rep = np.tile(synth.random_sequence(700, rng), 40)
    withn = g[:30_000].copy()
    withn[5000:5600] = ord("N"); withn[12_000] = ord("N"); withn[29_990:] = ord("N")
    low = np.frombuffer(b"ACACACACACGTGTGTGTGT" * 1500, np.uint8).copy()
    pal = np.concatenate([g[:9000], synth.revcomp(g[:9000])])
    names, panel = synth.panel_genome(3, 1, 40_000, seed=4)
    nstart = g[:20000].copy()
    nstart[3] = ord("N"); nstart[11] = ord("n"); nstart[17] = ord("R")  # N inside the first k-1 bases: hashed as the letter N
    nstart[6000:6030] = ord("N")
    return {"random": g, "tandem": rep, "with_n": withn, "n_at_start": nstart, "low_complexity": low, "palindrome": pal,
            "panel": np.concatenate(panel), "short": g[:150], "tiny": g[:19]}


@needs_ref
@pytest.mark.parametrize("w,s,k", [(1000, 20, 19), (5000, 130, 19), (500, 10, 16), (2000, 64, 21), (100, 3, 19)])
def test_host_index_builder_matches_reference_addMinmers(w, s, k):
    for name, seq in _cases_for_index().items():
        ref = refh.add_minmers(seq, k, w, s, seq_id=3)
        got = hostlib.add_minmers(seq, k, w, s, seq_id=3)
        assert len(ref) == len(got), (name, len(ref), len(got))
        for f in ("hash", "wpos", "wpos_end", "seqId", "strand"):
            assert np.array_equal(ref[f], got[f]), (name, f)


@needs_ref
@pytest.mark.parametrize("w,s,k,chunk,warm", [(1000, 20, 19, 3000, 2000), (5000, 130, 19, 7000, 10000), (500, 10, 16, 1000, 1000),
                                              (2000, 64, 21, 2500, 4000), (100, 3, 19, 333, 200)])
def test_chunked_window_scan_equals_the_whole_contig_scan(w, s, k, chunk, warm):
    """the GPU index builder cuts a contig into chunks, scans each with its own window machine after a warm-up and
    stitches them (inherited record starts, state digests, re-scan of chunks whose warm state cannot be trusted): same
    records as one machine over the whole contig == the reference's addMinmers, on every kind of input"""
    rescanned = 0
    for name, seq in _cases_for_index().items():
        ref = refh.add_minmers(seq, k, w, s, seq_id=3)
        got, r = hostlib.add_minmers_chunked(seq, k, w, s, chunk, warm, seq_id=3)
        rescanned += r
        assert len(ref) == len(got), (name, len(ref), len(got), r)
        for f in ("hash", "wpos", "wpos_end", "seqId", "strand"):
            assert np.array_equal(ref[f], got[f]), (name, f, r)
    print("chunks re-scanned from exact state:", rescanned)


def _tail_params(R):
    p = R.p
    tp = hostlib.TailParams()
    for n in ("kmerSize", "segLength", "sketchSize", "filterMode", "numMappingsForSegment", "numMappingsForShortSequence",
              "block_length", "chain_gap", "mergeMappings", "stage1_topANI_filter", "keep_low_pct_id", "skip_self",
              "skip_prefix", "prefix_delim", "filterLengthMismatches", "legacy_output", "report_ANI_percentage",
              "percentageIdentity", "ANIDiff", "ANIDiffConf", "kmerComplexityThreshold"):
        setattr(tp, n, getattr(p, n))
    return tp


def _records_from_reference_stages(R, d, ri, seg_length, k):
    """device-format records for one read, produced by the reference's own stage functions"""
    read = d["reads"][ri]
    _, start, length = synth.split_segments([len(read)], seg_length, k)
    segs = np.zeros(len(start), dtype=capi.segment_dtype)
    seg_res = np.zeros(len(start), dtype=capi.segres_dtype)
    cands, loci = [], []
    for i in range(len(start)):
        frag = read[start[i] : start[i] + length[i]]
        o = R.map_fragment(d["rnames"][ri], frag, full_len=len(read), seq_counter=ri)
        segs[i] = (start[i], length[i], ri, -1, -1)
        raw = refh.sketch_sequence(frag, k, R.p.sketchSize)
        seg_res[i]["sketch_raw_count"] = len(raw)
        seg_res[i]["sketch_max_hash"] = raw["hash"][-1] if len(raw) else 0
        seg_res[i]["sketch_size"] = len(o["sketch"])
        seg_res[i]["first_candidate"] = len(cands)
        seg_res[i]["n_candidates"] = len(o["l1"])
        for ci, c in enumerate(o["l1"]):
            l2 = o["l2"][o["l2_cand"] == ci]
            cands.append((c["seqId"], c["rangeStartPos"], c["rangeEndPos"], c["intersectionSize"], i, len(loci), len(l2), 0))
            loci.extend(l2.tolist())
    return (segs, seg_res, np.array(cands, dtype=capi.l1_dtype) if cands else np.zeros(0, capi.l1_dtype),
            np.array(loci, dtype=capi.l2_dtype) if loci else np.zeros(0, capi.l2_dtype))


def _paf_fields(m, qname, names, lens):
    return (qname, int(m["queryLen"]), int(m["queryStartPos"]), int(m["queryEndPos"]), "+" if m["strand"] == 1 else "-",
            names[m["refSeqId"]], int(lens[m["refSeqId"]]), int(m["refStartPos"]), int(m["refEndPos"]),
            int(m["conservedSketches"]), int(m["blockLength"]))


@needs_ref
@pytest.mark.parametrize("which,args", [("random", ["-s", "5000", "--pi", "85"]),
                                        ("panel", ["-s", "5000", "--pi", "85"]),
                                        ("panel", ["-s", "2000", "--pi", "90", "-J", "25", "--noHgFilter", "-n", "3"]),
                                        ("panel", ["-s", "2000", "--pi", "90", "-J", "25", "--hgFilterAniDiff", "2", "--hgFilterConf", "99", "-n", "3"]),
                                        ("random", ["-s", "5000", "--pi", "85", "-f", "none"]),
                                        ("random", ["-s", "5000", "--pi", "85", "--noMerge"])])
def test_host_tail_matches_reference_mapModule(workdir, which, args):
    d = datasets.make_random_set(workdir, tag="tl") if which == "random" else datasets.make_panel_set(workdir, tag="tlp",
                                                                                                      n_strains=3, chrom_len=60_000)
    R = refh.RefSession(["-r", d["ref"], "-q", d["qry"], "-t", "2"] + args)
    try:
        tail = hostlib.HostTail(_tail_params(R), R.contig_names, R.contig_len)
        n_cmp = 0
        for ri in range(len(d["reads"])):
            if len(d["reads"][ri]) < R.p.kmerSize:
                continue
            segs, seg_res, cands, loci = _records_from_reference_stages(R, d, ri, R.p.segLength, R.p.kmerSize)
            text, n = tail.map_read(d["rnames"][ri], len(d["reads"][ri]), ri, segs, seg_res, cands, loci)
            ref = R.map_read(d["rnames"][ri], d["reads"][ri], ri)
            got = [tuple(l.split("\t")) for l in text.splitlines()]
            if len(ref) == 0 and len(got) == 1 and len(d["reads"][ri]) > R.p.segLength and \
                    int(got[0][3]) - int(got[0][2]) == R.p.segLength:
                continue  # reference UB on n_merged (see refh.is_uninitialised_n_merged_case)
            assert len(got) == len(ref), (ri, len(got), len(ref))
            for g, m in zip(got, ref):
                exp = _paf_fields(m, d["rnames"][ri], R.contig_names, R.contig_len)
                assert tuple(str(x) for x in exp) == g[:11], (ri, exp, g)
                idv = float(g[12].split(":")[2])
                assert abs(idv - float(m["nucIdentity"])) <= 1e-4
                n_cmp += 1
        assert n_cmp > 0
        tail.close()
    finally:
        R.close()


@needs_ref
@pytest.mark.parametrize("which,args,threads", [("random", ["-s", "5000", "--pi", "85"], 1), ("panel", ["-s", "5000", "--pi", "85"], 5),
                                                ("panel", ["-s", "1000", "--pi", "90", "-J", "40", "--kmerThreshold", "1"], 3)])
def test_host_index_equals_reference_sketch(workdir, which, args, threads):
    """skch::Sketch of the product (build + index + frequency filter) == the reference's Sketch members"""
    d = datasets.make_random_set(workdir, tag="hx") if which == "random" else datasets.make_panel_set(workdir, tag="hxp")
    R = refh.RefSession(["-r", d["ref"], "-q", d["ref"], "-t", "2"] + args)
    try:
        seqs = np.concatenate(d["genome"])
        offs = np.zeros(len(d["genome"]) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(g) for g in d["genome"]])
        pct = float(args[args.index("--kmerThreshold") + 1]) if "--kmerThreshold" in args else 0.001
        hi = hostlib.HostIndex.build(seqs, offs, R.p.kmerSize, R.p.segLength, R.p.sketchSize, threads=threads, kmer_pct_threshold=pct)
        mi, keys, offs2, pts, fr = hi.arrays()
        ref_mi = R.index()
        rkeys, roffs, rpts, rfr = R.lookup()
        assert hi.freq_threshold == R.freq_threshold()
        assert len(mi) == len(ref_mi)
        for f in ("hash", "wpos", "wpos_end", "seqId", "strand"):
            assert np.array_equal(mi[f], ref_mi[f]), f
        assert np.array_equal(keys, rkeys) and np.array_equal(offs2, roffs) and np.array_equal(fr, rfr)
        for f in ("pos", "hash", "seqId", "side"):
            assert np.array_equal(pts[f], rpts[f]), f
        hi.close()
    finally:
        R.close()


@pytest.mark.parametrize("n,threads", [(1500, 1), (60_000, 4), (150_000, 8)])
def test_run_wide_one_to_one_step_equals_its_plain_statement(n, threads):
    """-f one-to-one, the step mapQuery runs over ALL mappings at the end (computeMap.hpp:358-405): the product sorts through
    (key, index) pairs, sweeps the reference axis contig by contig on several threads and formats the PAF text in slices;
    same bytes as std::sort on the records + one serial sweep (filter.hpp:333-394) + one stream, on random mappings with many
    equal keys, equal identities and mappings that span a whole contig"""
    import ctypes as C

    L = hostlib.lib()
    L.skch_one_to_one_selftest.restype = C.c_int64
    L.skch_one_to_one_selftest.argtypes = [C.c_int64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    for seed in (1, 2, 3):
        tf, tp = C.c_double(), C.c_double()
        for span_every in (50, 0):  # contigs chained into few sweep units by spanning mappings / every contig on its own
            d = L.skch_one_to_one_selftest(n, seed, threads, 64, max(10, n // 2), span_every, C.byref(tf), C.byref(tp))
            print(f"n={n} seed={seed} span_every={span_every}: fast {tf.value * 1e3:.1f} ms, plain {tp.value * 1e3:.1f} ms")
            assert d == 0


def test_threaded_exact_sort_equals_std_sort_on_every_pattern():
    """sortExactlyLikeStd (libstdc++'s own partition / loop / heap / insertion routines with the recursive call handed to
    other threads) leaves (key, index) pairs exactly where std::sort leaves them -- ties included -- on random keys with many
    ties, sorted, reversed, organ-pipe and constant inputs, and on an antiqsort adversary built against std::sort itself,
    which drives the quicksort phase to its depth limit so that the heap-sort branch of the threaded version runs"""
    import ctypes as C

    L = hostlib.lib()
    L.skch_sort_selftest.restype = C.c_int64
    L.skch_sort_selftest.argtypes = [C.c_int64, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_int64)]
    heap_hits = 0
    for pattern in range(7):
        for n, threads in ((33_000, 2), (70_001, 5), (250_000, 8)):
            hb = C.c_int64()
            assert L.skch_sort_selftest(n, 11 + pattern, threads, pattern, C.byref(hb)) == 0, (pattern, n, threads)
            if pattern >= 5:
                heap_hits += hb.value
    assert heap_hits > 0  # the adversary did reach introsort's depth limit in the threaded code


def test_paf_text_without_a_stream_equals_the_stream_text():
    """reportReadMappings (computeMap.hpp:1758-1805) writes every field through operator<<; the product appends the same
    characters with std::to_chars (integers; %g with precision 6 for the mapping quality, identity, complexity and Jaccard
    values). Same bytes on 200 k random mappings per seed -- arbitrary floats, dyadic identities (exact decimal ties),
    0 and 1 -- in all eight output modes (legacy / percent identity / --noMerge)."""
    import ctypes as C

    L = hostlib.lib()
    L.skch_format_selftest.restype = C.c_int
    L.skch_format_selftest.argtypes = [C.c_int64, C.c_uint64]
    for seed in (1, 2, 3):
        assert L.skch_format_selftest(200_000, seed) == 0


def test_path_limits_are_checked_without_a_device():
    """mm_params_check: the limits of the device path (k, shared-memory budget of the sketch kernel) answered before any
    reference is read -- skch::Sketch calls it first -- and without a GPU"""
    import ctypes as C

    L = capi.lib()
    L.mm_params_check.restype = C.c_int
    L.mm_params_check.argtypes = [C.c_void_p]
    L.mm_last_error.restype = C.c_char_p
    L.mm_last_error.argtypes = [C.c_void_p]

    def check(k, seg, s):
        p = capi.Params(kmer_size=k, seg_length=seg, sketch_size=s)
        return L.mm_params_check(C.byref(p))

    assert check(19, 5000, 220) == 0
    assert check(16, 1000, 40) == 0
    assert check(19, 10000, 1000) == 0
    assert check(40, 5000, 220) != 0 and b"k-mer size" in L.mm_last_error(None)
    assert check(19, 400000, 220) != 0 and b"shared-memory" in L.mm_last_error(None)
