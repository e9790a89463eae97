"""The index image built on the device (mm_index_build) and the same index uploaded from host arrays (mm_index_upload)
are one image: the same header, the same bytes in every region, the same mapping results. The one freedom is where the
hash table keeps a key, which follows the order in which the device inserts the keys."""
import numpy as np
import pytest

from conftest import have_gpu
from mashmap_b200 import synth

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_gpu(), reason="no GPU")]

# mm_blob_header (mashmap_b200/csrc/mm_internal.h): the regions in image order, with their element size in bytes
REGIONS = (("idx_hash", 8), ("idx_wpos", 4), ("idx_wend", 4), ("idx_strand", 1), ("contig_start", 8), ("idx2_hash", 8),
           ("idx2_wend", 4), ("tab", 16), ("pts", 8), ("contig_len", 4), ("contig_name_id", 4), ("contig_group", 4),
           ("cutoffs", 4), ("min_hits", 4))
HEADER = np.dtype([("magic", "<u8"), ("total_bytes", "<u8"), ("n_minmers", "<u8"), ("n_keys", "<u8"), ("n_points", "<u8"),
                   ("n_contigs", "<i4"), ("tab_log2", "<i4"), ("n_cutoffs", "<i4"), ("n_min_hits", "<i4")]
                  + [("off_" + name, "<u8") for name, _ in REGIONS])


def read_image(ctx):
    """host copy of the context's index image and its header"""
    import torch
    from mashmap_b200 import dist

    ptr, n = ctx.index_blob()
    img = dist.wrap_device_memory(ptr, n, torch.device("cuda", ctx.device)).cpu().numpy()
    return img, img[: HEADER.itemsize].view(HEADER)[0]


def region(img, h, name):
    """the bytes a region holds; the padding up to the next region is never written"""
    n_mi, n_c = int(h["n_minmers"]), int(h["n_contigs"])
    count = {"contig_start": n_c + 1, "tab": 1 << int(h["tab_log2"]), "pts": int(h["n_points"]), "contig_len": n_c,
             "contig_name_id": n_c, "contig_group": n_c, "cutoffs": int(h["n_cutoffs"]), "min_hits": int(h["n_min_hits"])}
    size = dict(REGIONS)[name]
    off = int(h["off_" + name])
    return img[off : off + count.get(name, n_mi) * size]


def occupied_slots(tab_bytes):
    t = tab_bytes.view(np.uint64).reshape(-1, 2)
    return {tuple(x) for x in t[(t[:, 0] != 0) | (t[:, 1] != 0)].tolist()}


def canon(seg_res, cands, loci):
    """per segment: its results, candidates and their loci, without where the slices landed in the batch-wide arrays
    (that follows the order in which the CTAs reserved them)"""
    out = []
    for sr in seg_res:
        c = cands[sr["first_candidate"] : sr["first_candidate"] + sr["n_candidates"]]
        out.append((tuple(int(sr[f]) for f in ("sketch_max_hash", "sketch_raw_count", "sketch_size", "n_points", "minimum_hits",
                                               "best_intersection", "n_candidates")),
                    [(tuple(int(x[f]) for f in ("seqId", "rangeStartPos", "rangeEndPos", "intersectionSize", "segment", "n_loci")),
                      loci[x["first_locus"] : x["first_locus"] + x["n_loci"]].tobytes()) for x in c]))
    return out


def test_device_built_and_uploaded_index_images_are_the_same():
    from mashmap_b200 import capi, hostlib

    k, seg, s = 19, 2000, 60
    genome = synth.random_genome(3, 300_000, seed=11)
    reads, _ = synth.simulate_reads(genome, 120, 6000, 0.01, 0.08, seed=12)
    offs = np.zeros(len(genome) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(c) for c in genome])

    built = capi.Context(kmer_size=k, seg_length=seg, sketch_size=s)
    built.index_build(np.concatenate(genome), offs, keep_lookup=True)
    mi, keys, key_offs, pts, freq = built.index_download()
    uploaded = capi.Context(kmer_size=k, seg_length=seg, sketch_size=s)
    uploaded.index_upload(mi, keys, key_offs, pts, freq, np.diff(offs).astype(np.int32))
    for ctx in (built, uploaded):
        ctx.tables_upload(hostlib.sketch_cutoffs(s, k), hostlib.min_hits_table(s, k, 0.85))

    img_b, h_b = read_image(built)
    img_u, h_u = read_image(uploaded)
    assert h_b.tobytes() == h_u.tobytes(), (h_b, h_u)
    assert h_b["n_minmers"] == len(mi) > 0 and h_b["n_keys"] == len(keys) > 0 and h_b["n_points"] == len(pts)
    for name, _ in REGIONS:
        if name != "tab":
            assert np.array_equal(region(img_b, h_b, name), region(img_u, h_u, name)), name
    slots = occupied_slots(region(img_b, h_b, "tab"))
    assert len(slots) == len(keys)
    assert slots == occupied_slots(region(img_u, h_u, "tab"))

    lens = [len(r) for r in reads]
    ridx, start, length = synth.split_segments(lens, seg, k)
    roffs = np.zeros(len(lens) + 1, dtype=np.int64)
    roffs[1:] = np.cumsum(lens)
    segs = np.zeros(len(ridx), dtype=capi.segment_dtype)
    segs["offset"] = roffs[ridx] + start
    segs["length"] = length
    segs["seq_counter"] = ridx
    segs["name_id"] = -1
    segs["ref_group"] = -1
    bases = np.concatenate(reads)
    res_b = built.map_segments(bases, segs)
    res_u = uploaded.map_segments(bases, segs)
    assert len(res_b[1]) > 0 and len(res_b[2]) > 0
    assert canon(*res_b) == canon(*res_u)
    built.close()
    uploaded.close()
