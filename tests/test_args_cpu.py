"""The product's option parser fills skch::Parameters exactly as the reference's parseandSave does
(reference src/map/include/parseCmdArgs.hpp:257-659: defaults, automatic sketch size from the file size, --dense,
filter modes, chaining / block-length defaults, skip-self when no query is given ...). CPU only. The reference's
Parameters for every command line here are stored in tests/golden/reference_params.json (written by
tests/golden/make_reference_params.py through oracle/_ref), so the comparison needs no reference build."""
import json
import os

import pytest

import datasets
import refh
from mashmap_b200 import hostlib

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_params.json")

OPTION_SETS = [
    [],
    ["-s", "5000", "--pi", "85"],
    ["-s", "3000", "--pi", "90", "-f", "one-to-one"],
    ["-s", "5000", "--pi", "95", "--dense"],
    ["-s", "2000", "--pi", "80", "-k", "16", "-J", "25", "--noHgFilter"],
    ["-s", "10000", "--pi", "90", "-n", "3", "--noMerge", "-f", "none"],
    ["-s", "5000", "-X", "-Y", "#", "--lowerTriangular"],
    ["-s", "5000", "-c", "20000", "-l", "10000", "--kmerThreshold", "0.1", "--kmerComplexity", "0.5"],
    ["-s", "1000", "--pi", "99", "--hgFilterAniDiff", "0.5", "--hgFilterConf", "99.0", "--filterLengthMismatches"],
    ["-s", "5000", "-M", "--legacy", "--reportPercentage", "--sparsifyMappings", "0.5"],
    ["-s", "5000", "--numMappingsForShortSeq", "4", "-n", "2", "--dropLowMapId"],
]


@pytest.fixture(scope="module")
def d(workdir):
    return datasets.make_panel_set(workdir, tag="args", n_strains=2, chrom_len=40_000)


def cli_args(d, opts, with_query):
    return ["-r", d["ref"]] + (["-q", d["qry"]] if with_query else []) + ["-t", "2"] + opts


def params_key(opts, with_query):
    return " ".join(["with query" if with_query else "no query"] + opts)


def size_args(path):
    return ["-r", path, "-q", path, "-s", "5000", "--pi", "85"]


def write_sparse_fasta(path, size):
    with open(path, "wb") as fh:
        fh.write(b">c\nACGT\n")
        fh.truncate(size)


def reference_params(key):
    """skch::Parameters the reference's parseandSave filled for the command line `key`, as {field: value}"""
    with open(GOLDEN) as f:
        return json.load(f)[key]


@pytest.mark.parametrize("opts", OPTION_SETS, ids=lambda o: " ".join(o) or "defaults")
@pytest.mark.parametrize("with_query", [True, False])
def test_parameters_equal_reference(d, opts, with_query):
    args = cli_args(d, opts, with_query)
    ref = reference_params(params_key(opts, with_query))
    ours = hostlib.HostIndex.from_cli(args)
    p = ours.params_into(refh.OrcParams())
    for name, _ in refh.OrcParams._fields_:
        a, b = ref[name], getattr(p, name)
        assert a == b, (name, a, b, args)
    ours.close()


SIZES = [2**31 - 1000, 2**31 + 1000, 3_100_000_000, 5_000_000_000, 2**32 + 4096]


@pytest.mark.parametrize("size", SIZES)
def test_reference_size_wraps_like_the_reference(tmp_path, size):
    """map_parameters.hpp:41 keeps referenceSize in an offset_t (int32): for files >= 2 GiB the value wraps and is
    sign-extended into recommendedSketchSize (parseCmdArgs.hpp:304,639), so the automatic sketch size differs from the
    one the formula gives for the true size. The product reproduces that (a sparse file stands in for the FASTA)."""
    f = str(tmp_path / "big.fa")
    write_sparse_fasta(f, size)
    ref = reference_params(f"size {size}")
    ours = hostlib.HostIndex.params_from_cli(size_args(f))
    p = ours.params_into(refh.OrcParams())
    ours.close()
    assert p.referenceSize == ref["referenceSize"]
    assert p.sketchSize == ref["sketchSize"]
