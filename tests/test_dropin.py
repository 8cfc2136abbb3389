"""Drop-in check (pytest -m gpu), for five command lines of the reference front end.

Every test first compares what libaugb200.so returns for the test's command line and input (the Viterbi paths, and the sampled
paths where the command line samples) with the reference's own results for the same command line, stored under tests/golden/ by
the make_golden*.py scripts.  That part needs nothing outside the repository.

Where the reference sources have been built into oracle/_ref/ by oracle/Makefile, the test then also runs the reference's own
front end with its three DP entry points bound to libaugb200.so (host/augshim.cc -> oracle/_ref/augustus_b200): it must print the
same GFF as the unmodified reference binary (oracle/_ref/augustus).  The reference binary is the checker there, the GPU library is
what runs the DP in augustus_b200."""
import gzip
import json
import os
import subprocess

import pytest

from augustus_b200 import Decoder, params, synth
from tests import util

pytestmark = pytest.mark.gpu

REFDIR = os.path.join(util.ROOT, "oracle", "_ref")
REF = os.path.join(REFDIR, "augustus")
DROPIN = os.path.join(REFDIR, "augustus_b200")
CFG = os.path.join(REFDIR, "config")

HAVE_BINARIES = os.path.exists(REF) and os.path.exists(DROPIN) and os.path.isdir(CFG)
EXAMPLE = os.path.join(util.GOLDEN, "example.fa")


def _same_paths(blob_name, seqs, refs):
    """Viterbi paths of the library == the reference's (states exactly, log probability within 1e-6 relative)."""
    dec = Decoder(util.blob_bytes(blob_name), 0)
    try:
        paths = dec.decode_batch(seqs)
    finally:
        dec.close()
    assert len(paths) == len(refs) == len(seqs)
    for p, ref in zip(paths, refs):
        assert p.status == 0 and p.as_tuples() == [tuple(s) for s in ref["states"]]
        assert abs(p.log_prob - ref["log_prob"]) <= 1e-6 * abs(ref["log_prob"])
    return paths


def _same_samples(blob_name, dna, ref_samples):
    """The 99 sampled paths of a process that starts with this sequence (rand() stream at position 0) == the reference's."""
    dec = Decoder(util.blob_bytes(blob_name), 0)
    try:
        dec.set_rand_position(0)
        _, samples = dec.decode_batch_sampling([dna], 100)
    finally:
        dec.close()
    assert len(samples[0]) == len(ref_samples) == 99
    for mine, theirs in zip(samples[0], ref_samples):
        assert mine.status == 0 and mine.as_tuples() == [tuple(x) for x in theirs["states"]]


def _run(exe, args, fasta):
    env = dict(os.environ, AUGUSTUS_CONFIG_PATH=CFG)
    r = subprocess.run([exe] + list(args) + [fasta], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-2000:]
    lines = r.stdout.splitlines()
    # the trailer echoes argv[0]; everything else must be identical
    if "# command line:" in lines:
        lines = lines[: lines.index("# command line:")]
    return lines


def _same_gff(args, fasta):
    want = _run(REF, args, fasta)
    got = _run(DROPIN, args, fasta)
    assert any(l.split("\t")[2:3] == ["CDS"] for l in want if not l.startswith("#")), "reference predicted nothing: weak test"
    assert got == want
    return want


def test_example_fa_human_ab_initio_gff_identical():
    """BASELINE.json configs[0]: examples/example.fa --species=human (two sequences, two GC classes)."""
    _same_paths("human", [dna for _, dna in util.read_fasta(EXAMPLE)], util.golden_paths()["example"])
    if HAVE_BINARIES:
        _same_gff(["--species=human", "--softmasking=0"], EXAMPLE)


def test_example_fa_utr_on_gff_identical_and_equals_reference_golden():
    """--UTR=on (71 states); the CDS / UTR features also equal the reference's own expected file
    tests/short/examples/expected_results/test_utr_on/aug_utr_on.gff (committed as tests/golden/aug_utr_on.gff): from the paths of
    the library (CDS parts, transcription start and end sites) and, with the reference build, from the drop-in's GFF."""
    seqs = util.read_fasta(EXAMPLE)
    paths = _same_paths("human_utr", [dna for _, dna in seqs], util.golden_paths(utr=True)["example"])
    par = params.parse(util.blob_bytes("human_utr"))
    for (name, _), p in zip(seqs, paths):
        assert util.path_features(p.as_tuples(), par) == util.gff_features(os.path.join(util.GOLDEN, "aug_utr_on.gff"), name)
    if not HAVE_BINARIES:
        return
    got = _same_gff(["--species=human", "--UTR=on", "--softmasking=0"], EXAMPLE)
    feats = [tuple(l.split("\t")[:8]) for l in got if not l.startswith("#")]
    gold = [tuple(l.rstrip("\n").split("\t")[:8]) for l in open(os.path.join(util.GOLDEN, "aug_utr_on.gff")) if not l.startswith("#") and "\t" in l]
    assert feats == gold


def test_sampling_posteriors_gff_identical():
    """--sample=100 --alternatives-from-sampling=true: the posterior probabilities and alternative transcripts in the GFF
    come from the Viterbi path + 99 sampled paths per sequence.  Two sequences in one process share one rand() stream
    (vitmatrix.cc:300); the shim carries the stream position across calls (augb200_set_rand_position).  Stored reference results:
    the Viterbi paths of both sequences, and the sampled paths of HS08198 in a process of its own (ref_samples.json.gz)."""
    seqs = util.read_fasta(EXAMPLE)
    _same_paths("human", [dna for _, dna in seqs], util.golden_paths()["example"])
    _same_samples("human", seqs[1][1], util.golden_samples()["example_HS08198"]["samples"])
    if HAVE_BINARIES:
        _same_gff(["--species=human", "--softmasking=0", "--sample=100", "--alternatives-from-sampling=true"], EXAMPLE)


def test_fly_defaults_softmasked_window_gff_identical(tmp_path):
    """--species=fly with its defaults (UTR on, softmasking on, sample=100) on a soft-masked chr2L window (config 3 shape).  Stored
    reference results: ref_paths_softmask.json (Viterbi path) and ref_samples_softmask.json.gz (99 sampled paths)."""
    name, dna = util.read_fasta(os.path.join(util.GOLDEN, "fly_softmask_window.fa"))[0]
    _same_paths("fly_softmask_utr", [dna], [json.load(open(os.path.join(util.GOLDEN, "ref_paths_softmask.json")))["masked"]])
    (_, rec), = json.load(gzip.open(os.path.join(util.GOLDEN, "ref_samples_softmask.json.gz"), "rt")).items()
    _same_samples("fly_softmask_utr", dna, rec["samples"])
    if not HAVE_BINARIES:
        return
    fa = str(tmp_path / "fly.fa")
    synth.write_fasta(fa, [dna], [name])
    _same_gff(["--species=fly"], fa)


def test_synthetic_50k_window_gff_identical(tmp_path):
    _same_paths("human", [synth.window(3, 50000)], [util.golden_paths()["synthetic50k"][3]])
    if not HAVE_BINARIES:
        return
    fa = str(tmp_path / "syn.fa")
    synth.write_fasta(fa, [synth.window(3, 50000)], ["w3"])
    _same_gff(["--species=human", "--softmasking=0"], fa)
