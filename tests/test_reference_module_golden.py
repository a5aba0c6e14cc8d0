"""
Against the output directory of the REFERENCE'S OWN nn-classification module (tests/golden/reference_module/, made by
tests/golden/make_reference_module_golden.py: genomad/modules/nn_classification.py::main executed unmodified with the reference's
sequence.py / utils.py / _paths.py / model definition / nn_classifier.h5; only tensorflow and keras replaced by the NumPy stand-in
tests/golden/keras_shim.py).  CPU: the oracle pipeline and the host-side writers of genomad_b200 reproduce it.  GPU: the module.
"""
import json
import shutil
from pathlib import Path

import numpy as np
import pytest
import torch

from genomad_b200 import _paths, nn_classification, utils
from oracle import igloo_model as M
from oracle import tokenizer as T

RUNS = (("run_default", False), ("run_single_window_cleanup", True))
HEADER = "seq_name\tchromosome_score\tplasmid_score\tvirus_score"


@pytest.fixture(scope="module")
def gold(golden_dir):
    return golden_dir / "reference_module"


def _oracle(path, single, w):
    names, ids, _, tok = T.encode_fasta(path, single_window=single)
    p = np.concatenate([M.forward(tok[i:i + 8], w) for i in range(0, len(tok), 8)])
    return names, ids, T.segment_mean(p, ids, len(names))


def test_oracle_pipeline_matches_reference_module_run(gold, weights_npz, tmp_path):
    w = M.load_npz_weights(weights_npz)
    fa = gold / "input" / "toy.fna"
    pv = gold / "input" / "toy_find_proviruses" / "toy_provirus.fna"
    assert pv.exists()
    for run, single in RUNS:
        d = gold / run
        for path, npz, key, tsv in ((fa, "toy_nn_classification.npz", "contig_names", "toy_nn_classification.tsv"),
                                    (pv, "toy_provirus_nn_classification.npz", "provirus_names", "toy_provirus_nn_classification.tsv")):
            names, ids, pred = _oracle(path, single, w)
            z = np.load(d / npz)
            assert sorted(z.files) == sorted([key, "predictions"])
            assert z["predictions"].dtype == np.float32 and z["predictions"].shape == (len(names), 3)
            assert list(z[key]) == list(names) and z[key].dtype.kind == "U"
            assert np.abs(pred - z["predictions"]).max() <= 5e-5               # fp32 summation order (oracle vs NumPy stand-in)
            assert np.array_equal(pred.argmax(1), z["predictions"].argmax(1))
            # the TSV the reference wrote == genomad_b200's writer on the reference's predictions, byte for byte
            out = tmp_path / f"{run}_{tsv}"
            nn_classification._write_tsv(out, z[key], z["predictions"])
            assert out.read_bytes() == (d / tsv).read_bytes()
            assert (d / tsv).read_text().splitlines()[0] == HEADER
        if not single:
            # window -> contig bookkeeping of the encoding stage (N rule: ctg_c's 2nd window dropped; ctg_d's short tail dropped)
            ids_main = np.load(d / "toy_seq_window_id.npz")
            names, ids, _ = _oracle(fa, False, w)
            assert sorted(ids_main.files) == ["contig_ids", "contig_names"]
            assert list(ids_main["contig_names"]) == list(names) and ids_main["contig_ids"].tolist() == ids.tolist() == [0, 0, 0, 1, 2, 2, 3, 4]
            ids_pv = np.load(d / "toy_provirus_window_id.npz")
            assert sorted(ids_pv.files) == ["provirus_ids", "provirus_names"] and ids_pv["provirus_ids"].tolist() == [0, 0, 1]


def test_native_reader_matches_reference_encoding_stage(gold):
    """The native FASTA reader (csrc/fasta.cpp through sequence.ParsedFasta: index, window rules, N rule, padding, upper-casing)
    against what the reference's encoding stage produced for the same file: names, window -> contig ids (values and dtypes) and,
    after the oracle tokenizer, the very tokens the reference wrote into its TFRecord files -- bit for bit."""
    from genomad_b200 import sequence
    toks = np.load(gold / "run_default" / "encoded_tokens.npz")
    for path, id_npz, nk, ik, tk in ((gold / "input" / "toy.fna", "toy_seq_window_id.npz", "contig_names", "contig_ids", "sequences"),
                                     (gold / "input" / "toy_find_proviruses" / "toy_provirus.fna", "toy_provirus_window_id.npz",
                                      "provirus_names", "provirus_ids", "proviruses")):
        ref = np.load(gold / "run_default" / id_npz)
        for threads in (1, 3):
            p = sequence.ParsedFasta(path, False, threads)
            try:
                assert p.check()
                idx = p.index()
                assert idx.names.tolist() == ref[nk].tolist() and idx.names.dtype == ref[nk].dtype
                assert idx.contig_ids.tolist() == ref[ik].tolist() and idx.contig_ids.dtype == ref[ik].dtype
                enc = p.encode()
                assert np.array_equal(T.tokenize_windows(enc.windows), toks[tk])
                # streamed block export == whole export
                out = np.empty((2, 6000), np.uint8)
                p.export_windows(1, 2, out)
                assert np.array_equal(out, enc.windows[1:3])
            finally:
                p.close()
        # --single-window: first window of every record
        p = sequence.ParsedFasta(path, True, 2)
        try:
            first = np.concatenate([[0], np.flatnonzero(np.diff(ref[ik])) + 1])
            assert np.array_equal(T.tokenize_windows(p.encode().windows), toks[tk][first])
        finally:
            p.close()


def test_output_surface_matches_reference_module_run(gold, tmp_path):
    """File names, the execution-info JSON and the skip decision inputs, from the host code alone (no GPU)."""
    o = _paths.NNOutputs("toy", Path("OUT"))
    ours = {str(p.relative_to("OUT")) for p in (o.nn_classification_log, o.nn_classification_execution_info, o.nn_classification_npz_output,
                                                o.nn_classification_output, o.provirus_nn_classification_npz_output,
                                                o.provirus_nn_classification_output, o.seq_window_id_output, o.provirus_window_id_output)}
    ref_default = set(json.loads((gold / "run_default" / "files.json").read_text()))
    ref_single = set(json.loads((gold / "run_single_window_cleanup" / "files.json").read_text()))
    tfrec = {f for f in ref_default if f.endswith(".tfrec")}
    assert tfrec == {"toy_nn_classification/toy_encoded_sequences/8.tfrec", "toy_nn_classification/toy_encoded_proviruses/3.tfrec"}
    assert ours == ref_default - tfrec                       # .tfrec intermediates are opt-in here (--write-tfrecords)
    assert ref_single == {f for f in ours if "encoded" not in f}     # --cleanup removes both encoded directories
    fa = tmp_path / "toy.fna"
    shutil.copy(gold / "input" / "toy.fna", fa)
    for run, single in RUNS:
        ref = json.loads((gold / run / "toy_nn_classification.json").read_text())
        mine = tmp_path / f"{run}.json"
        utils.write_execution_info("nn_classification", fa, {"single_window": single}, mine)
        got = json.loads(mine.read_text())
        assert list(got) == list(ref) == ["module", "input", "input_md5", "start_time", "parameters"]
        assert {k: v for k, v in got.items() if k != "start_time"} == {k: v for k, v in ref.items() if k != "start_time"}
        assert mine.read_text().count("\n") == (gold / run / "toy_nn_classification.json").read_text().count("\n")
        assert utils.compare_executions(fa, {"single_window": single}, gold / run / "toy_nn_classification.json")
        assert not utils.compare_executions(fa, {"single_window": not single}, gold / run / "toy_nn_classification.json")


_EVENTS = (
    ("executing", r"Executinggenomadnn-classification\."),
    ("previous_execution_detected", r"Previousexecutiondetected"),
    ("input_or_parameters_changed", r"Theinputfileortheparameterschanged"),
    # the path may contain dots (e.g. a temporary directory under a user name like first.last): it runs to the first "directory."
    ("mkdir_module", r"Creatingthe(?:(?!directory\.).)*?/toy_nn_classificationdirectory\."),
    ("mkdir_encoded_sequences", r"Creatingthe(?:(?!directory\.).)*?/toy_encoded_sequencesdirectory\."),
    ("mkdir_encoded_proviruses", r"Creatingthe(?:(?!directory\.).)*?/toy_encoded_provirusesdirectory\."),
    ("skip_sequence_encoding", r"toy_encoded_sequenceswasfound\.Skippingsequenceencoding"),
    ("skip_provirus_encoding", r"toy_encoded_proviruseswasfound\.Skippingprovirusencoding"),
    ("encoded_sequences", r"Encodedsequencedatawrittento"),
    ("encoded_proviruses", r"Encodedprovirusdatawrittento"),
    ("skip_sequence_classification", r"toy_nn_classification\.npzwasfound\.Skippingsequenceclassification"),
    ("skip_provirus_classification", r"toy_provirus_nn_classification\.npzwasfound\.Skippingprovirusclassification"),
    ("sequences_classified", r"Sequencesclassified\."),
    ("proviruses_classified", r"Provirusesclassified\."),
    ("sequence_npz_written", r"Sequenceclassificationinbinaryformatwrittento"),
    ("provirus_npz_written", r"Provirusclassificationinbinaryformatwrittento"),
    ("delete_encoded_sequences", r"Deletingencodedsequencedata\."),
    ("delete_encoded_proviruses", r"Deletingencodedprovirusdata\."),
    ("sequence_tsv_written", r"Sequenceclassificationintabularformatwrittento"),
    ("provirus_tsv_written", r"Provirusclassificationintabularformatwrittento"),
    ("finished", r"geNomadnn-classificationfinished!"),
)


def _events(text):
    """The module's log as a sequence of events: header panel and timestamps dropped, ALL white space removed (rich wraps long
    lines, also inside paths), every message pattern located, ordered by position."""
    import re
    body = "\n".join(l for l in text.splitlines() if not l.lstrip().startswith(("│", "╭", "╰")))
    body = re.sub(r"^\[\d\d:\d\d:\d\d\] ", "", body, flags=re.M)
    flat = re.sub(r"\s+", "", body)
    found = [(m.start(), name) for name, pat in _EVENTS for m in re.finditer(pat, flat)]
    return [name for _, name in sorted(found)]


def _skip_restart_scenarios(gold, fa, out):
    """Second and later runs in the same directory, against the reference module's logs of the same scenarios
    (tests/golden/reference_module/scenario_logs.json): nothing changed -> every step skipped; the provirus NPZ lost -> only the
    provirus classification is redone; --restart; parameter change (--single-window, --cleanup)."""
    ref = json.loads((gold / "scenario_logs.json").read_text())
    o = _paths.NNOutputs("toy", out)
    watched = (o.nn_classification_npz_output, o.provirus_nn_classification_npz_output)

    def run(name, *args):
        before = {p.name: p.stat().st_mtime_ns for p in watched if p.exists()}
        nn_classification.main(fa, out, *args)
        mine, want = _events(o.nn_classification_log.read_text()), _events(ref[name])
        assert mine == want, (name, mine, want)
        return before, {p.name: p.stat().st_mtime_ns for p in watched if p.exists()}
    b, a = run("rerun_unchanged", False, 4, False, 2, False, False)
    assert a == b                                              # nothing rewritten
    o.provirus_nn_classification_npz_output.unlink()
    b, a = run("provirus_npz_lost", False, 4, False, 2, False, False)
    assert a["toy_nn_classification.npz"] == b["toy_nn_classification.npz"] and "toy_provirus_nn_classification.npz" in a
    run("restart", False, 4, True, 2, False, False)
    run("parameter_change_single_window_cleanup", True, 4, False, 2, False, True)
    assert not o.encoded_sequences_dir.exists() and not o.encoded_proviruses_dir.exists()
    z = np.load(o.nn_classification_npz_output)
    r = np.load(gold / "run_single_window_cleanup" / "toy_nn_classification.npz")
    assert list(z["contig_names"]) == list(r["contig_names"]) and np.abs(z["predictions"] - r["predictions"]).max() <= 1e-4


def _run_module_and_compare(gold, tmp_path):
    """genomad_b200.nn_classification.main on the golden input, both runs: same files, names, NPZ keys / dtypes, JSON, log messages;
    scores within 1e-4 of the reference module's, TSV equal up to one unit in the 4th decimal."""
    for run, single in RUNS:
        work = tmp_path / run
        shutil.copytree(gold / "input", work)
        out = work / "out"
        out.mkdir()
        shutil.move(str(work / "toy_find_proviruses"), str(out / "toy_find_proviruses"))
        # the reference compares the md5 of the input with the one in the find-proviruses execution info: same file content here
        nn_classification.main(work / "toy.fna", out, single, 4, False, 2, False, single)
        d = gold / run
        ref_files = {f for f in json.loads((d / "files.json").read_text()) if not f.endswith(".tfrec")}
        got_files = {str(p.relative_to(out)) for p in out.rglob("*") if p.is_file() and "find_proviruses" not in str(p)}
        assert got_files == ref_files, (run, got_files ^ ref_files)
        sub = out / "toy_nn_classification"
        for npz, key, tsv in (("toy_nn_classification.npz", "contig_names", "toy_nn_classification.tsv"),
                              ("toy_provirus_nn_classification.npz", "provirus_names", "toy_provirus_nn_classification.tsv")):
            z, r = np.load(sub / npz), np.load(d / npz)
            assert sorted(z.files) == sorted(r.files)
            assert list(z[key]) == list(r[key]) and z[key].dtype == r[key].dtype
            assert z["predictions"].dtype == r["predictions"].dtype == np.float32 and z["predictions"].shape == r["predictions"].shape
            assert np.abs(z["predictions"] - r["predictions"]).max() <= 1e-4
            assert np.array_equal(z["predictions"].argmax(1), r["predictions"].argmax(1))
            mine, ref = (sub / tsv).read_text().splitlines(), (d / tsv).read_text().splitlines()
            assert mine[0] == ref[0] == HEADER and len(mine) == len(ref)
            for a, b in zip(mine[1:], ref[1:]):
                fa_, fb_ = a.split("\t"), b.split("\t")
                assert fa_[0] == fb_[0] and len(fa_) == len(fb_) == 4
                assert all(len(x) == 6 and abs(float(x) - float(y)) <= 1.0001e-4 for x, y in zip(fa_[1:], fb_[1:]))
        if not single:
            for f, keys in (("toy_encoded_sequences/toy_seq_window_id.npz", ("contig_names", "contig_ids")),
                            ("toy_encoded_proviruses/toy_provirus_window_id.npz", ("provirus_names", "provirus_ids"))):
                z, r = np.load(sub / f), np.load(d / Path(f).name)
                assert sorted(z.files) == sorted(r.files) == sorted(keys)
                for k in keys:
                    assert z[k].tolist() == r[k].tolist() and z[k].dtype == r[k].dtype
        got = json.loads((sub / "toy_nn_classification.json").read_text())
        ref = json.loads((d / "toy_nn_classification.json").read_text())
        assert list(got) == list(ref) and {k: v for k, v in got.items() if k != "start_time"} == {k: v for k, v in ref.items() if k != "start_time"}
        mine, ref = _events((out / "toy_nn_classification.log").read_text()), _events((d / "log_without_timestamps.txt").read_text())
        assert mine == ref and len(ref) >= 12, (run, mine, ref)          # same messages in the same order
        if not single:
            _skip_restart_scenarios(gold, work / "toy.fna", out)


def test_module_host_logic_matches_reference_module_run(gold, tmp_path, weights_npz, monkeypatch):
    """The module driver's host side (index, provirus twin, writers, cleanup, log) with the CUDA classifier replaced by the CPU
    oracle, against the reference module's output directory -- what the GPU test below checks with the real classifier."""
    w = M.load_npz_weights(weights_npz)

    def oracle_classify(clf, parsed, offsets, info, contig_reduce="gather"):
        windows = parsed.export_windows(0, parsed.n_windows, np.zeros((max(1, parsed.n_windows), 6000), np.uint8))
        tok = T.tokenize_windows(windows)
        p = np.concatenate([M.forward(tok[i:i + 8], w) for i in range(0, len(tok), 8)])
        return T.segment_mean(p, np.repeat(np.arange(len(offsets) - 1), np.diff(offsets)), len(offsets) - 1)
    monkeypatch.setattr(nn_classification, "_make_classifier", lambda batch_size, device: object())
    monkeypatch.setattr(nn_classification, "_classify_parsed", oracle_classify)
    _run_module_and_compare(gold, tmp_path)


def test_reference_consumer_accepts_our_outputs(gold, golden_dir, tmp_path, weights_npz):
    """Drop-in on the consumer side (INTEGRATION.md level 1): the REFERENCE'S real aggregated-classification module
    (genomad/modules/aggregated_classification.py) ran on a directory written by genomad_b200's nn-classification module -- its
    required-file list, the md5 cross-check against our execution-info JSON, the NPZ keys -- and what it consumed and produced is
    stored (tests/golden/reference_consumer/, make_reference_consumer_golden.py).  The same directory written now has the same
    files and nn-classification NPZs, and genomad_b200's own aggregated-classification produces from those NPZs what the reference
    produced, byte for byte."""
    import sys
    from genomad_b200 import aggregated_classification as our_agg
    sys.path.insert(0, str(golden_dir))
    import make_reference_consumer_golden as G
    ref = golden_dir / "reference_consumer"
    fa, out = G.build_case(gold, tmp_path / "case", weights_npz)
    files = sorted(str(p.relative_to(out)) for p in out.rglob("*") if p.is_file())
    assert files == json.loads((ref / "files.json").read_text())
    for npz, key in (("toy_nn_classification.npz", "contig_names"), ("toy_provirus_nn_classification.npz", "provirus_names")):
        z, r = np.load(out / "toy_nn_classification" / npz), np.load(ref / "consumed" / npz)
        assert sorted(z.files) == sorted(r.files) == sorted([key, "predictions"])
        assert z[key].tolist() == r[key].tolist() and z[key].dtype == r[key].dtype
        assert z["predictions"].dtype == r["predictions"].dtype and np.abs(z["predictions"] - r["predictions"]).max() <= 1e-6
        shutil.copy(ref / "consumed" / npz, out / "toy_nn_classification" / npz)     # the reference's exact inputs
    our_agg.main(fa, out, restart=False, verbose=False)
    expected = sorted(p.name for p in (ref / "expected").iterdir())
    assert expected == ["toy_aggregated_classification.npz", "toy_aggregated_classification.tsv",
                        "toy_provirus_aggregated_classification.npz", "toy_provirus_aggregated_classification.tsv"]
    for name in expected:
        if name.endswith(".tsv"):
            assert (out / "toy_aggregated_classification" / name).read_bytes() == (ref / "expected" / name).read_bytes(), name
        else:
            z, r = np.load(out / "toy_aggregated_classification" / name), np.load(ref / "expected" / name)
            assert sorted(z.files) == sorted(r.files)
            for k in z.files:
                assert z[k].dtype == r[k].dtype and np.array_equal(z[k], r[k]), (name, k)


@pytest.mark.gpu
def test_module_matches_reference_module_run(gold, tmp_path):
    """The same comparison with the real classifier on the B200."""
    _run_module_and_compare(gold, tmp_path)
