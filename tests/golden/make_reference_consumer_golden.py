#!/usr/bin/env python
"""
The REFERENCE'S real aggregated-classification module (genomad/modules/aggregated_classification.py, loaded like
make_aggregate_golden.py) run on an output directory written by genomad_b200's nn-classification module, with the CUDA classifier
replaced by the CPU oracle, plus marker-classification files (seeded random features / scores, names from our outputs).  It exits
on any missing file or md5 mismatch, so a stored result means it accepted our directory.

    python tests/golden/make_reference_consumer_golden.py     # needs the reference checkout -> tests/golden/reference_consumer/

Stored: the list of files the reference module found, the two nn-classification NPZs it consumed (consumed/) and the TSV / NPZ it
produced from them (expected/).  tests/test_reference_module_golden.py::test_reference_consumer_accepts_our_outputs rebuilds the
directory with `build_case` and checks genomad_b200's aggregated-classification against them.
"""
import json
import shutil
import sys
import tempfile
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
OUT = HERE / "reference_consumer"


def build_case(gold_module: Path, work: Path, weights_npz: Path):
    """nn-classification of gold_module/input into work/out (oracle classifier), then marker-classification files; -> (fasta, out)."""
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(HERE))
    from genomad_b200 import nn_classification, utils
    from oracle import igloo_model as M, tokenizer as T
    import make_aggregate_golden as G
    w = M.load_npz_weights(weights_npz)

    def oracle_classify(clf, parsed, offsets, info, contig_reduce="gather"):
        windows = parsed.export_windows(0, parsed.n_windows, np.zeros((max(1, parsed.n_windows), 6000), np.uint8))
        tok = T.tokenize_windows(windows)
        p = np.concatenate([M.forward(tok[i:i + 8], w) for i in range(0, len(tok), 8)])
        return T.segment_mean(p, np.repeat(np.arange(len(offsets) - 1), np.diff(offsets)), len(offsets) - 1)
    shutil.copytree(gold_module / "input", work)
    out = work / "out"
    out.mkdir()
    shutil.move(str(work / "toy_find_proviruses"), str(out / "toy_find_proviruses"))
    fa = work / "toy.fna"
    saved = nn_classification._make_classifier, nn_classification._classify_parsed
    nn_classification._make_classifier = lambda batch_size, device: object()
    nn_classification._classify_parsed = oracle_classify
    try:
        nn_classification.main(fa, out, False, 4, False, 2, False, False)
    finally:
        nn_classification._make_classifier, nn_classification._classify_parsed = saved
    nn_dir = out / "toy_nn_classification"
    names = np.load(nn_dir / "toy_nn_classification.npz")["contig_names"]
    pnames = np.load(nn_dir / "toy_provirus_nn_classification.npz")["provirus_names"]
    rng = np.random.default_rng(3)
    mk = out / "toy_marker_classification"
    mk.mkdir()
    utils.write_execution_info("marker_classification", fa, {}, mk / "toy_marker_classification.json")
    np.savez_compressed(mk / "toy_features.npz", contig_names=names, contig_features=rng.random((len(names), 25)).astype(np.float32))
    np.savez_compressed(mk / "toy_provirus_features.npz", provirus_names=pnames,
                        provirus_features=rng.random((len(pnames), 25)).astype(np.float32))
    np.savez_compressed(mk / "toy_marker_classification.npz", contig_names=names, predictions=G._scores(rng, len(names), np.float32))
    np.savez_compressed(mk / "toy_provirus_marker_classification.npz", provirus_names=pnames,
                        predictions=G._scores(rng, len(pnames), np.float32))
    return fa, out


def main():
    import make_aggregate_golden as G
    with tempfile.TemporaryDirectory() as td:
        fa, out = build_case(HERE / "reference_module", Path(td) / "case", ROOT / "genomad_b200" / "data" / "nn_classifier.npz")
        files = sorted(str(p.relative_to(out)) for p in out.rglob("*") if p.is_file())
        agg, ref_utils = G.load_reference_module()
        ref_utils.metadata = types.SimpleNamespace(version=lambda _name: "reference-from-source")
        agg.main(fa, out, restart=False, verbose=False)          # sys.exit(1) on any missing file / md5 mismatch
        if OUT.exists():
            shutil.rmtree(OUT)
        (OUT / "consumed").mkdir(parents=True)
        (OUT / "expected").mkdir()
        (OUT / "files.json").write_text(json.dumps(files, indent=1) + "\n")
        for name in ("toy_nn_classification.npz", "toy_provirus_nn_classification.npz"):
            shutil.copy(out / "toy_nn_classification" / name, OUT / "consumed" / name)
        for p in sorted((out / "toy_aggregated_classification").iterdir()):
            if p.suffix in (".tsv", ".npz"):
                shutil.copy(p, OUT / "expected" / p.name)
    print("wrote", OUT, sorted(p.name for p in (OUT / "expected").iterdir()))


if __name__ == "__main__":
    main()
