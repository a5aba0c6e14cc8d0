"""CPU tests of the host side: FASTA/windowing vs reference golden vectors, weights/H5 reader, C-ABI exports,
module driver output surface (with a stub classifier -- the real one needs a B200)."""
import ctypes
import gzip
import json
import re

import numpy as np
import pytest

from genomad_b200 import _paths, engine, h5lite, nn_classification, sequence, utils, weights
from oracle import tokenizer as T


@pytest.fixture(scope="module")
def enc(golden_dir):
    return json.loads((golden_dir / "encoder_golden.json").read_text())


# ------------------------------------------------------------------------------------------ sequence
def test_iter_fasta_matches_reference(enc, tmp_path):
    for name, case in enc["fasta"].items():
        p = tmp_path / f"{name}.fna"
        p.write_text(case["text"], newline="")
        got = [[h, sequence.accession(h), s.decode()] for h, s in sequence.iter_fasta(p)]
        assert got == [list(r) for r in case["records"]], name
        assert sequence.check_fasta(p) == case["check_fasta"], name


def test_old_mac_newlines_and_gzip(tmp_path):
    text = ">a x\rACGT\rAC\r>b\rTT\r"
    p = tmp_path / "mac.fna"
    p.write_text(text, newline="")
    assert [(h, s) for h, s in sequence.iter_fasta(p)] == [("a x", b"ACGTAC"), ("b", b"TT")]
    assert [(h, s.encode()) for h, s in T.read_fasta(p)] == [("a x", b"ACGTAC"), ("b", b"TT")]
    g = tmp_path / "x.fna.gz"
    with gzip.open(g, "wt") as fh:
        fh.write(">a\nNNACGTNN\n")
    assert list(sequence.iter_fasta(g)) == [("a", b"ACGT")]
    assert sequence.is_compressed(g) == sequence.Compression.gzip


def test_window_spans_match_reference(enc):
    for case in enc["windows"]:
        assert [e - s for s, e in sequence.window_spans(case["len"])] == case["multi"]
        assert [e - s for s, e in sequence.window_spans(case["len"], single_window=True)] == case["single"]


def test_encode_fasta_matches_oracle(enc, tmp_path):
    rng = np.random.default_rng(3)
    recs = []
    for i, ln in enumerate([10000, 400, 2499, 14500, 6000, 30000, 8499]):
        s = np.frombuffer(b"ACGTNacgtnRY", np.uint8)[rng.choice(12, ln, p=[.2, .2, .2, .2, .04, .03, .03, .03, .03, .01, .02, .01])]
        recs.append(f">c{i} some description\n" + "\n".join(s.tobytes().decode()[k:k + 70] for k in range(0, ln, 70)))
    for case in enc["nrule"]:
        recs.append(f">{case['name']}\n{case['raw']}")
    p = tmp_path / "mix.fna"
    p.write_text("\n".join(recs) + "\n")
    for single in (False, True):
        e = sequence.encode_fasta(p, single_window=single)
        names, ids, ascii_arr, _tok = T.encode_fasta(p, single_window=single)
        assert list(e.names) == list(names)
        assert np.array_equal(e.contig_ids, ids)
        assert np.array_equal(e.windows, ascii_arr)
        assert e.offsets[-1] == len(ids) and np.all(np.diff(e.offsets) >= 1)
    for case in enc["nrule"]:
        q = tmp_path / "n.fna"
        q.write_text(f">x\n{case['raw']}\n")
        assert len(sequence.encode_fasta(q).contig_ids) == len(case["kept"]), case["name"]


# ------------------------------------------------------------------------------------------ weights
def test_weights_npz_and_shapes(weights_npz):
    w = weights.load_weights(weights_npz)
    assert w["c1w"].shape == (6, 257, 128) and w["ig1_random_patches"].dtype == np.int32
    # spot values recorded from the H5 during the survey (SURVEY.md Appendix A)
    assert np.allclose(w["c1w"][0, 0, :3], [-0.0358333, 0.0309101, 0.0279195], atol=1e-7)
    assert np.allclose(w["d2b"], [0.0138235, -0.0161939, -0.0010647], atol=1e-7)
    assert w["ig0_random_patches"][0, :, 0].tolist() == [296, 948, 3644, 4375]
    assert w["ig1_random_patches"][1, :, 0].tolist() == [958, 1714, 3162, 5978]
    assert float(np.abs(w["ig0_w_mult"]).max()) < 1e-30          # the shipped patch weights are numerically dead
    z = np.load(weights_npz)
    assert str(z["__sha256__"]) == "834bcb03aeb1ff484dc7c1f7c00fb951708a91ed03d8a233cd176390930761a1"


def test_h5lite_reads_reference_file_if_present(weights_npz, golden_dir, tmp_path):
    """The reference's nn_classifier.h5, rebuilt byte for byte from its stored non-payload bytes and the weights' arrays
    (tests/golden/make_h5_skeleton.py)."""
    import hashlib
    import sys
    sys.path.insert(0, str(golden_dir))
    import make_h5_skeleton
    raw = make_h5_skeleton.rebuild(golden_dir / "nn_classifier_h5_skeleton.npz", weights_npz)
    assert hashlib.sha256(raw).hexdigest() == str(np.load(weights_npz)["__sha256__"])
    ref = tmp_path / "nn_classifier.h5"
    ref.write_bytes(raw)
    f = h5lite.H5File(ref)
    z = np.load(weights_npz)
    assert len(f.datasets) == 32
    for k, v in f.datasets.items():
        assert np.array_equal(v, z[k]), k
    assert f.offsets["/model/conv1d/kernel:0"] == 1087096
    assert f.attrs["/"]["keras_version"] == "2.7.0"
    w = weights.load_weights(ref)
    assert np.array_equal(w["c2w"], z["/model/conv1d_1/kernel:0"])


def test_weights_validation_rejects_bad_shapes(weights_npz):
    z = np.load(weights_npz)
    raw = {k: z[k] for k in z.files if k.startswith("/")}
    raw["/model/conv1d_1/kernel:0"] = raw["/model/conv1d_1/kernel:0"][:5]
    with pytest.raises(ValueError):
        weights._validate(raw)


# ------------------------------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol(repo_root):
    header = (repo_root / "include" / "gnm.h").read_text()
    declared = set(re.findall(r"\b(gnm_[a-z_0-9]+)\s*\(", header))
    assert declared >= {"gnm_create", "gnm_encode", "gnm_forward_ascii", "gnm_segment_mean", "gnm_classify_host"}
    lib = engine.load_library()
    for name in sorted(declared):
        assert hasattr(lib, name), f"libgnm.so does not export {name}"
    assert set(engine.EXPORTS) == declared
    assert b"sm_100a" in lib.gnm_version()


def _pack_patches(patches, w_mult, w_summer):
    """gnm_pack_patches through ctypes -> dict of numpy arrays (host only)."""
    lib = engine.load_library()
    lay = (ctypes.c_int * 4)()
    assert lib.gnm_pack_patches(None, None, None, None, None, None, None, None, None, None, None, lay) == 0
    band_rows, n_bands, slots, group_max = list(lay)
    out = {"band_rows": band_rows, "n_bands": n_bands, "slots": slots, "group_max": group_max,
           "slot_of": np.empty(8400, np.int32), "ent_pos": np.empty(slots, np.int32), "ent_w": np.empty((slots, 128), np.float32),
           "groups": np.empty((8400, 2), np.int32), "band_first": np.empty(n_bands + 1, np.int32),
           "frag": np.empty((slots, 2, 4, 4, 4), np.uint32)}
    n_groups = ctypes.c_int(8400)
    unscale = ctypes.c_float(0)
    p = np.ascontiguousarray(patches, np.int32)
    wm = np.ascontiguousarray(w_mult, np.float32)
    ws = np.ascontiguousarray(w_summer, np.float32)
    rc = lib.gnm_pack_patches(p.ctypes.data, wm.ctypes.data, ws.ctypes.data, out["slot_of"].ctypes.data, out["ent_pos"].ctypes.data,
                              out["ent_w"].ctypes.data, out["groups"].ctypes.data, ctypes.byref(n_groups), out["band_first"].ctypes.data,
                              out["frag"].ctypes.data, ctypes.byref(unscale), None)
    assert rc == 0, lib.gnm_last_error()
    out["groups"] = out["groups"][:n_groups.value]
    out["unscale"] = unscale.value
    return out


def _frag_halves(words):
    """uint32 words of two fp16 -> float32 [..., 2] (low half first)."""
    w = np.ascontiguousarray(words, np.uint32)
    return w.view(np.uint16).reshape(w.shape + (2,)).view(np.float16).astype(np.float32)


@pytest.mark.parametrize("kind", ["random", "one_position", "ends", "one_band", "band_edges"])
def test_patch_packing_for_the_fused_gather(kind):
    """Host logic of the fused IGLOO kernel (csrc/api.cu pack_patches; kernel side csrc/wv_gather.cuh): every (patch, k) entry
    lands in exactly one position group of <= 4 entries that share a position inside the right band, and the mma B fragments
    reproduce the folded weights w_mult * w_summer / 32 (reference igloo.py:199-204) to fp32 accuracy.  Then the kernel's
    arithmetic is replayed in NumPy on random activations: sum over the fragment lanes of (hi16 + lo16 row) x (hi + lo weight
    half) with the kernel's channel mapping == the plain dot product."""
    rng = np.random.default_rng(5)
    if kind == "random":
        patches = rng.integers(0, 5997, size=(2100, 4), dtype=np.int32)
    elif kind == "one_position":
        patches = np.full((2100, 4), 3001, np.int32)
    elif kind == "ends":
        patches = np.tile(np.asarray([0, 1, 5995, 5996], np.int32), (2100, 1))
    elif kind == "one_band":                                       # 8,400 entries on the 24 positions of one band: 350 per position
        patches = (2400 + rng.integers(0, 24, size=(2100, 4))).astype(np.int32)
    else:                                                          # only first / last positions of bands, incl. the short last band
        edges = np.array([0, 23, 24, 47, 5975, 5976, 5996, 5995, 2399, 2400], np.int32)
        patches = edges[rng.integers(0, len(edges), size=(2100, 4))]
    w_mult = (rng.standard_normal((2100, 4, 128)) * 0.05).astype(np.float32)
    w_mult[7] = 0.0                                               # an all-zero patch
    w_mult[8, 1, :5] = [1e-9, -3e-7, 2.5, -1e-4, 6e-6]              # a wide dynamic range inside one entry
    w_summer = rng.standard_normal(512).astype(np.float32)
    o = _pack_patches(patches, w_mult, w_summer)
    R, NB, GM = o["band_rows"], o["n_bands"], o["group_max"]
    assert NB * R >= 5997 > (NB - 1) * R and R % 8 == 0 and GM == 4

    # slots: a permutation of the 8,400 entries, sorted by position, folded weights exact
    flat_pos = patches.reshape(-1)
    slot_of = o["slot_of"]
    assert sorted(slot_of.tolist()) == list(range(8400))
    assert np.array_equal(o["ent_pos"][slot_of], flat_pos)
    assert np.all(np.diff(o["ent_pos"][:8400]) >= 0)
    folded = (w_mult.reshape(8400, 128) * np.tile(w_summer.reshape(4, 128), (2100, 1))) * np.float32(1 / 32)
    assert np.array_equal(o["ent_w"][slot_of], folded.astype(np.float32))

    # groups: cover every slot once, in order; one position per group; row / band consistent; band table monotone
    g = o["groups"]
    first, row, ne = g[:, 0], g[:, 1] & 31, g[:, 1] >> 8
    assert first[0] == 0 and np.array_equal(first[1:], first[:-1] + ne[:-1]) and first[-1] + ne[-1] == 8400
    assert ne.min() >= 1 and ne.max() <= GM
    bf = o["band_first"]
    assert bf[0] == 0 and bf[-1] == len(g) and np.all(np.diff(bf) >= 0)
    band_of_group = np.searchsorted(bf, np.arange(len(g)), side="right") - 1
    for i in range(len(g)):
        pos = o["ent_pos"][first[i]:first[i] + ne[i]]
        assert np.all(pos == pos[0]) and pos[0] == band_of_group[i] * R + row[i] and row[i] < R
    # a run of one position longer than 4 is split into consecutive groups, never merged across positions
    same = o["ent_pos"][first[1:]] == o["ent_pos"][first[:-1]]
    assert np.all(ne[:-1][same] == GM)

    # fragments -> weights: w[e][k] = (hi + lo) * unscale, channel mapping k0 = 64 kh + 16 ks + 2 tig, (k0, k0+1 | k0+8, k0+9)
    halves = _frag_halves(o["frag"][:8400])                      # [e][kh][ks][tig][word 4][half 2]
    w_rec = np.zeros((8400, 128), np.float64)
    for kh in range(2):
        for ks in range(4):
            for tig in range(4):
                k0 = 64 * kh + 16 * ks + 2 * tig
                hi_b0, hi_b1, lo_b0, lo_b1 = (halves[:, kh, ks, tig, j].astype(np.float64) for j in range(4))
                w_rec[:, [k0, k0 + 1]] = hi_b0 + lo_b0
                w_rec[:, [k0 + 8, k0 + 9]] = hi_b1 + lo_b1
    w_rec *= o["unscale"]
    ref = o["ent_w"][:8400].astype(np.float64)
    scale = np.abs(ref).max()
    assert np.abs(w_rec - ref).max() <= 2.0 ** -21 * scale        # hi + lo carry >= 21 bits of the largest weight
    big = np.abs(ref) >= scale * 2.0 ** -10
    assert np.abs(w_rec[big] / ref[big] - 1).max() <= 2.0 ** -20
    assert np.all(o["frag"][8400:] == 0)                          # padding slots

    # replay of wv_gather_kernel's gather on 8 windows of random activations (hi16 / lo16 planes of 32 * y)
    y = (rng.standard_normal((8, 5997, 128)) * 3).astype(np.float32) * np.float32(32)
    y_hi = y.astype(np.float16)
    y_lo = (y - y_hi.astype(np.float32)).astype(np.float16)
    for gi in rng.choice(len(g), size=min(64, len(g)), replace=False):
        e0, n_e = int(first[gi]), int(ne[gi])
        pos = int(o["ent_pos"][e0])
        a_hi, a_lo = y_hi[:, pos, :].astype(np.float64), y_lo[:, pos, :].astype(np.float64)
        got = np.zeros((8, n_e))
        for kh in range(2):
            for ks in range(4):
                for tig in range(4):
                    k0 = 64 * kh + 16 * ks + 2 * tig
                    ks4 = [k0, k0 + 1, k0 + 8, k0 + 9]
                    for t in range(n_e):
                        hh = halves[e0 + t, kh, ks, tig].astype(np.float64)          # [word][half]
                        b_hi = np.array([hh[0, 0], hh[0, 1], hh[1, 0], hh[1, 1]])    # column 2t   (hi weight half)
                        b_lo = np.array([hh[2, 0], hh[2, 1], hh[3, 0], hh[3, 1]])    # column 2t+1 (lo weight half)
                        got[:, t] += (a_hi[:, ks4] + a_lo[:, ks4]) @ (b_hi + b_lo)
        got *= o["unscale"]
        want = (y[:, pos, :].astype(np.float64)) @ ref[e0:e0 + n_e].T
        tol = 1e-6 * max(np.abs(want).max(), 1.0)
        assert np.abs(got - want).max() <= tol, (kind, gi, np.abs(got - want).max(), tol)


def test_integration_md_ctypes_stub(repo_root, weights_npz):
    """The reference-side binding shown in INTEGRATION.md (level 2) is executable as printed: it binds libgnm.so, fills
    gnm_weights through genomad_b200.weights, and -- on a box without a GPU -- gnm_create fails loudly through
    gnm_last_error (there is no CPU fallback); with a GPU it classifies."""
    import torch
    text = (repo_root / "INTEGRATION.md").read_text()
    block = text[text.index("```python\nimport ctypes as C, numpy as np"):]
    block = block[len("```python\n"):block.index("\n```")]
    assert "class GnmModel" in block and "gnm_classify_host" in block
    block = block.replace('C.CDLL("libgnm.so")', f'C.CDLL({str(repo_root / "genomad_b200" / "libgnm.so")!r})')
    ns = {}
    exec(compile(block, "INTEGRATION.md", "exec"), ns)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            ns["GnmModel"](weights_npz, 8)
    else:
        m = ns["GnmModel"](weights_npz, 8)
        p = m.predict(np.full((2, 6000), ord("A"), np.uint8))
        assert p.shape == (2, 3) and np.allclose(p.sum(1), 1, atol=1e-5)


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(engine.GnmError):
        engine.Classifier()
    # C ABI level: create must fail loudly without a device
    lib = engine.load_library()
    w = weights.load_weights()
    cw = weights.to_c_struct(w, engine._Weights, engine._IglooW, engine._BnW)
    h = ctypes.c_void_p()
    assert lib.gnm_create(0, ctypes.byref(cw), 8, ctypes.byref(h)) != 0
    assert b"no CUDA device" in lib.gnm_last_error() or b"CUDA" in lib.gnm_last_error()


# ------------------------------------------------------------------------------------------ module driver
class _StubClassifier:
    """Deterministic stand-in (hash of the window bytes) so the driver's plumbing can run without a GPU."""
    device = 0
    calls = 0

    def classify_host(self, windows):
        _StubClassifier.calls += 1
        s = windows.astype(np.float64).sum(axis=1)
        p = np.stack([np.sin(s) ** 2, np.cos(s) ** 2 * 0.5, np.cos(s) ** 2 * 0.5], axis=1)
        return p.astype(np.float32)


@pytest.fixture
def stub_driver(monkeypatch):
    _StubClassifier.calls = 0
    monkeypatch.setattr(nn_classification, "_make_classifier", lambda batch_size, device: _StubClassifier())

    def fake_classify(clf, parsed, offsets, info, contig_reduce="gather"):
        windows = parsed.export_windows(0, parsed.n_windows, np.zeros((max(1, parsed.n_windows), 6000), np.uint8))
        return T.segment_mean(clf.classify_host(windows), np.repeat(np.arange(len(offsets) - 1), np.diff(offsets)),
                              len(offsets) - 1)
    monkeypatch.setattr(nn_classification, "_classify_parsed", fake_classify)
    return _StubClassifier


def _write_fasta(path, n=5, seed=0):
    rng = np.random.default_rng(seed)
    with open(path, "w") as fh:
        for i in range(n):
            s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 10000)].tobytes().decode()
            fh.write(f">contig_{i:03d} d\n")
            for k in range(0, len(s), 60):
                fh.write(s[k:k + 60] + "\n")


def test_main_output_surface_and_restart(tmp_path, stub_driver, capsys):
    fa = tmp_path / "sample.fna"
    _write_fasta(fa)
    out = tmp_path / "out"
    nn_classification.main(fa, out, False, 128, False, 4, True, False)
    o = _paths.NNOutputs("sample", out)
    assert o.nn_classification_log.exists() and o.nn_classification_execution_info.exists()
    info = json.loads(o.nn_classification_execution_info.read_text())
    assert set(info) == {"module", "input", "input_md5", "start_time", "parameters"}
    assert info["module"] == "nn_classification" and info["parameters"] == {"single_window": False}
    assert info["input_md5"] == utils.get_md5(fa) and info["input"] == "sample.fna"
    z = np.load(o.nn_classification_npz_output)
    assert set(z.files) == {"contig_names", "predictions"}
    assert z["predictions"].dtype == np.float32 and z["predictions"].shape == (5, 3)
    assert list(z["contig_names"]) == [f"contig_{i:03d}" for i in range(5)]
    ids = np.load(o.seq_window_id_output)
    assert set(ids.files) == {"contig_names", "contig_ids"} and ids["contig_ids"].tolist() == [0, 0, 1, 1, 2, 2, 3, 3, 4, 4]
    lines = o.nn_classification_output.read_text().splitlines()
    assert lines[0] == "seq_name\tchromosome_score\tplasmid_score\tvirus_score"
    for name, row, line in zip(z["contig_names"], z["predictions"], lines[1:]):
        assert line == f"{name}\t" + "\t".join(f"{x:.4f}" for x in row)      # format(np.float32, '.4f'), as the reference
    assert "finished" in o.nn_classification_log.read_text()
    # second run: everything is skipped
    calls = stub_driver.calls
    nn_classification.main(fa, out, False, 128, False, 4, False, False)
    assert stub_driver.calls == calls
    assert "Skipping sequence classification" in o.nn_classification_log.read_text()
    # --restart recomputes; changed parameters recompute; --cleanup removes the encoded dir
    nn_classification.main(fa, out, False, 128, True, 4, False, False)
    assert stub_driver.calls == calls + 1
    nn_classification.main(fa, out, True, 128, False, 4, False, True)
    assert stub_driver.calls == calls + 2
    assert not o.encoded_sequences_dir.exists()
    assert np.load(o.nn_classification_npz_output)["predictions"].shape == (5, 3)


def test_main_errors_exit_1(tmp_path, stub_driver):
    dup = tmp_path / "dup.fna"
    dup.write_text(">a\nACGT\n>a\nACGT\n")
    with pytest.raises(SystemExit) as e:
        nn_classification.main(dup, tmp_path / "o1", False, 128, False, 1, False, False)
    assert e.value.code == 1
    empty = tmp_path / "empty.fna"
    empty.write_text("")
    with pytest.raises(SystemExit) as e:
        nn_classification.main(empty, tmp_path / "o2", False, 128, False, 1, False, False)
    assert e.value.code == 1
    only_n = tmp_path / "n.fna"
    only_n.write_text(">a\nNNNN\n")
    with pytest.raises(SystemExit) as e:
        nn_classification.main(only_n, tmp_path / "o3", False, 128, False, 1, False, False)
    assert e.value.code == 1


def test_main_compressed_prefix_and_provirus_twin(tmp_path, stub_driver):
    fa = tmp_path / "s.fna"
    _write_fasta(fa, n=2)
    gz = tmp_path / "sample2.fna.gz"
    gz.write_bytes(gzip.compress(fa.read_bytes()))
    out = tmp_path / "out"
    out.mkdir()
    o = _paths.NNOutputs("sample2", out)
    # fake a finished find-proviruses run on the same input
    o.find_proviruses_dir.mkdir()
    utils.write_execution_info("find_proviruses", gz, {}, o.find_proviruses_execution_info)
    o.find_proviruses_output.write_text("seq_name\tx\ncontig_000|provirus_1_5000\t1\n")
    o.find_proviruses_nucleotide_output.write_text(">contig_000|provirus_1_5000\n" + "ACGT" * 1250 + "\n")
    o.find_proviruses_proteins_output.write_text("")
    o.find_proviruses_genes_output.write_text("")
    nn_classification.main(gz, out, False, 64, False, 1, False, False)
    assert o.nn_classification_npz_output.exists()
    z = np.load(o.provirus_nn_classification_npz_output)
    assert set(z.files) == {"provirus_names", "predictions"} and z["predictions"].shape == (1, 3)
    assert set(np.load(o.provirus_window_id_output).files) == {"provirus_names", "provirus_ids"}
    assert o.provirus_nn_classification_output.read_text().splitlines()[1].startswith("contig_000|provirus_1_5000\t")


def test_cli_options_match_reference():
    from click.testing import CliRunner
    from genomad_b200 import cli
    r = CliRunner().invoke(cli.cli, ["nn-classification", "--help"])
    assert r.exit_code == 0
    for opt in ("--restart", "--threads", "-t", "--verbose", "--quiet", "-v", "-q", "--cleanup", "--single-window",
                "--batch-size", "INPUT", "OUTPUT"):
        assert opt in r.output, opt


# ------------------------------------------------------------------------------------------ native FASTA reader
def test_native_fasta_matches_reference_golden(enc, tmp_path):
    """csrc/fasta.cpp against the records the REAL reference reader produced (incl. CRLF, junk before '>', empty records)."""
    for name, case in enc["fasta"].items():
        p = tmp_path / f"{name}.fna"
        p.write_text(case["text"], newline="")
        pf = sequence.ParsedFasta(p)
        e = pf.encode()
        want = [(r[1], r[2]) for r in case["records"]]
        assert list(e.names) == [w[0] for w in want], name
        assert pf.check() == case["check_fasta"], name
        got_first = [bytes(e.windows[e.offsets[i]]).rstrip(b"N")[:len(w[1])] for i, w in enumerate(want)]
        for g, w in zip(got_first, want):
            stripped = w[1].upper()[:6000].rstrip("N").encode()
            assert g[:len(stripped)] == stripped, name


def test_native_fasta_equals_python_statement_and_oracle(enc, tmp_path):
    rng = np.random.default_rng(8)
    recs = []
    for i, ln in enumerate([10000, 400, 2499, 2500, 14500, 6000, 30000, 8499, 1, 12000]):
        s = np.frombuffer(b"ACGTNacgtnRY-", np.uint8)[rng.choice(13, ln, p=[.2, .2, .2, .2, .04, .03, .03, .03, .03, .01, .01, .01, .01])]
        width = int(rng.integers(20, 90))
        recs.append(f">c{i}\tdesc {i}\n" + "\n".join(s.tobytes().decode()[k:k + width] for k in range(0, ln, width)))
    for case in enc["nrule"]:
        recs.append(f">{case['name']}\n{case['raw']}")
    recs.append(">only_n\nNNNNnnnn")
    recs.append(">empty")
    text = "leading junk\n" + "\n".join(recs) + "\n"
    for eol in ("\n", "\r\n", "\r"):
        p = tmp_path / "mix.fna"
        p.write_text(text.replace("\n", eol), newline="")
        for single in (False, True):
            a = sequence.encode_fasta(p, single_window=single)            # native
            b = sequence.encode_fasta_py(p, single_window=single)         # python statement
            names, ids, ascii_arr, _ = T.encode_fasta(p, single_window=single)   # oracle (reference transcription)
            for x in (b,):
                assert list(a.names) == list(x.names) and np.array_equal(a.offsets, x.offsets)
                assert np.array_equal(a.contig_ids, x.contig_ids) and np.array_equal(a.windows, x.windows)
            assert list(a.names) == list(names) and np.array_equal(a.contig_ids, ids) and np.array_equal(a.windows, ascii_arr)
    for case in enc["nrule"]:
        q = tmp_path / "n.fna"
        q.write_text(f">x\n{case['raw']}\n")
        assert sequence.ParsedFasta(q).n_windows == len(case["kept"]), case["name"]


def test_native_fasta_check_and_gzip(tmp_path):
    d = tmp_path / "dup.fna"
    d.write_text(">a 1\nACGT\n>a 2\nGGGG\n")
    assert not sequence.ParsedFasta(d).check() and not sequence.check_fasta(d)
    e = tmp_path / "empty.fna"
    e.write_text("no header here\n")
    pf = sequence.ParsedFasta(e)
    assert not pf.check() and pf.n_windows == 0 and pf.encode().windows.shape == (0, 6000)
    g = tmp_path / "z.fna.gz"
    with gzip.open(g, "wt") as fh:
        fh.write(">k x\nnnACGTacgtNN\n")
    enc_ = sequence.encode_fasta(g)
    assert list(enc_.names) == ["k"] and bytes(enc_.windows[0][:8]) == b"ACGTACGT" and enc_.windows[0][8] == ord("N")
    out = np.zeros((4, 6000), np.uint8)
    enc2 = sequence.ParsedFasta(g).encode(out)
    assert enc2.windows.base is out or np.shares_memory(enc2.windows, out)


def test_native_fasta_property_random_texts(tmp_path):
    """Property test: random FASTA-like texts (odd line breaks, N runs, lower case, junk, '>' inside lines) -- the native
    reader, the Python statement and the oracle's transcription of the reference reader must agree exactly."""
    from hypothesis import given, settings, strategies as st

    alphabet = "ACGTNnacgtRY>- \t"
    line = st.text(alphabet=alphabet, min_size=0, max_size=90)
    rec = st.tuples(st.text(alphabet="abcXYZ_01 \t|", min_size=1, max_size=12), st.lists(line, min_size=0, max_size=6),
                    st.integers(0, 3))
    texts = st.tuples(st.lists(line, max_size=2), st.lists(rec, min_size=0, max_size=6), st.sampled_from(["\n", "\r\n", "\r"]))

    @settings(max_examples=150, deadline=None)
    @given(texts)
    def check(t):
        junk, recs, eol = t
        parts = [ln.lstrip(">") for ln in junk]
        for name, lines, big in recs:
            if not name.split():
                name = "x" + name
            parts.append(">" + name)
            parts += [ln.lstrip(">") for ln in lines]          # a body line starting with '>' would be a header
            if big:
                parts.append("ACGTNACGT" * (300 * big))       # enough sequence for several windows sometimes
        text = eol.join(parts) + (eol if parts else "")
        p = tmp_path / "h.fna"
        p.write_text(text, newline="")
        a = sequence.encode_fasta(p)
        b = sequence.encode_fasta_py(p)
        names, ids, ascii_arr, _ = T.encode_fasta(p)
        assert list(a.names) == list(b.names) == list(names)
        assert np.array_equal(a.offsets, b.offsets) and np.array_equal(a.contig_ids, ids)
        assert np.array_equal(a.windows, b.windows) and np.array_equal(a.windows, ascii_arr)
        pf = sequence.ParsedFasta(p)
        assert pf.check() == sequence.check_fasta(p)

    check()


def test_tf32_three_pass_split_error_level():
    """The tensor-core logits GEMM (csrc/logits_tc.cuh) multiplies TF32 halves: x = hi + lo with the low 13 mantissa bits of
    both cleared, D = Ahi*Bhi + Alo*Bhi + Ahi*Blo.  NumPy emulation of exactly that split on a [64 x 2100] x [2100 x 749]
    product: the error against float64 must stay at fp32-GEMM level (the plain fp32 product is the yardstick), including
    for the ~1e-32 magnitudes of the shipped patch weights (TF32 keeps fp32's exponent range)."""
    rng = np.random.default_rng(3)

    def split(x):
        x = x.astype(np.float32)
        hi = (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
        lo = ((x - hi).astype(np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
        return hi.astype(np.float64), lo.astype(np.float64)

    for scale_a, scale_b in ((1.0, 1.0), (50.0, 1e-3), (1e-31, 1e-31 * 1e25)):
        a = (rng.standard_normal((64, 2100)) * scale_a).astype(np.float32)
        b = (rng.standard_normal((2100, 749)) * scale_b).astype(np.float32)
        exact = a.astype(np.float64) @ b.astype(np.float64)
        ah, al = split(a)
        bh, bl = split(b)
        tc = ah @ bh + al @ bh + ah @ bl                       # products and sums in float64: isolates the split error
        fp32 = (a @ b).astype(np.float64)
        denom = np.abs(a).astype(np.float64) @ np.abs(b).astype(np.float64)
        err_tc = (np.abs(tc - exact) / denom).max()
        err_32 = (np.abs(fp32 - exact) / denom).max()
        assert err_tc < 4e-6, (scale_a, scale_b, err_tc)       # 2^-20 + 2^-20 per product, before fp32 accumulation
        assert err_tc < 40 * max(err_32, 1e-7)


def test_native_fasta_streaming_block_export(tmp_path):
    """Index-then-stream: any block of the global window list, in any order and with any thread count, equals the same rows
    of the one-shot export -- for wrapped, single-line and ragged records, records that lose windows to the N rule, and
    after gnm_fasta_release_before dropped the pages behind the cursor (they are re-read from the page cache)."""
    rng = np.random.default_rng(11)
    recs = []
    for i, (ln, width) in enumerate([(61000, 60), (150000, 0), (7000, 80), (30011, 70), (45000, -1), (2600, 50), (90000, 61)]):
        s = np.frombuffer(b"ACGTacgtN", np.uint8)[rng.choice(9, ln, p=[.23, .23, .23, .23, .02, .02, .01, .01, .02])].copy()
        if i == 3:
            s[6000:10500] = ord("N")                       # window 1 is dropped (> 4000 N), later windows are kept
        t = s.tobytes().decode()
        if width == 0:
            body = t                                        # one line
        elif width < 0:                                     # ragged line lengths
            cuts = np.cumsum(rng.integers(1, 200, 2000)); cuts = cuts[cuts < ln]
            body = "\n".join(t[a:b] for a, b in zip(np.r_[0, cuts], np.r_[cuts, ln]))
        else:
            body = "\n".join(t[k:k + width] for k in range(0, ln, width))
        recs.append(f">r{i} w={width}\n{body}\n")
    p = tmp_path / "stream.fna"
    p.write_text("".join(recs))
    ref = sequence.encode_fasta_py(p)
    pf = sequence.ParsedFasta(p, threads=3)
    full = pf.encode()
    assert np.array_equal(full.windows, ref.windows) and np.array_equal(full.offsets, ref.offsets)
    n = pf.n_windows
    assert n == ref.windows.shape[0] > 60
    buf = np.zeros((17, 6000), np.uint8)
    for first in list(rng.permutation(n))[:40] + [0, n - 1, n]:
        cnt = int(min(rng.integers(0, 18), n - first))
        got = pf.export_windows(int(first), cnt, buf)
        assert np.array_equal(got, ref.windows[first:first + cnt])
    pf.release_before(n // 2)
    pf.release_before(n)
    assert np.array_equal(pf.export_windows(0, 5, buf), ref.windows[:5])
    pf.close()


def test_bench_synthetic_fasta_and_stream_helpers(tmp_path):
    """bench.py's synthetic inputs: the FASTA writer's window arithmetic agrees with the reader (configs 1 and 4 shapes in
    miniature), and the counter-based window stream is a pure function of (seed, index) on NumPy and on torch alike."""
    import importlib.util
    import torch
    from pathlib import Path as _P
    spec = importlib.util.spec_from_file_location("bench_mod", _P(__file__).resolve().parents[1] / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from genomad_b200 import synth
    for n_contigs, ln, exact in ((7, 10_000, True), (3, 100_000, False), (5, 8_499, False), (2, 2_000, True)):
        fa = tmp_path / f"b_{ln}.fna"
        bench.write_fasta(fa, n_contigs, ln, seed=0, exact_rng=exact)
        pf = sequence.ParsedFasta(fa)
        assert pf.check() and pf.n_contigs == n_contigs and pf.n_windows == bench.count_windows(ln, n_contigs)
        assert list(pf.index().names) == [f"contig_{i:03d}" for i in range(n_contigs)]
        pf.close()
    idx = np.array([0, 1, 999_999, 123_456])
    a = synth.windows_numpy(idx, seed=1)
    assert a.shape == (4, 6000) and set(np.unique(a)) <= set(b"ACGTNR")
    assert np.array_equal(a[3], synth.windows_numpy([123_456], seed=1)[0])             # pure function of the index
    assert not np.array_equal(a[0], synth.windows_numpy([0], seed=2)[0])               # ... and of the seed
    t = synth.windows_torch(123_455, 3, 1, "cpu").numpy()
    assert np.array_equal(t, synth.windows_numpy(np.arange(123_455, 123_458), seed=1))
    sub = synth.subsample_indices(256, 100_000, seed=1)
    assert len(sub) == 256 == len(set(sub.tolist())) and np.all(np.diff(sub) > 0)
    assert (synth.windows_numpy(sub, seed=1) == ord("N")).any(1).sum() >= 4                # the dirty sub-stream is represented


def _bgzf(data: bytes, block: int = 65280) -> bytes:
    """BGZF (bgzip) container: independent gzip members with a 'BC' extra field carrying the block size, plus the empty EOF block."""
    import struct
    import zlib
    out = bytearray()
    for i in list(range(0, len(data), block)) + [None]:
        chunk = b"" if i is None else data[i:i + block]
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        bsize = 18 + len(comp) + 8
        out += b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1)
        out += comp + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk))
    return bytes(out)


def test_native_gzip_and_bgzf_inputs(tmp_path):
    """gzip input is inflated natively (csrc/fasta.cpp: gnm_fasta_open_gz): single member, concatenated members and BGZF
    (block-parallel) must give exactly the windows of the plain file; a truncated stream is an error, not a short read."""
    rng = np.random.default_rng(31)
    recs = []
    for i, ln in enumerate([30000, 6100, 250000, 2600, 9000]):
        t = np.frombuffer(b"ACGTacgtN", np.uint8)[rng.choice(9, ln, p=[.23, .23, .23, .23, .02, .02, .01, .01, .02])].tobytes().decode()
        recs.append(f">g{i} x\n" + "\n".join(t[k:k + 60] for k in range(0, ln, 60)) + "\n")
    text = "".join(recs).encode()
    plain = tmp_path / "p.fna"
    plain.write_bytes(text)
    ref = sequence.encode_fasta(plain)
    cut = len(recs[0]) + len(recs[1]) + 1000                      # member boundary in the middle of a record
    variants = {"single.fna.gz": gzip.compress(text), "multi.fna.gz": gzip.compress(text[:cut]) + gzip.compress(text[cut:]),
                "bgzf.fna.gz": _bgzf(text), "bgzf_small.fna.gz": _bgzf(text, block=4096)}
    for name, blob in variants.items():
        p = tmp_path / name
        p.write_bytes(blob)
        assert gzip.decompress(blob) == text, name                 # the fixtures are valid gzip for any reader
        for th in (1, 5):
            pf = sequence.ParsedFasta(p, threads=th)
            assert pf._text is None                                 # native path, not Python's gzip
            e = pf.encode()
            assert list(e.names) == list(ref.names) and np.array_equal(e.offsets, ref.offsets), name
            assert np.array_equal(e.windows, ref.windows), name
            pf.close()
    bad = tmp_path / "trunc.fna.gz"
    bad.write_bytes(gzip.compress(text)[:-200])
    with pytest.raises(RuntimeError):
        sequence.ParsedFasta(bad)
