"""CPU tests: the oracle against golden vectors made by the real reference code (tests/golden/make_golden.py)."""
import hashlib
import json

import numpy as np
import pytest
import torch

from oracle import igloo_model as M
from oracle import tokenizer as T


@pytest.fixture(scope="module")
def enc(golden_dir):
    return json.loads((golden_dir / "encoder_golden.json").read_text())


def test_tokenizer_literal_matches_reference(enc):
    for case in enc["tokenize"]:
        assert T.tokenize_dna_literal(case["seq"].encode("ascii")) == case["tokens"], case["seq"]


def test_survey_kat():
    assert T.tokenize_dna_literal(b"ACGTNACGTACGTTTTT") == [28, 0, 0, 0, 0, 28, 109, 178, 199, 28, 112, 192, 256, 256]


def test_tokenizer_closed_form_matches_reference_batch(enc, golden_dir):
    ref = np.load(golden_dir / "encoder_batch_tokens.npz")["tokens"]
    raws = enc["batch"]["raw"]
    a = np.frombuffer(b"".join(r.upper().encode("ascii").ljust(6000, b"N") for r in raws), np.uint8).reshape(-1, 6000)
    tok = T.tokenize_windows(a)
    assert tok.dtype == np.uint16 and tok.shape == (len(raws), 5997)
    assert np.array_equal(tok, ref)
    assert hashlib.sha256(tok.tobytes()).hexdigest() == enc["batch"]["tokens_sha256"]
    # literal loop agrees too (a few rows; it is slow)
    for i in (0, 1, 5):
        assert T.tokenize_dna_literal(a[i].tobytes()) == ref[i].tolist()


def test_c_oracle_tokenizer_and_window_rules(enc, golden_dir):
    """oracle/tokenizer_c.c (plain C, built with gcc) against the vectors made by the real reference code, and against the NumPy
    closed form: adversarial strings of any length, the seeded batch, and the reference module's own encoding-stage tokens."""
    from oracle import build_c as OC
    for case in enc["tokenize"]:
        assert OC.tokenize(case["seq"].encode("ascii")) == case["tokens"], case["seq"]
    ref = np.load(golden_dir / "encoder_batch_tokens.npz")["tokens"]
    raws = enc["batch"]["raw"]
    a = np.frombuffer(b"".join(r.upper().encode("ascii").ljust(6000, b"N") for r in raws), np.uint8).reshape(-1, 6000)
    assert np.array_equal(OC.tokenize_windows(a), ref)
    rng = np.random.default_rng(9)
    r = np.frombuffer(b"ACGTNRacgtn-", np.uint8)[rng.integers(0, 12, (64, 6000))]
    assert np.array_equal(OC.tokenize_windows(r), T.tokenize_windows(r))
    # FASTA -> windows -> tokens of the reference module run (N rule, short tail, lower case, IUPAC), both window modes
    toks = np.load(golden_dir / "reference_module" / "run_default" / "encoded_tokens.npz")
    ids = np.load(golden_dir / "reference_module" / "run_default" / "toy_seq_window_id.npz")["contig_ids"]
    for single in (False, True):
        wins, got_ids = [], []
        for cid, (_, seq) in enumerate(T.read_fasta(golden_dir / "reference_module" / "input" / "toy.fna", strip_n=True)):
            raw = seq.encode("ascii")
            starts, lengths = OC.window_plan(raw, single)
            py = [w for n, w in enumerate(T.seq_windows(seq, max_windows=1 if single else None)) if not (n > 0 and w.count("N") > 4000)]
            assert [raw[s:s + l].decode() for s, l in zip(starts, lengths)] == py
            for s, l in zip(starts, lengths):
                wins.append(raw[s:s + l].upper().ljust(6000, b"N"))
                got_ids.append(cid)
        arr = np.frombuffer(b"".join(wins), np.uint8).reshape(-1, 6000)
        if single:
            first = np.concatenate([[0], np.flatnonzero(np.diff(ids)) + 1])
            assert np.array_equal(OC.tokenize_windows(arr), toks["sequences"][first])
        else:
            assert got_ids == ids.tolist() and np.array_equal(OC.tokenize_windows(arr), toks["sequences"])


def test_c_oracle_matches_literal_loop_on_random_strings():
    """Property check: the C tokenizer == the literal transcription of the reference loop, for strings of any length
    (0 .. 40; the Python-slice corner below 4 bases included) over an alphabet with invalid and lower-case bytes."""
    from hypothesis import given, settings, strategies as st
    from oracle import build_c as OC

    @settings(max_examples=400, deadline=None)
    @given(st.text(alphabet="ACGTNacgtR-", min_size=0, max_size=40))
    def check(sq):
        b = sq.encode("ascii")
        assert OC.tokenize(b) == T.tokenize_dna_literal(b)
    check()
    # window plan == the Python generator + N rule on structured random sequences
    rng = np.random.default_rng(4)
    for _ in range(60):
        n = int(rng.integers(1, 30000))
        sq = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes())
        for _ in range(int(rng.integers(0, 3))):                      # N runs, some longer than 4,000
            a = int(rng.integers(0, n)); ln = int(rng.integers(1, 7000))
            sq[a:a + ln] = b"N" * len(sq[a:a + ln])
        sq = bytes(sq).strip(b"N")
        if not sq:
            continue
        for single in (False, True):
            starts, lengths = OC.window_plan(sq, single)
            s = sq.decode()
            py = [w for k, w in enumerate(T.seq_windows(s, max_windows=1 if single else None)) if not (k > 0 and w.count("N") > 4000)]
            assert [s[a:a + l] for a, l in zip(starts, lengths)] == py


def test_seq_windows_lengths(enc):
    for case in enc["windows"]:
        s = "A" * case["len"]
        assert [len(w) for w in T.seq_windows(s)] == case["multi"]
        assert [len(w) for w in T.seq_windows(s, max_windows=1)] == case["single"]


def test_n_rule(enc, tmp_path):
    for case in enc["nrule"]:
        p = tmp_path / "x.fna"
        p.write_text(f">x\n{case['raw']}\n")
        names, ids, ascii_arr, tok = T.encode_fasta(p)
        assert len(ids) == len(case["kept"]), case["name"]


def test_read_fasta_quirks(enc, tmp_path):
    for name, case in enc["fasta"].items():
        p = tmp_path / f"{name}.fna"
        p.write_text(case["text"], newline="")
        got = [[h, T.accession(h), s] for h, s in T.read_fasta(p)]
        assert got == [list(r) for r in case["records"]], name


def test_model_frozen_vectors(golden_dir, weights_npz):
    g = np.load(golden_dir / "model_golden.npz")
    w = M.load_npz_weights(weights_npz)
    tok = T.tokenize_windows(g["ascii"])
    p = M.forward(tok[:6], w, torch.float64)
    assert np.abs(p - g["shipped_fp64"][:6]).max() < 1e-12
    # SURVEY Appendix C cross-check vectors (fp64), independently derived during the survey
    appendix_c = np.array([[0.00000000, 0.00011596, 0.99988404], [0.99973547, 0.00026453, 0.0],
                           [0.19144470, 0.05451930, 0.75403600], [0.96907142, 0.03092858, 0.0],
                           [0.05019702, 0.06085832, 0.88894466]])
    assert np.abs(p[:5] - appendix_c).max() < 5e-9


def test_two_formulations_agree(golden_dir, weights_npz):
    g = np.load(golden_dir / "model_golden.npz")
    w = M.load_npz_weights(weights_npz)
    tok = T.tokenize_windows(g["ascii"][2:6])
    for ww in (w, M.synthetic_igloo_weights(w)):
        a = M.forward(tok, ww, torch.float64)
        b = M.forward_as_written(tok, ww, torch.float64)
        assert np.abs(a - b).max() < 1e-12
        c = M.forward_as_written(tok, ww, torch.float32)
        assert np.abs(a - c).max() < 5e-5


def test_synthetic_weights_make_attention_live(golden_dir, weights_npz):
    g = np.load(golden_dir / "model_golden.npz")
    w = M.load_npz_weights(weights_npz)
    ws = M.synthetic_igloo_weights(w)
    tok = T.tokenize_windows(g["ascii"][4:6])
    _, parts = M.forward(tok, w, torch.float32, return_intermediates=True)
    assert float(parts["ig0"]["logits"].abs().max()) == 0.0  # shipped weights: attention is exactly uniform
    _, parts = M.forward(tok, ws, torch.float64, return_intermediates=True)
    assert float(parts["ig0"]["alpha"].max()) > 5.0 / 749    # synthetic weights: far from uniform


def test_oracle_model_matches_reference_graph(golden_dir, weights_npz):
    """The model oracle against vectors produced by the REFERENCE'S OWN model definition: genomad/neural_network/{model,igloo}.py
    imported by path and executed -- create_classifier(), load_weights(nn_classifier.h5), predict -- on a NumPy stand-in for the
    TensorFlow / Keras calls they make (tests/golden/keras_shim.py, generator make_reference_graph_golden.py; neither library
    exists in this image).  In fp64 the oracle and the reference graph must agree to rounding (structure: layer sequence, the
    gather_nd / transpose / reshape chain, pooling, softmax axes, dataset -> layer mapping), with the shipped weights AND with
    synthetic O(1) IGLOO weights (live gather / logits / softmax); in fp32 to summation-order noise.  TensorFlow's own fp32
    arithmetic is not pinned by this."""
    g = np.load(golden_dir / "reference_graph_golden.npz")
    tok = g["tokens"]
    assert tok.shape == (24, 5997) and np.array_equal(tok, T.tokenize_windows(g["windows"]))
    w = M.load_npz_weights(weights_npz)
    wsyn = M.synthetic_igloo_weights(w)
    # the loader of the reference graph consumed all 32 datasets of the file, each into the variable of the same name
    rep = [str(r) for r in g["load_report"]]
    assert len(rep) == 32 and len({r.split(" -> ")[1].split(" ")[0] for r in rep}) == 32
    assert "/model/igloo1d_kernel/random_patches:0 -> igloo1d_kernel/random_patches (2100, 4, 1) int32" in rep
    assert "/dense_2/dense_2/kernel:0 -> dense_2/kernel (512, 3) float32" in rep
    # the encoder the reference builds: conv -> IGLOO#0 on conv1's output, two more convs -> IGLOO#1, concatenate, dense, BN, relu
    names = [str(n) for n in g["layer_names"]]
    enc = names[:names.index("|")]
    assert [n for n in enc if n.startswith(("conv1d", "igloo1d", "concat", "dense", "batch"))] == \
        ["conv1d", "igloo1d_kernel", "conv1d_1", "conv1d_2", "igloo1d_kernel_1", "concatenate", "dense", "batch_normalization"]
    for key, ww in (("shipped", w), ("synthetic", wsyn)):
        o64 = np.concatenate([M.forward(tok[i:i + 8], ww, torch.float64) for i in range(0, 24, 8)])
        o32 = np.concatenate([M.forward(tok[i:i + 8], ww, torch.float32) for i in range(0, 24, 8)])
        d64 = np.abs(o64 - g[key + "_fp64"]).max()
        d32 = np.abs(o32 - g[key]).max()
        assert d64 <= 1e-11, (key, d64)
        assert d32 <= 5e-5 and np.abs(o32 - g[key + "_fp64"]).max() <= 5e-5, (key, d32)
        assert np.array_equal(o32.argmax(1), g[key + "_fp64"].argmax(1))
    # live weights really exercise the attention: the synthetic probabilities differ from the shipped ones
    assert np.abs(g["synthetic_fp64"] - g["shipped_fp64"]).max() > 1e-3


def test_reference_graph_golden_is_reproducible(golden_dir):
    """The committed fixture against a second, independent build of the reference graph from its source that re-predicted three
    of its windows (tests/golden/reference_graph_rerun.npz, `make_reference_graph_golden.py --rerun`): the fixture must be what
    the committed generator produces."""
    g = np.load(golden_dir / "reference_graph_golden.npz")
    r = np.load(golden_dir / "reference_graph_rerun.npz")
    assert r["pick"].tolist() == [0, 13, 20]
    assert np.abs(r["shipped"] - g["shipped"][r["pick"]]).max() <= 1e-6
    assert [str(x) for x in g["load_report"]] == [str(x) for x in r["load_report"]]


def test_keras_stand_in_semantics():
    """Spot checks of tests/golden/keras_shim.py against hand-computed values of the Keras / TF definitions it follows."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
    import keras_shim as K
    saved = {k: sys.modules.get(k) for k in ("tensorflow", "keras", "keras.layers", "keras.regularizers")}
    try:
        tf, keras = K.install()
        kl = keras.layers
        # causal Conv1D: y[t] = b + sum_j x[t - (k-1) + j] W[j]
        c = kl.Conv1D(1, 3, padding="causal")
        x = np.arange(1, 6, dtype=np.float32).reshape(1, 5, 1)
        c._run(x)
        c.kernel.value = np.array([1, 10, 100], np.float32).reshape(3, 1, 1)
        c.bias.value = np.array([0.5], np.float32)
        assert np.allclose(c._run(x)[0, :, 0], [100.5, 210.5, 321.5, 432.5, 543.5])
        # gather_nd with index depth 1, MaxPool1D valid, softmax, one_hot, BN inference, LeakyReLU
        m = np.arange(24, dtype=np.float32).reshape(4, 3, 2)
        assert np.array_equal(tf.gather_nd(m, np.array([[[3], [0]]])), m[[3, 0]][None])
        assert np.array_equal(kl.MaxPool1D(pool_size=2)._run(np.array([[[1.], [5.], [2.], [3.], [9.]]]))[0, :, 0], [5., 3.])
        assert np.allclose(tf.nn.softmax(np.array([[0., np.log(3.)]], np.float32)), [[0.25, 0.75]])
        assert np.array_equal(tf.one_hot(np.array([[2, 0]]), depth=3), [[[0, 0, 1], [1, 0, 0]]])
        bn = kl.BatchNormalization()
        bn._run(np.zeros((1, 2), np.float32))
        bn.gamma.value, bn.beta.value = np.array([2., 1.], np.float32), np.array([0.5, 0.], np.float32)
        bn.moving_mean.value, bn.moving_variance.value = np.array([1., 0.], np.float32), np.array([0.003, 0.999], np.float32)
        assert np.allclose(bn._run(np.array([[3., 2.]], np.float32)), [[2 * 2 / np.sqrt(0.004) + 0.5, 2.0]], rtol=1e-6)
        assert np.allclose(kl.LeakyReLU(negative_slope=0.1)._run(np.array([[-2., 3.]], np.float32)), [[-0.2, 3.]])
        # default layer names follow creation order per class
        assert [kl.Dense(1).name, kl.Dense(1).name, kl.Conv1D(1, 1, padding="causal").name] == ["dense", "dense_1", "conv1d_1"]
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_segment_mean():
    p = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], np.float32)
    out = T.segment_mean(p, np.array([0, 0, 2, 2]))
    assert out.shape == (3, 3)
    assert np.allclose(out, [[.5, .5, 0], [0, 0, 0], [.5, .5, 1]])
