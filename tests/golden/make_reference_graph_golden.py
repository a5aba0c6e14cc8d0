#!/usr/bin/env python
"""
Golden vectors from THE REFERENCE'S OWN MODEL DEFINITION: /root/reference/genomad/neural_network/{model,igloo}.py are imported by
file path and executed (create_classifier() -> load_weights(nn_classifier.h5) -> predict) on top of tests/golden/keras_shim.py, a
NumPy stand-in for the TensorFlow / Keras calls those two files make (neither library exists in this image).  What the vectors pin
is the graph the reference builds -- layer sequence, weight shapes and names, the gather_nd / transpose / reshape chain of the IGLOO
layer, pooling, softmax axes, how the H5 datasets map to layers --, i.e. everything oracle/igloo_model.py had restated by hand; what
they do not pin is TensorFlow's own fp32 arithmetic.

    python tests/golden/make_reference_graph_golden.py     # needs /root/reference; ~2 min -> tests/golden/reference_graph_golden.npz
    python tests/golden/make_reference_graph_golden.py --rerun     # a second, independent build -> reference_graph_rerun.npz

Stored: token batch (24 windows: 16 of the counter stream incl. N / IUPAC windows + 8 worst-case families), the reference graph's
probabilities in fp32 and in fp64 arithmetic, with the shipped weights and with synthetic O(1) IGLOO weights (assigned to the
reference layers' variables), per-layer
taps of window 0 (conv outputs, IGLOO outputs) and the file-dataset -> layer/variable assignment the loader made.
"""
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
REF = Path("/root/reference/genomad")
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import keras_shim  # noqa: E402


def load_reference_model_module():
    keras_shim.install()
    pkg = types.ModuleType("genomad")
    pkg.__path__ = [str(REF)]
    sub = types.ModuleType("genomad.neural_network")
    sub.__path__ = [str(REF / "neural_network")]
    sys.modules["genomad"], sys.modules["genomad.neural_network"] = pkg, sub
    mods = {}
    for name in ("igloo", "model"):
        spec = importlib.util.spec_from_file_location(f"genomad.neural_network.{name}", REF / "neural_network" / f"{name}.py")
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"genomad.neural_network.{name}"] = mod
        setattr(sub, name, mod)
        spec.loader.exec_module(mod)
        mods[name] = mod
    pkg.neural_network = sub
    return mods["model"], mods["igloo"]


def igloo_layers(clf, igloo_mod):
    enc = [l for l in clf.layers if isinstance(l, keras_shim.Model)][0]
    return enc, [l for l in enc.layers if isinstance(l, igloo_mod.IGLOO1D_kernel)]


def set_synthetic(clf, igloo_mod, wsyn):
    """Assign oracle.igloo_model.synthetic_igloo_weights to the reference layers' variables (IGLOO kernel s <-> keys ig{s}_*)."""
    _, kernels = igloo_layers(clf, igloo_mod)
    assert [k.name for k in kernels] == ["igloo1d_kernel", "igloo1d_kernel_1"]
    for s, k in enumerate(kernels):
        for v in k._vars:
            arr = wsyn[f"ig{s}_{v.name}"]
            assert tuple(arr.shape) == tuple(v.shape), (v.name, arr.shape, v.shape)
            v.value = np.ascontiguousarray(arr)


def main():
    from genomad_b200 import synth
    from oracle import igloo_model as M, tokenizer as T
    import precision_study
    np.random.seed(0)                                          # the reference draws random patches at build time (then overwritten)
    model_mod, igloo_mod = load_reference_model_module()
    clf = model_mod.create_classifier()
    clf.load_weights(REF / "data" / "nn_classifier.h5")
    idx = synth.subsample_indices(2048, 1_000_000, seed=1)
    a_all = synth.windows_numpy(idx, seed=1)
    dirty = np.flatnonzero((a_all == ord("N")).any(1))[:4]
    clean = np.flatnonzero(~(a_all == ord("N")).any(1))[:12]
    pick = np.concatenate([clean, dirty])
    a = np.concatenate([a_all[pick], precision_study.make_windows(8, seed=101)])
    tok = T.tokenize_windows(a).astype(np.int64)
    p_shipped = clf.predict(tok, batch_size=8)
    keras_shim.set_float(np.float64)
    p_shipped64 = clf.predict(tok, batch_size=8)
    keras_shim.set_float(np.float32)

    # per-layer taps of window 0 through the reference graph (encoder internals)
    enc, kernels = igloo_layers(clf, igloo_mod)
    taps = {}
    x = tok[:1]
    for lay in enc.layers[1:]:
        if isinstance(lay, keras_shim.Concatenate):
            break
        if isinstance(lay, igloo_mod.IGLOO1D_kernel):
            taps[f"{lay.name}_out"] = lay._run(x)
            continue
        x = lay._run(x)
        if isinstance(lay, keras_shim.LeakyReLU):
            taps[f"act_after_{lay.name}"] = x[:, ::499, :8].copy()      # thin slice of the activation

    w = M.load_npz_weights(ROOT / "genomad_b200" / "data" / "nn_classifier.npz")
    wsyn = M.synthetic_igloo_weights(w)
    set_synthetic(clf, igloo_mod, wsyn)
    p_syn = clf.predict(tok, batch_size=8)
    keras_shim.set_float(np.float64)
    p_syn64 = clf.predict(tok, batch_size=8)
    keras_shim.set_float(np.float32)
    report = np.array([f"{a} -> {b} {c} {d}" for a, b, c, d in clf.load_report])
    out = ROOT / "tests" / "golden" / "reference_graph_golden.npz"
    np.savez_compressed(out, windows=a, tokens=tok.astype(np.uint16), shipped=p_shipped, synthetic=p_syn, shipped_fp64=p_shipped64, synthetic_fp64=p_syn64,
                        load_report=report,
                        layer_names=np.array([l.name for l in enc.layers] + ["|"] + [l.name for l in clf.layers]),
                        **{f"tap_{k}": v for k, v in taps.items()})
    # immediate cross-check against the oracle (the test repeats it from the stored file)
    o_shipped = np.concatenate([M.forward(tok[i:i + 8], w) for i in range(0, len(tok), 8)])
    o_syn = np.concatenate([M.forward(tok[i:i + 8], wsyn) for i in range(0, len(tok), 8)])
    import torch
    o_shipped64 = np.concatenate([M.forward(tok[i:i + 8], w, torch.float64) for i in range(0, len(tok), 8)])
    o_syn64 = np.concatenate([M.forward(tok[i:i + 8], wsyn, torch.float64) for i in range(0, len(tok), 8)])
    print("reference graph vs oracle, fp32: shipped max |dp| %.3e, synthetic IGLOO weights max |dp| %.3e" %
          (np.abs(o_shipped - p_shipped).max(), np.abs(o_syn - p_syn).max()))
    print("reference graph vs oracle, fp64: shipped max |dp| %.3e, synthetic IGLOO weights max |dp| %.3e" %
          (np.abs(o_shipped64 - p_shipped64).max(), np.abs(o_syn64 - p_syn64).max()))
    print("layers:", [l.name for l in enc.layers])
    print("wrote", out)


def rerun():
    """Rebuild the reference graph from its source and re-predict three windows of the committed fixture, with the loader's
    dataset -> variable assignment, into reference_graph_rerun.npz (tests/test_oracle_golden.py compares the fixture with it)."""
    np.random.seed(0)
    model_mod, _ = load_reference_model_module()
    clf = model_mod.create_classifier()
    clf.load_weights(REF / "data" / "nn_classifier.h5")
    g = np.load(ROOT / "tests" / "golden" / "reference_graph_golden.npz")
    pick = np.array([0, 13, 20])
    p = clf.predict(g["tokens"][pick].astype(np.int64), batch_size=3)
    report = np.array([f"{a} -> {b} {c} {d}" for a, b, c, d in clf.load_report])
    out = ROOT / "tests" / "golden" / "reference_graph_rerun.npz"
    np.savez_compressed(out, pick=pick, shipped=p, load_report=report)
    print("wrote", out)


if __name__ == "__main__":
    rerun() if "--rerun" in sys.argv else main()
