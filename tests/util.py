"""Shared helpers for the parity tests: run the same model directory + inputs through two libraries exporting the
reference's C ABI (the B200 engine and the reference-compiled oracle) and compare every requested tensor.

The reference's outputs are stored under tests/golden/reference/ (one .npz per case), so the suite compares against the
original project without needing it.  `reference_outputs` loads a case; with OSB_RECORD_REFERENCE set to the oracle library
(oracle/_ref/liboracle_ref.so, built by __graft_entry__.build() next to the reference sources) it runs the reference and
stores the case instead -- see tests/golden/make_golden.py."""
import os

import numpy as np

from onnxstream_b200.model import Model

REFERENCE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
SAMPLE = 1024      # tensors larger than this are stored as a fixed, seeded sample of their elements


def golden_sample(a):
    """`a` itself when it is small; otherwise the same SAMPLE elements (chosen from its size alone) that are stored for a
    reference tensor of that size."""
    a = np.asarray(a)
    if a.size <= SAMPLE:
        return a
    idx = np.sort(np.random.default_rng(a.size).permutation(a.size)[:SAMPLE])
    return a.reshape(-1)[idx]


class Reference(dict):
    """name -> the reference's tensor (golden_sample() of it when large); `shapes`: name -> its full shape."""

    def __init__(self, tensors, shapes):
        super().__init__(tensors)
        self.shapes = shapes


def reference_outputs(case, run):
    """What the reference returned for `case`.  `run(lib) -> {name: array}` computes it with the library at `lib`; it is
    called only when recording (OSB_RECORD_REFERENCE=<oracle library>)."""
    fn = os.path.join(REFERENCE_DIR, case + ".npz")
    lib = os.environ.get("OSB_RECORD_REFERENCE")
    if lib:
        out = {k: np.asarray(v) for k, v in run(lib).items() if v is not None}
        os.makedirs(REFERENCE_DIR, exist_ok=True)
        np.savez_compressed(fn, **{"t:" + k: golden_sample(v) for k, v in out.items()},
                            **{"s:" + k: np.asarray(v.shape, np.int64) for k, v in out.items()})
    assert os.path.exists(fn), f"no stored reference output for {case!r} (tests/golden/make_golden.py records it)"
    z = np.load(fn)
    return Reference({k[2:]: z[k] for k in z.files if k.startswith("t:")}, {k[2:]: tuple(int(x) for x in z[k]) for k in z.files if k.startswith("s:")})


def run_model(lib, model_dir, inputs, options=(), extra_outputs=(), wp="nocache", parts=None, ranges=None, upcast=(), b200_options=(), runs=1, plain_abi=False):
    m = Model(lib, 4, wp, plain_abi=plain_abi)   # 4 pthreadpool workers for the CPU oracle (0 = every core: slow on many-core hosts); the GPU engine ignores it
    for o in options:
        m.set_option(o, True)
    for name, val in b200_options:
        m.lib.model_set_option(m.h, name.encode(), int(val))
    if parts is not None:
        m.set_attention_parts(parts)
    for k, (mn, mx) in (ranges or {}).items():
        m.set_range(k, mn, mx)
    for p in upcast:
        m.add_upcast_pattern(p)
    for e in extra_outputs:
        m.add_extra_output(e)
    m.read_file(model_dir.rstrip("/") + "/model.txt")
    out = None
    for _ in range(runs):
        m.clear_tensors()
        for k, v in inputs.items():
            m.add_tensor(k, v)
        m.run()
        out = {}
        for n in m.get_all_tensor_names():
            t = m.get_tensor(n)
            if t is None and not plain_abi:
                t = m.get_tensor_i64(n)
            out[n] = t
    return out, m


def report(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    d = np.abs(a - b)
    denom = max(np.abs(b).max(), 1e-12)
    return dict(max_abs=float(d.max()) if d.size else 0.0, rel_to_max=float(d.max() / denom) if d.size else 0.0,
                rms=float(np.sqrt((d ** 2).mean())) if d.size else 0.0, ref_rms=float(np.sqrt((b ** 2).mean())) if b.size else 0.0)
