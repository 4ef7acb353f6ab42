"""GPU parity: the B200 engine vs the reference's own Model::run() (oracle/_ref) on the same model directories and
seeded inputs, both driven through the reference's C ABI (model_new_2 / model_read_file / push / model_run_2 /
model_get_tensor).  Sizes are the tiny variants of every BASELINE architecture so the CPU oracle finishes in seconds.
The oracle's outputs are stored under tests/golden/reference/ (tests/util.py reference_outputs), so these tests need only
the engine and a GPU.

Tolerances (stated per SURVEY section 7.2 "Numerical parity definition"):
  * fp32 mode  : |err| <= 2e-4 * max|ref|   (different summation order only; observed ~1e-6)
  * fp16 mode  : |err| <= 2e-2 * max|ref|   (fp16 storage at node boundaries, fp32 accumulation; observed ~2e-3).  The oracle
                 here runs the reference with m_use_fp16_arithmetic: XNNPACK f16 elementwise ops + the shim's
                 fp16-storage/fp32-arithmetic Conv/FC (oracle/xnn_shim.cpp).
"""
import os
import tempfile

import numpy as np
import pytest

from onnxstream_b200 import emit
from util import golden_sample, reference_outputs, run_model, report

pytestmark = pytest.mark.gpu

FP16 = ("use_fp16_arithmetic", "fuse_ops_in_attention")
TOL = {"float32": 2e-4, "float16": 2e-2}


@pytest.fixture(scope="module")
def workdir():
    with tempfile.TemporaryDirectory(prefix="osb200_t_") as d:
        yield d


def _models(workdir, wdtype):
    out = {}
    cfg = emit.UNetConfig.tiny(8)
    d = os.path.join(workdir, f"unet_{wdtype}") + "/"
    emit.emit_unet(d, cfg, wdtype, seed=0)
    out["unet"] = (d, emit.unet_inputs(cfg), "out_5F_sample")
    cfgx = emit.UNetConfig.tiny(8, sdxl=True)
    d = os.path.join(workdir, f"sdxl_{wdtype}") + "/"
    emit.emit_unet(d, cfgx, wdtype, seed=3)
    out["sdxl_unet"] = (d, emit.unet_inputs(cfgx), "out_5F_sample")
    vc = emit.VAEConfig.tiny(8)
    d = os.path.join(workdir, f"vae_{wdtype}") + "/"
    emit.emit_vae_decoder(d, vc, wdtype)
    out["vae"] = (d, {"input_2E_1": np.random.default_rng(5).standard_normal((1, 4, 8, 8)).astype(np.float32)}, "outsample")
    cc = emit.CLIPConfig.tiny()
    d = os.path.join(workdir, f"clip_{wdtype}") + "/"
    emit.emit_text_encoder(d, cc, wdtype)
    out["clip"] = (d, {"input_5F_ids": np.random.default_rng(6).integers(0, cc.vocab, (1, cc.tokens)).astype(np.int64)}, "last_5F_hidden_5F_state")
    return out


@pytest.fixture(scope="module")
def models32(workdir):
    return _models(workdir, "float32")


@pytest.fixture(scope="module")
def models16(workdir):
    return _models(workdir, "float16")


def _oracle(case, d, inputs, opts, **kw):
    """The reference's outputs for `case` (tests/golden/reference/<case>.npz: the model directory, inputs and options here)."""
    return reference_outputs(case, lambda lib: run_model(lib, d, inputs, opts, **kw)[0])


@pytest.mark.parametrize("arch", ["unet", "sdxl_unet", "vae", "clip"])
@pytest.mark.parametrize("fuse,nhwc", [(0, 0), (1, 1)])
def test_fp32_parity(engine_lib, models32, arch, fuse, nhwc):
    d, inputs, out = models32[arch]
    ref = _oracle(arch + "32", d, inputs, ())
    got, m = run_model(engine_lib, d, inputs, (), b200_options=(("b200_fuse_nodes", fuse), ("b200_keep_nhwc", nhwc)))
    assert set(got) == set(ref), (sorted(got), sorted(ref))
    r = report(golden_sample(got[out]), ref[out])
    assert r["rel_to_max"] <= TOL["float32"], r
    assert m.stats()["kernel_launches"] > 0


@pytest.mark.parametrize("arch", ["unet", "sdxl_unet", "vae", "clip"])
@pytest.mark.parametrize("fuse,nhwc,impl", [(0, 0, 1), (1, 1, 0)])
def test_fp16_parity(engine_lib, models16, arch, fuse, nhwc, impl):
    d, inputs, out = models16[arch]
    ref = _oracle(arch + "16", d, inputs, FP16)
    truth = _oracle(arch + "16as32", d, inputs, ())          # same fp16 weights, fp32 arithmetic
    got, m = run_model(engine_lib, d, inputs, FP16, b200_options=(("b200_fuse_nodes", fuse), ("b200_keep_nhwc", nhwc), ("b200_gemm_impl", impl)))
    got[out] = golden_sample(got[out])
    r = report(got[out], ref[out])
    # (1) close to the reference's own fp16 mode ...
    assert r["rel_to_max"] <= 1.5 * TOL["float16"], r
    # (2) ... and no further from the fp32-arithmetic result than the reference's fp16 mode is (x2 slack + fp16 resolution):
    # two valid fp16 evaluations of a deep GroupNorm network differ from each other by about as much as each differs from fp32
    e_ref = report(ref[out], truth[out])["rms"]
    e_got = report(got[out], truth[out])["rms"]
    assert e_got <= 2.0 * e_ref + 2e-3 * report(truth[out], truth[out])["ref_rms"], (e_got, e_ref, r)
    if impl == 0 and arch != "clip":
        assert m.stats()["tc_launches"] > 0, "the tcgen05 path did not run"


def test_fp16_weights_fp32_arithmetic(engine_lib, models16):
    """fp16 blobs with m_use_fp16_arithmetic off: weights are up-converted at load (src/onnxstream.cpp:2892-2900)."""
    d, inputs, out = models16["unet"]
    ref = _oracle("unet16as32", d, inputs, ())
    got, _ = run_model(engine_lib, d, inputs, ())
    assert report(golden_sample(got[out]), ref[out])["rel_to_max"] <= TOL["float32"]


def test_intermediates_match(engine_lib, models32):
    """m_extra_outputs (src/onnxstream.h:954): a few intermediates, which also forces the fused groups around them apart."""
    d, inputs, out = models32["unet"]
    lines = open(d + "model.txt").read().splitlines()
    names = []
    for want in ("Conv", "InstanceNormalization", "Softmax", "Gemm", "Resize", "Concat"):
        for l in lines:
            if f":{want}*" in l:
                names.append(l.split("*output:")[1].split("(")[0])
                break
    ref = _oracle("unet32_intermediates", d, inputs, (), extra_outputs=names)
    got = run_model(engine_lib, d, inputs, (), extra_outputs=names)[0]
    for n in names + [out]:
        assert got[n].shape == ref.shapes[n], n
        r = report(golden_sample(got[n]), ref[n])
        assert r["rel_to_max"] <= 5e-4, (n, r)


def test_streaming_ring_bound(engine_lib, models16):
    """The HBM weight ring never exceeds one node's footprint (north star: peak resident weights <= largest node)."""
    d, inputs, out = models16["unet"]
    got, m = run_model(engine_lib, d, inputs, FP16, wp="ram+nocache", runs=2)
    st = m.stats()
    assert st["weight_ring_bytes"] <= st["weight_largest_node_bytes"] + 8192
    assert st["weight_peak_live_bytes"] <= st["weight_ring_bytes"]
    total = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d) if f.endswith(".bin"))
    assert abs(st["weight_bytes_streamed"] - total) <= 8 * 4096   # every float blob crosses PCIe exactly once per run (int64 shape constants stay on the host)
    assert st["weight_resident_bytes"] == 0


@pytest.mark.parametrize("wp", ["prefetch", "ram+nocache", "ram+prefetch"])
def test_providers_agree(engine_lib, models16, wp):
    d, inputs, out = models16["unet"]
    a, _ = run_model(engine_lib, d, inputs, FP16, wp="nocache")
    b, _ = run_model(engine_lib, d, inputs, FP16, wp=wp, runs=2)
    assert np.array_equal(a[out], b[out])


def test_resident_and_graph_bit_identical(engine_lib, models16):
    d, inputs, out = models16["unet"]
    a, _ = run_model(engine_lib, d, inputs, FP16, wp="ram+nocache")
    b, m = run_model(engine_lib, d, inputs, FP16, wp="ram+nocache", b200_options=(("b200_resident_weights", 1), ("b200_cuda_graph", 1)), runs=5)
    assert np.array_equal(a[out], b[out])
    assert m.stats()["graph_replays"] >= 1
    assert m.run_resident(3) > 0


def test_in_memory_weights(engine_lib, workdir):
    """model_read_string + model_add_weights_file ('ram' provider), the WASM-style flow (src/exports.cpp:92-96,150-167)."""
    from onnxstream_b200.model import Model
    cfg = emit.UNetConfig.tiny(8)
    g = emit.emit_unet(None, cfg, "float32", seed=9, keep_in_memory=True)
    inputs = emit.unet_inputs(cfg)

    def run(lib):
        m = Model(lib, 0, "ram")
        m.read_string(g.text())
        names = m.get_weights_names()
        for dt, fn in names:
            m.add_weights_file(dt, fn, g.blobs[fn][1])
        for k, v in inputs.items():
            m.add_tensor(k, v)
        m.run()
        return {"out_5F_sample": m.get_tensor("out_5F_sample")}
    ref = reference_outputs("unet32_seed9_ram", run)["out_5F_sample"]
    got = run(engine_lib)["out_5F_sample"]
    assert report(golden_sample(got), ref)["rel_to_max"] <= 2e-4


def test_batch_siblings(engine_lib, models16):
    """Tensors pushed twice under the same name run as a batch: weights fetched once, every op loops over the samples
    (src/onnxstream.cpp:3040-3050, 3817-3857)."""
    from onnxstream_b200.model import Model
    d, inputs, out = models16["unet"]
    inputs2 = {k: (v + 0.25 if v.dtype == np.float32 and v.size > 1 else v) for k, v in inputs.items()}
    single = [run_model(engine_lib, d, i, FP16)[0][out] for i in (inputs, inputs2)]
    m = Model(engine_lib, 0, "nocache")
    for o in FP16:
        m.set_option(o, True)
    m.read_file(d + "model.txt")
    for i in (inputs, inputs2):
        for k, v in i.items():
            m.add_tensor(k, v)
    m.run()
    assert m.get_all_tensor_names().count(out) == 2
    # both siblings against their single-sample runs (model_get_tensor = first sibling, model_ext_get_tensor_at = any)
    for k in range(2):
        assert report(m.get_tensor(out, k), single[k])["rel_to_max"] <= 2e-3, k
    assert report(m.get_tensor(out, 0), m.get_tensor(out, 1))["rel_to_max"] > 1e-2      # they really are different samples


def test_uint8_qdq_mode(engine_lib, models32):
    """m_use_uint8_qdq (src/onnxstream.cpp:3006-3031, 3104-3434): every op output is percentile-quantised to uint8 storage and
    dequantised on use -- GPU radix-select percentiles per reference chunk + XNNPACK's f32->qu8 conversion.  Both sides run with
    the same pool size (4), i.e. the same chunking.  The engine keeps conv trunks NHWC, so a chunk holds other elements than the
    reference's NCHW chunk: ranges agree statistically, not bitwise -- the bar is "no further from the fp32 result than the
    reference's own qdq mode" (x2 + slack)."""
    refs = {arch: (_oracle(arch + "32", models32[arch][0], models32[arch][1], ()),
                   _oracle(arch + "32qdq", models32[arch][0], models32[arch][1], ("use_uint8_qdq",))) for arch in ("unet", "vae")}
    for arch in ("unet", "vae"):
        d, inputs, out = models32[arch]
        truth, ref = refs[arch]
        got, m = run_model(engine_lib, d, inputs, ("use_uint8_qdq",))
        got[out] = golden_sample(got[out])
        e_ref, e_got = report(ref[out], truth[out]), report(got[out], truth[out])
        assert e_ref["rms"] > 0, "the reference's qdq run is identical to fp32: the mode did not engage"
        assert e_got["rms"] > 0, "the engine's qdq run is identical to fp32: the mode did not engage"
        assert e_got["rms"] <= 2.0 * e_ref["rms"] + 0.02 * e_got["ref_rms"], (arch, e_got, e_ref)


def _qu8_chain(d):
    """A graph whose every node has a uint8 kernel in the reference under m_use_uint8_arithmetic: Conv 3x3 -> Conv 1x1 -> Add -> Mul ->
    Reshape/Transpose -> MatMul.  Inputs are percentile-quantised at push (plain NCHW on both sides: identical chunks), every op
    output takes its scale from m_range_data: the whole chain is integer arithmetic."""
    g = emit.GraphBuilder(d, "uint8", seed=11)
    x = g.input("x", (1, 16, 12, 12))
    z = g.input("z", (1, 32, 12, 12))
    c1 = g.conv(x, 32, 3, name="c1")
    c2 = g.conv(c1, 32, 1, name="c2")
    a = g.node("Add", [c2, z], [c2.shape], name="add1")
    m = g.node("Mul", [a, c1], [a.shape], name="mul1")
    r = g.node("Reshape", [m, g.i64([1, 32, 144])], [(1, 32, 144)])
    t = g.node("Transpose", [r], [(1, 144, 32)], [("perm", "0,2,1")])
    y = g.linear(t, 32, bias=False, name="fc1")
    g.mark_output(y)
    g.finish()
    ranges = {"c1": (-2.5, 2.5), "c2": (-2.0, 2.2), "add1": (-4.0, 4.5), "mul1": (-6.0, 7.0), "fc1": (-9.0, 9.5)}
    rng = np.random.default_rng(12)
    inputs = {"x": rng.standard_normal((1, 16, 12, 12)).astype(np.float32), "z": (rng.standard_normal((1, 32, 12, 12)) * 1.5 + 0.3).astype(np.float32)}
    return y.name, ranges, inputs


def test_uint8_arithmetic_chain_bit_exact(engine_lib, workdir):
    """m_use_uint8_arithmetic end to end, BIT-EXACT against the reference: XNNPACK's real qu8 convolution / fully-connected / add /
    multiply kernels in oracle/_ref vs the engine's uint8 kernels (u8 x u8 -> s32, zero-point handling, fp32 requantisation
    clamp(lrintf(acc * sx*sw/sy)) + zy; fixed-point add), percentile quantisation of the graph inputs included."""
    d = os.path.join(workdir, "qu8chain") + "/"
    out, ranges, inputs = _qu8_chain(d)
    opts = ("use_uint8_arithmetic",)
    extra = ["c1", "c2", "add1", "mul1"]
    names = {}
    for l in open(d + "model.txt").read().splitlines():
        nm = l.split(":")[0]
        if nm in extra:
            names[nm] = l.split("*output:")[1].split("(")[0]
    ref = _oracle("qu8_chain", d, inputs, opts, ranges=ranges, extra_outputs=list(names.values()))
    got, m = run_model(engine_lib, d, inputs, opts, ranges=ranges, extra_outputs=list(names.values()))
    for nm, tn in list(names.items()) + [("fc1", out)]:
        assert got[tn].shape == ref.shapes[tn], nm
        got[tn] = golden_sample(got[tn])
        bad = int((got[tn] != ref[tn]).sum())
        assert bad == 0, f"{nm}: {bad} of {ref[tn].size} values differ from the reference (max {float(np.abs(got[tn] - ref[tn]).max()):.4g})"


def test_tiled_vae_decode_batched(engine_lib, workdir):
    """SURVEY section 8 f3: sd.cpp's tiled VAE decode (src/sd.cpp:1258-1346, 2399-2503) with ALL tiles as batch siblings of one run.
    (1) batched == tile-by-tile on the engine; (2) engine == the reference decoding tile by tile + the same feather blend."""
    from onnxstream_b200.model import Model
    from onnxstream_b200 import tiled_vae as tv
    vc = emit.VAEConfig.tiny(8)          # the decoder graph is built for 8x8 latent tiles -> 64x64 pixel tiles
    d = os.path.join(workdir, "vae_tiles") + "/"
    emit.emit_vae_decoder(d, vc, "float16")
    latent = np.random.default_rng(3).standard_normal((1, 4, 20, 14)).astype(np.float32)    # 3 x 2 overlapping tiles (stride 6)

    def mk(lib):
        m = Model(lib, 4, "nocache")
        for o in FP16:
            m.set_option(o, True)
        m.read_file(d + "model.txt")
        return m
    kw = dict(tile=8, stride=6)
    img_r = reference_outputs("vae_tiles16", lambda lib: {"image": tv.tiled_decode(mk(lib), latent, "input_2E_1", "outsample", batched=False, **kw)[0]})
    img_b, n = tv.tiled_decode(mk(engine_lib), latent, "input_2E_1", "outsample", batched=True, **kw)
    img_s, _ = tv.tiled_decode(mk(engine_lib), latent, "input_2E_1", "outsample", batched=False, **kw)
    up = img_b.shape[-1] // 14
    assert n == 6 and img_b.shape == (1, 3, 20 * up, 14 * up) and up in (4, 8) and img_r.shapes["image"] == img_b.shape
    assert report(img_b, img_s)["rel_to_max"] <= 2e-3          # same kernels, batch siblings vs separate runs
    assert report(golden_sample(img_b), img_r["image"])["rel_to_max"] <= 3e-2, report(golden_sample(img_b), img_r["image"])


def test_force_fp16_storage(engine_lib, models32):
    """m_force_fp16_storage (src/onnxstream.cpp:3764-3808): fp32 arithmetic, fp16 storage between ops."""
    d, inputs, out = models32["unet"]
    truth = _oracle("unet32", d, inputs, ())
    ref = _oracle("unet32f16s", d, inputs, ("force_fp16_storage",))
    got, _ = run_model(engine_lib, d, inputs, ("force_fp16_storage",))
    got[out] = golden_sample(got[out])
    e_ref, e_got = report(ref[out], truth[out]), report(got[out], truth[out])
    assert e_ref["rms"] > 0 and e_got["rms"] > 0, "storage rounding did not engage"
    assert report(got[out], ref[out])["rel_to_max"] <= 1e-2
    assert e_got["rms"] <= 2.0 * e_ref["rms"] + 1e-3 * e_got["ref_rms"], (e_got, e_ref)


def test_range_calibration(engine_lib, models32):
    """m_range_data_calibrate (src/onnxstream.cpp:2983-3004) on the engine: one calibration run records a percentile range per op;
    sanity: every Conv / MatMul has a finite, ordered range that brackets most of that op's output."""
    from onnxstream_b200.model import Model
    d, inputs, out = models32["unet"]
    m = Model(engine_lib, 4, "nocache")
    m.lib.model_set_option(m.h, b"b200_range_data_calibrate", 1)
    m.add_extra_output  # noqa: B018 (API presence)
    m.read_file(d + "model.txt")
    for k, v in inputs.items():
        m.add_tensor(k, v)
    m.run()
    import tempfile
    fn = tempfile.mktemp(suffix=".txt")
    m.lib.model_ext_write_range_data.argtypes = [__import__("ctypes").c_void_p, __import__("ctypes").c_char_p]
    m.lib.model_ext_write_range_data.restype = __import__("ctypes").c_void_p
    assert not m.lib.model_ext_write_range_data(m.h, fn.encode())
    lines = [l for l in open(fn).read().splitlines() if l]
    recorded = {l.split(",")[0]: (float(l.split(",")[1]), float(l.split(",")[2])) for l in lines}
    convs = [l.split(":")[0] for l in open(d + "model.txt").read().splitlines() if ":Conv*" in l]
    # every float-producing step leaves a range under the name of the op that pushed it (fused groups: their last op)
    assert len(recorded) > 100, len(recorded)
    assert all(lo < hi and np.isfinite(lo) and np.isfinite(hi) for lo, hi in recorded.values())
    assert sum(1 for c in convs if c in recorded) >= len(convs) // 4, "no Conv output range was recorded"


def test_errors_are_reported(engine_lib, workdir):
    from onnxstream_b200.model import Model, OnnxStreamError
    m = Model(engine_lib, 0, "nocache")
    with pytest.raises(OnnxStreamError):
        m.read_file(os.path.join(workdir, "does_not_exist", "model.txt"))
    m.read_string("a:Frobnicate*input:x(1,2)*output:y(1,2)\n")
    m.add_tensor("x", np.zeros((1, 2), np.float32))
    with pytest.raises(OnnxStreamError, match="Frobnicate"):
        m.run()
    m2 = Model(engine_lib, 0, "nocache")
    m2.read_string("a:Add*input:x(1,2);z(1,2)*output:y(1,2)\n")
    m2.add_tensor("x", np.zeros((1, 2), np.float32))
    with pytest.raises(OnnxStreamError, match="input tensor not found"):
        m2.run()
    m3 = Model(engine_lib, 0, "nocache")
    m3.read_string("a:Sigmoid*input:x(1,2)*output:y(1,3)\n")
    m3.add_tensor("x", np.zeros((1, 2), np.float32))
    with pytest.raises(OnnxStreamError, match="unexpected shape of output"):
        m3.run()


def test_cpp_dropin(models32):
    """The reference's OWN exports.cpp + onnxstream.h (unmodified, compiled in place) on top of compat_onnxstream.cpp and the
    B200 engine: proves the C++ boundary (Model members, WeightsProvider contract, m_data hand-off) end to end."""
    lib = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "build", "link_test", "libonnxstream_ref_exports.so")
    if not os.path.exists(lib):
        pytest.skip("build/link_test not built (scripts/link_reference_apps.sh needs /root/reference)")
    d, inputs, out = models32["unet"]
    ref = _oracle("unet32", d, inputs, ())
    for wp in ("nocache", "ram+prefetch"):
        got, _ = run_model(lib, d, inputs, (), wp=wp, runs=2, plain_abi=True)
        assert report(golden_sample(got[out]), ref[out])["rel_to_max"] <= TOL["float32"], wp


UPCAST = ("_2F_input_5F_layernorm_2F_", "_2F_post_5F_attention_5F_layernorm_2F_", "_2F_norm_2F_")


@pytest.mark.parametrize("mode", ["float32", "float16"])
def test_llama_decode_parity(engine_lib, workdir, mode):
    """BASELINE config[4] hot path at toy size: Llama decode step with KV cache, grouped-KV ScaledDotProductAttention rewrite
    (src/onnxstream.cpp:3643-3695, 7767-7882), int64 token / position inputs (Gather), rotary, RMSNorm kept in fp32 through
    m_requires_upcast (src/llm.cpp:385-389).  logits and the grown KV cache are compared."""
    cfg = emit.LlamaConfig.tiny()
    d = os.path.join(workdir, f"llama_{mode}") + "/"
    emit.emit_llama_decode(d, cfg, mode)
    inputs = emit.llama_inputs(cfg)
    opts = ("use_scaled_dp_attn_op",) + (("use_fp16_arithmetic",) if mode == "float16" else ())
    kw = dict(extra_outputs=("opkv0", "opkv3"), upcast=UPCAST if mode == "float16" else ())
    ref = _oracle("llama_tiny_" + mode, d, inputs, opts, **kw)
    got = run_model(engine_lib, d, inputs, opts, **kw)[0]
    for n in ("logits", "opkv0", "opkv3"):
        assert got[n].shape == ref[n].shape
        assert report(got[n], ref[n])["rel_to_max"] <= TOL[mode], n
    # shape / index path is bit-exact: the appended cache row position and the gathered embedding row
    assert np.array_equal(got["opkv0"][:, :, :-1], ref["opkv0"][:, :, :-1]) or mode == "float16"


@pytest.mark.parametrize("wdtype", ["float16", "uint8"])
def test_llama_decode_midsize_fused_paths(engine_lib, workdir, wdtype):
    """The decode-step fusions at a size where they engage (hidden 256, 300 cached positions, 259-entry vocabulary): grouped q/k/v and
    gate/up GEMVs (fp16 and uint8 weights dequantised in registers), SiLU-gate pass, fused RMSNorm / rotary steps, split-KV decode
    attention, the row-padded copy of a weight whose N is not 16-byte granular, two-source Concat -- streamed, resident and graph-replay
    runs against ONE reference run, and the plan must really contain the fused steps."""
    from onnxstream_b200.model import plan_summary
    cfg = emit.LlamaConfig(vocab=259, hidden=256, heads=4, kv_heads=2, head_dim=64, mlp=512, layers=2, past=300, max_pos=512)
    d = os.path.join(workdir, f"llama_mid_{wdtype}") + "/"
    emit.emit_llama_decode(d, cfg, wdtype)
    inputs = emit.llama_inputs(cfg)
    mask = np.ones((1, cfg.past + 1), np.int64); mask[0, 5:40] = 0          # padded positions: the additive mask matters
    inputs["attention_5F_mask"] = mask
    opts = ("use_scaled_dp_attn_op", "use_fp16_arithmetic")
    kw = dict(extra_outputs=("opkv0", "opkv3"), upcast=UPCAST)
    rep = plan_summary(open(d + "model.txt").read(), use_scaled_dp_attn_op=True, library_path=engine_lib)
    last = rep.splitlines()[-1]
    for kind in ("RMSNORM=5", "ROPE=4", "GEMV_GROUP=2", "SWIGLU=2", "SDPA=2", "LINEAR=4"):
        assert kind in last, last
    ref = _oracle("llama_mid_%s_as32" % wdtype, d, inputs, ("use_scaled_dp_attn_op",), extra_outputs=("opkv0", "opkv3"))     # fp32 arithmetic on the same blobs
    ref16 = _oracle("llama_mid_%s" % wdtype, d, inputs, opts, **kw)
    tol = TOL["float16"] if wdtype == "float16" else 5e-2
    base_err = report(ref16["logits"], ref["logits"])["rel_to_max"]
    for b200 in ((), (("b200_resident_weights", 1),), (("b200_resident_weights", 1), ("b200_cuda_graph", 1))):
        got, m = run_model(engine_lib, d, inputs, opts, wp="ram+nocache", b200_options=b200, runs=4 if b200 else 1, **kw)
        for n in ("logits", "opkv0", "opkv3"):
            assert got[n].shape == ref.shapes[n]
            got[n] = golden_sample(got[n])
            assert report(got[n], ref16[n])["rel_to_max"] <= tol, (n, b200)
        # no further from the fp32-arithmetic result than the reference's own fp16 mode (x2 + slack)
        assert report(got["logits"], ref["logits"])["rel_to_max"] <= 2 * base_err + 2e-3, b200
        if len(b200) == 2:
            assert m.stats()["graph_replays"] >= 1


def test_llama_decode_graph_replay_follows_token_ids(engine_lib, workdir):
    """int64 graph inputs and CUDA graphs: token ids / positions / mask reach the device through int64 mirrors (Gather indices, Cast),
    so the captured decode step can be REPLAYED with new ids.  A captured model fed a sequence of different (id, position) pairs must
    reproduce what a fresh eager model computes for each of them; the KV cache stays in HBM (b200_keep_inputs) after the first push."""
    from onnxstream_b200.model import Model
    cfg = emit.LlamaConfig.tiny()
    d = os.path.join(workdir, "llama_graph") + "/"
    emit.emit_llama_decode(d, cfg, "float16")
    base = emit.llama_inputs(cfg)
    opts = ("use_scaled_dp_attn_op", "use_fp16_arithmetic")

    def mk(graph):
        m = Model(engine_lib, 0, "ram+nocache")
        for o in opts:
            m.set_option(o, True)
        for p in UPCAST:
            m.add_upcast_pattern(p)
        if graph:
            for k in ("b200_resident_weights", "b200_cuda_graph", "b200_keep_inputs", "b200_drop_unconverted_outputs"):
                m.lib.model_set_option(m.h, k.encode(), 1)
            m.lib.model_ext_add_output_convert(m.h, b"logits")
        m.read_file(d + "model.txt")
        return m

    def step(m, inp):
        m.clear_tensors()
        for k, v in inp.items():
            m.add_tensor(k, v)
        m.run()
        return m.get_tensor("logits")

    g = mk(True)
    small = {k: v for k, v in base.items() if not k.startswith("pkv")}
    step(g, base)                                    # everything pushed once; the cache stays on the device
    replays0 = None
    for t in range(8):
        cur = dict(small)
        cur["input_5F_ids"] = np.array([[(7 * t + 3) % cfg.vocab]], np.int64)
        cur["position_5F_ids"] = np.array([[(cfg.past - t) % cfg.max_pos]], np.int64)
        mask = np.ones((1, cfg.past + 1), np.int64); mask[0, :t] = 0
        cur["attention_5F_mask"] = mask
        got = step(g, cur)
        full = dict(base); full.update(cur)
        want = step(mk(False), full)
        assert report(got, want)["rel_to_max"] <= 2e-3, (t, report(got, want))
    st = g.stats()
    assert st["graph_replays"] >= 3, st               # the later steps really were graph replays


@pytest.mark.parametrize("fp16", [False, True])
def test_w8a32_parity(engine_lib, workdir, fp16):
    """BASELINE config[2] weight format at toy size: uint8 per-tensor asymmetric weights (onnx2txt percentile rule) streamed
    as uint8 and dequantised on the device, fp32 (W8A32) or fp16 activations."""
    cfg = emit.UNetConfig.tiny(8, sdxl=True)
    d = os.path.join(workdir, "sdxl_u8") + "/"
    emit.emit_unet(d, cfg, "uint8", seed=3)
    inputs = emit.unet_inputs(cfg)
    opts = FP16 if fp16 else ()
    ref = _oracle("sdxl_u8_" + ("16" if fp16 else "32"), d, inputs, opts)["out_5F_sample"]
    got, m = run_model(engine_lib, d, inputs, opts, wp="ram+nocache", runs=2)
    assert report(golden_sample(got["out_5F_sample"]), ref)["rel_to_max"] <= (TOL["float16"] if fp16 else TOL["float32"])
    u8 = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d) if f.endswith(".bin"))
    assert abs(m.stats()["weight_bytes_streamed"] - u8) <= 8 * 4096      # uint8 bytes cross PCIe, not their fp32 expansion


def test_maxpool_trilu_scatternd_argmax(engine_lib, workdir):
    """The four remaining op types of the reference's run() loop (src/onnxstream.cpp:8075 MaxPool, 7883 Trilu, 7939 ScatterND,
    6930 ArgMax) in small graphs, engine vs the reference itself: floats within the fp32 bar, index results bit-exact."""
    rng = np.random.default_rng(7)
    # MaxPool after a Conv (YOLO SPPF shapes: k2 s2 p0, and k5 s1 p2 whose padding must be ignored, not zero-filled)
    d = os.path.join(workdir, "maxpool") + "/"
    g = emit.GraphBuilder(d, "float32", seed=11)
    x = g.input("x", (1, 8, 12, 12))
    c = g.conv(x, 16, 3)
    p1 = g.node("MaxPool", [c], [(1, 16, 6, 6)], [("ceil_mode", "0"), ("dilations", "1,1"), ("kernel_shape", "2,2"), ("pads", "0,0,0,0"), ("strides", "2,2")], out_names=["poola"])
    p2 = g.node("MaxPool", [c], [(1, 16, 12, 12)], [("ceil_mode", "0"), ("dilations", "1,1"), ("kernel_shape", "5,5"), ("pads", "2,2,2,2"), ("strides", "1,1")], out_names=["poolb"])
    g.finish()
    inputs = {"x": (rng.standard_normal((1, 8, 12, 12)) - 1.0).astype(np.float32)}   # mostly negative: zero padding would win the max
    # the same graphs and inputs as test_cpu.py's index-op cases
    refs = {opts: _oracle("index_g_maxpool" + ("16" if opts else ""), d, inputs, opts) for opts in ((), FP16)}
    for opts in ((), FP16):
        ref = refs[opts]
        got = run_model(engine_lib, d, inputs, opts)[0]
        for n in ("poola", "poolb"):
            assert got[n].shape == ref.shapes[n]
            assert report(golden_sample(got[n]), ref[n])["rel_to_max"] <= (TOL["float16"] if opts else TOL["float32"]), (n, opts)

    # Trilu (upper, k = 1) on a float32 matrix, then a scalar Mul so that the result is an activation output
    d = os.path.join(workdir, "trilu") + "/"
    g = emit.GraphBuilder(d, "float32", seed=12)
    m = g.input("m", (6, 7))
    t = g.node("Trilu", [m, g.const(np.asarray(1, dtype=np.int64))], [(6, 7)], [("upper", "1")])
    g.node("Mul", [t, g.scalar(2.0)], [(6, 7)], out_names=["tri"])
    g.finish()
    inputs = {"m": rng.standard_normal((6, 7)).astype(np.float32)}
    ref = _oracle("index_g_trilu", d, inputs, ())["tri"]
    got = run_model(engine_lib, d, inputs)[0]["tri"]
    assert np.array_equal(got, ref)
    assert np.array_equal(got, np.triu(inputs["m"], 1) * 2.0)

    # ScatterND with full-rank indices into a (4, 5) tensor
    d = os.path.join(workdir, "scatter") + "/"
    g = emit.GraphBuilder(d, "float32", seed=13)
    data = g.input("data", (4, 5))
    upd = g.input("upd", (2, 3))
    idx = np.asarray([[[0, 0], [1, 4], [3, 2]], [[2, 2], [0, 3], [3, 4]]], dtype=np.int64)
    s = g.node("ScatterND", [data, g.const(idx), upd], [(4, 5)])
    g.node("Mul", [s, g.scalar(1.0)], [(4, 5)], out_names=["scattered"])
    g.finish()
    inputs = {"data": rng.standard_normal((4, 5)).astype(np.float32), "upd": rng.standard_normal((2, 3)).astype(np.float32)}
    ref = _oracle("index_g_scatter", d, inputs, ())["scattered"]
    got = run_model(engine_lib, d, inputs)[0]["scattered"]
    want = inputs["data"].copy()
    want[idx[..., 0], idx[..., 1]] = inputs["upd"]
    assert np.array_equal(ref, want) and np.array_equal(got, want)

    # ArgMax over an int64 (1, D) tensor: first maximum wins
    d = os.path.join(workdir, "argmax") + "/"
    g = emit.GraphBuilder(d, "float32", seed=14)
    v = g.input("v", (1, 9))
    g.node("ArgMax", [v], [(1,)], [("axis", "-1"), ("keepdims", "0")], out_names=["arg"])
    g.finish()
    inputs = {"v": np.asarray([[3, -1, 7, 7, 2, 7, 0, -5, 6]], dtype=np.int64)}
    ref = _oracle("index_g_argmax", d, inputs, ())["arg"]
    got = run_model(engine_lib, d, inputs)[0]["arg"]
    assert np.array_equal(np.asarray(got).ravel(), [2]) and np.array_equal(np.asarray(ref).ravel(), [2])


@pytest.mark.xfail(strict=False, reason="written after round 1's GPU budget was spent: its first execution on a B200 is the driver's round-end run")
def test_exported_transformers_models_on_engine(engine_lib, workdir):
    """torch -> export_torch -> B200 engine: transformers' CLIPTextModel and LlamaForCausalLM (GQA, rotary, RMSNorm) with random weights;
    engine logits vs the reference's on the exported directory (the CPU suite already pins the reference against torch on the same export)."""
    torch = pytest.importorskip("torch")
    transformers = pytest.importorskip("transformers")
    from onnxstream_b200.export_torch import export_module

    class Wrap(torch.nn.Module):
        def __init__(s, m, f):
            super().__init__(); s.m = m; s.f = f

        def forward(s, ids):
            return s.f(s.m, ids)

    torch.manual_seed(0)
    clip = transformers.CLIPTextModel(transformers.CLIPTextConfig(vocab_size=100, hidden_size=32, intermediate_size=64, num_hidden_layers=2,
                                                                  num_attention_heads=4, max_position_embeddings=16)).eval()
    llama = transformers.LlamaForCausalLM(transformers.LlamaConfig(vocab_size=128, hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                                                                   num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=32)).eval()
    cases = [("clip", Wrap(clip, lambda m, ids: m(input_ids=ids).last_hidden_state), torch.randint(0, 100, (1, 16)), "last_hidden_state"),
             ("llama", Wrap(llama, lambda m, ids: m(input_ids=ids, use_cache=False).logits), torch.randint(0, 128, (1, 12)), "logits")]
    for name, w, ids, out in cases:
        for wd, opts in (("float32", ()), ("float16", FP16)):
            d = os.path.join(workdir, f"exp_{name}_{wd}") + "/"
            info = export_module(w, (ids,), d, wd, input_names=["input_ids"], output_names=[out])
            inputs = {info["inputs"][0]: ids.numpy().astype(np.int64)}
            ref = _oracle("export_%s_%s" % (name, wd), d, inputs, opts)     # the same exports as test_cpu.py's
            got = run_model(engine_lib, d, inputs, opts)[0][info["outputs"][0]]
            assert got.shape == ref.shapes[info["outputs"][0]]
            assert report(golden_sample(got), ref[info["outputs"][0]])["rel_to_max"] <= TOL[wd], (name, wd)
