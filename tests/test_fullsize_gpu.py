"""GPU parity at BASELINE sizes: the B200 engine vs the reference's own Model::run() (oracle/_ref) on the FULL-SIZE
synthetic graphs bench.py times -- not the tiny variants of test_models_gpu.py -- and on the one real model the reference
vendors (YOLOv8n, 233 ops, staged by oracle/Makefile under oracle/_ref/fixtures/ so nothing here reads /root/reference).

One reference run of a full-size graph costs minutes on the host cores, so the reference's outputs are stored under
tests/golden/reference/ (a fixed, seeded sample of each output; tests/util.py); the engine side runs in every mode (streamed
ring, HBM-resident, CUDA-graph replay) against that one stored result.

Tolerances (same bars as test_models_gpu.py; observed values in the assertion messages):
  * fp32 graphs                      : |err| <= 2e-4 * max|ref|
  * fp16 graphs vs the fp16 oracle   : |err| <= 3e-2 * max|ref|, and rms error vs the fp32-arithmetic truth no worse than 2x the
                                       reference's own fp16 mode (two valid fp16 evaluations of a 2000-op network)
  * W8A32 (uint8 weights, fp32 act.) : |err| <= 2e-4 * max|ref| (dequantisation is exact; only summation order differs)
"""
import os

import numpy as np
import pytest

from onnxstream_b200 import emit
from onnxstream_b200.model import Model
from util import golden_sample, reference_outputs, report

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHM = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
REF_THREADS = min(os.cpu_count() or 1, 32)
FP16 = ("use_fp16_arithmetic", "fuse_ops_in_attention")


def _model_dir(tag, emit_fn):
    d = os.path.join(SHM, f"osb200_full_{tag}") + "/"
    if not os.path.exists(d + "model.txt.done"):
        emit_fn(d)
        open(d + "model.txt.done", "w").write("ok")
    return d


def _run(lib, d, inputs, opts, outs, threads=4, wp="nocache", b200=(), runs=1, extra=()):
    m = Model(lib, threads, wp)
    for o in opts:
        m.set_option(o, True)
    for k, v in b200:
        m.lib.model_set_option(m.h, k.encode(), int(v))
    for e in extra:
        m.add_extra_output(e)
    m.read_file(d + "model.txt")
    res = None
    for _ in range(runs):
        m.clear_tensors()
        for k, v in inputs.items():
            m.add_tensor(k, v)
        m.run()
        res = {o: m.get_tensor(o) for o in outs}
    return res, m


def _reference(case, d, inputs, opts, outs, extra=()):
    """The reference's own Model::run on the host cores (stored; recomputed only when recording)."""
    def run(oracle_lib):
        import ctypes
        gomp = ctypes.CDLL(oracle_lib)                   # dlsym through the oracle's own dependencies: the libgomp IT links (torch's copy)
        # the shim's OpenMP loops: conftest caps them at 4 threads for the small tests
        gomp.omp_set_num_threads(REF_THREADS)
        try:
            res, m = _run(oracle_lib, d, inputs, opts, outs, threads=REF_THREADS, extra=extra)
            m.close()
        finally:
            gomp.omp_set_num_threads(int(os.environ.get("OMP_NUM_THREADS", "4")))
        return res
    return reference_outputs(case, run)


# ---------------------------------------------------------------------------------------------------------------------
# YOLOv8n: the reference's only vendored real model (examples/YOLOv8n_wasm/yolov8n_fp32: 64 Conv, 58 Sigmoid*Mul, Concat, Split,
# MaxPool, Resize, Slice, Softmax ...), real trained weights, 640x640 input
# ---------------------------------------------------------------------------------------------------------------------
YOLO = os.path.join(ROOT, "oracle", "_ref", "fixtures", "yolov8n_fp32") + "/"


def _yolo_extra():
    lines = open(YOLO + "model.txt").read().splitlines()
    convs = [l.split("*output:")[1].split("(")[0] for l in lines if ":Conv*" in l]
    others = [l.split("*output:")[1].split("(")[0] for l in lines if l.split("*")[0].endswith((":MaxPool", ":Resize", ":Softmax"))]
    return [convs[0], convs[7], convs[30], convs[-1]] + others[:4]


@pytest.mark.skipif(not os.path.exists(YOLO + "model.txt"), reason="YOLOv8n fixture not staged (oracle/Makefile copies it where /root/reference exists)")
@pytest.mark.parametrize("fuse", [0, 1])
def test_yolov8n_fp32(engine_lib, fuse):
    x = np.random.default_rng(0).random((1, 3, 640, 640)).astype(np.float32)
    extra = _yolo_extra()
    outs = ["output0"] + extra
    ref = _reference("yolov8n32", YOLO, {"images": x}, (), outs, extra=extra)
    got, m = _run(engine_lib, YOLO, {"images": x}, (), outs, b200=(("b200_fuse_nodes", fuse), ("b200_keep_nhwc", fuse)), extra=extra)
    for o in outs:
        assert got[o] is not None and got[o].shape == ref.shapes[o], o
        r = report(golden_sample(got[o]), ref[o])
        assert r["rel_to_max"] <= 2e-4, (o, r)
    assert m.stats()["kernel_launches"] > 0
    # fp32 convolutions run on the tensor cores too (bf16 triple split): the fp32 bar above is met THROUGH that path
    assert m.stats()["tc_launches"] > 40, m.stats()


@pytest.mark.skipif(not os.path.exists(YOLO + "model.txt"), reason="YOLOv8n fixture not staged")
def test_yolov8n_fp16_arithmetic(engine_lib):
    """fp32 blobs run in m_use_fp16_arithmetic mode (weights rounded to fp16 at load, src/onnxstream.cpp:2901-2909): the tcgen05 conv path."""
    x = np.random.default_rng(0).random((1, 3, 640, 640)).astype(np.float32)
    truth = _reference("yolov8n32_output", YOLO, {"images": x}, (), ["output0"])
    ref = _reference("yolov8n16_output", YOLO, {"images": x}, ("use_fp16_arithmetic",), ["output0"])
    got, m = _run(engine_lib, YOLO, {"images": x}, ("use_fp16_arithmetic",), ["output0"])
    got = {"output0": golden_sample(got["output0"])}
    e_ref = report(ref["output0"], truth["output0"])
    e_got = report(got["output0"], truth["output0"])
    # box coordinates reach ~640: compare relative to the tensor's range, and never worse than twice the reference's own fp16 error
    assert e_got["rms"] <= 2.0 * e_ref["rms"] + 1e-3 * e_got["ref_rms"], (e_got, e_ref)
    assert report(got["output0"], ref["output0"])["rel_to_max"] <= 3e-2
    assert m.stats()["tc_launches"] > 0, "the tcgen05 path did not run"


# ---------------------------------------------------------------------------------------------------------------------
# SD 1.5 UNet, the exact graph bench.py times (BASELINE config[1]): 2127 ops, 860 M params, 64x64 latent, fp16
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sd15():
    cfg = emit.UNetConfig.sd15(64)
    d = _model_dir("sd15_unet_fp16", lambda d: emit.emit_unet(d, cfg, "float16", seed=0))
    return d, emit.unet_inputs(cfg)


def _check_fp16(got, ref, truth, what):
    got = golden_sample(got)
    r = report(got, ref)
    assert r["rel_to_max"] <= 3e-2, (what, r)
    e_ref, e_got = report(ref, truth)["rms"], report(got, truth)["rms"]
    assert e_got <= 2.0 * e_ref + 2e-3 * report(truth, truth)["ref_rms"], (what, e_got, e_ref, r)


def test_sd15_unet_full_streamed_resident_graph(engine_lib, sd15):
    d, inputs = sd15
    out = "out_5F_sample"
    ref = _reference("sd15_full16", d, inputs, FP16, [out])[out]            # the reference's fp16 mode
    truth = _reference("sd15_full16as32", d, inputs, ("fuse_ops_in_attention",), [out])[out]   # same fp16 weights, fp32 arithmetic
    # (1) streamed: every run moves all 1.72 GB through the HBM ring (the north-star mode)
    got, m = _run(engine_lib, d, inputs, FP16, [out], wp="ram+nocache", runs=2)
    st = m.stats()
    _check_fp16(got[out], ref, truth, "streamed")
    assert st["weight_bytes_streamed"] > 1.6e9 and st["weight_ring_bytes"] <= st["weight_largest_node_bytes"] + 4096, st
    assert st["tc_launches"] > 200, st
    m.close()
    # (2) HBM-resident weights, eager; (3) the captured CUDA graph (third run captures, fourth replays)
    got2, m2 = _run(engine_lib, d, inputs, FP16, [out], wp="ram+nocache", b200=(("b200_resident_weights", 1),), runs=2)
    _check_fp16(got2[out], ref, truth, "resident")
    m2.close()
    got3, m3 = _run(engine_lib, d, inputs, FP16, [out], wp="ram+nocache", b200=(("b200_resident_weights", 1), ("b200_cuda_graph", 1)), runs=4)
    _check_fp16(got3[out], ref, truth, "graph replay")
    assert m3.stats()["graph_replays"] >= 1
    # the three modes run the same kernels on the same bytes; fp32 / fp64 atomics (single-launch GEMV, GroupNorm partials) make the
    # summation order vary from run to run, and a 2000-op fp16 network amplifies a flipped rounding to ~2e-3 of the output range
    assert report(got[out], got2[out])["rel_to_max"] <= 1e-2
    assert report(got3[out], got2[out])["rel_to_max"] <= 1e-2
    m3.close()


# ---------------------------------------------------------------------------------------------------------------------
# SDXL UNet topology (10-deep transformers, head dim 64, 2048-wide context, add-embedding), uint8 weights + fp32 activations
# (W8A32, BASELINE config[2]/[3]) at a 64x64 latent (SDXL Turbo's 512x512)
# ---------------------------------------------------------------------------------------------------------------------
def test_sdxl_unet_w8a32_full(engine_lib):
    cfg = emit.UNetConfig.sdxl(64)
    d = _model_dir("sdxl_unet_u8", lambda d: emit.emit_unet(d, cfg, "uint8", seed=0))
    inputs = emit.unet_inputs(cfg)
    out = "out_5F_sample"
    ref = _reference("sdxl_full_u8", d, inputs, ("fuse_ops_in_attention",), [out])[out]
    got, m = _run(engine_lib, d, inputs, ("fuse_ops_in_attention",), [out], wp="ram+nocache")
    r = report(golden_sample(got[out]), ref)
    assert r["rel_to_max"] <= 2e-4, r
    st = m.stats()
    assert st["weight_bytes_streamed"] > 2.0e9, st      # uint8 blobs cross PCIe as uint8
    m.close()


# ---------------------------------------------------------------------------------------------------------------------
# VAE decoder 4x64x64 -> 3x512x512 (BASELINE config[1]'s last stage), fp16
# ---------------------------------------------------------------------------------------------------------------------
def test_vae_decoder_full(engine_lib):
    cfg = emit.VAEConfig()
    d = _model_dir("vae_dec_fp16", lambda d: emit.emit_vae_decoder(d, cfg, "float16"))
    inputs = {"input_2E_1": np.random.default_rng(5).standard_normal((1, 4, cfg.latent, cfg.latent)).astype(np.float32)}
    out = "outsample"
    ref = _reference("vae_full16", d, inputs, FP16, [out])[out]
    truth = _reference("vae_full32", d, inputs, (), [out])[out]
    got, m = _run(engine_lib, d, inputs, FP16, [out], wp="ram+nocache")
    assert got[out].shape == (1, 3, 512, 512)
    _check_fp16(got[out], ref, truth, "vae decoder")
    m.close()
