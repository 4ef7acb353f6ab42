"""Generates the golden vectors in this directory from oracle/_ref (the reference's own sources compiled in place by
__graft_entry__.build() where the reference sources are present):  python tests/golden/make_golden.py
Each case = a seeded synthetic model directory (rebuilt deterministically by `build_case`) + inputs -> the reference output.
It then records tests/golden/reference/ by running the suite with OSB_RECORD_REFERENCE set (tests/util.py): every test
that compares with the reference stores the reference's outputs for its cases.  Without a GPU the GPU tests fail once
their reference outputs are recorded (the engine may abort the process), so every test function runs in a process of its own."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from onnxstream_b200 import emit  # noqa: E402

CASES = ["unet_tiny_fp32", "unet_tiny_fp16", "sdxl_tiny_fp32", "vae_tiny_fp32", "clip_tiny_fp32", "unet_tiny16_fp16_seed0", "unet_tiny16_fp16_seed1"]


def build_case(case: str, d: str):
    fp16 = case.endswith("fp16")
    wd = "float16" if fp16 else "float32"
    if case.startswith("unet_tiny16"):
        # smoke() and the 2-GPU test: sample `seed` of the 16x16-latent UNet
        cfg = emit.UNetConfig.tiny(16)
        emit.emit_unet(d, cfg, "float16", seed=0)
        return emit.unet_inputs(cfg, seed=int(case.rsplit("seed", 1)[1])), "out_5F_sample", True
    if case.startswith("unet_tiny"):
        cfg = emit.UNetConfig.tiny(8)
        emit.emit_unet(d, cfg, wd, seed=0)
        return emit.unet_inputs(cfg), "out_5F_sample", fp16
    if case.startswith("sdxl_tiny"):
        cfg = emit.UNetConfig.tiny(8, sdxl=True)
        emit.emit_unet(d, cfg, wd, seed=3)
        return emit.unet_inputs(cfg), "out_5F_sample", fp16
    if case.startswith("vae_tiny"):
        emit.emit_vae_decoder(d, emit.VAEConfig.tiny(8), wd)
        return {"input_2E_1": np.random.default_rng(5).standard_normal((1, 4, 8, 8)).astype(np.float32)}, "outsample", fp16
    if case.startswith("clip_tiny"):
        cc = emit.CLIPConfig.tiny()
        emit.emit_text_encoder(d, cc, wd)
        return {"input_5F_ids": np.random.default_rng(6).integers(0, cc.vocab, (1, cc.tokens)).astype(np.int64)}, "last_5F_hidden_5F_state", fp16
    raise KeyError(case)


if __name__ == "__main__":
    import tempfile
    from util import run_model
    oracle = os.path.join(ROOT, "oracle", "_ref", "liboracle_ref.so")
    for case in CASES:
        with tempfile.TemporaryDirectory() as d:
            d += "/"
            inputs, out_name, fp16 = build_case(case, d)
            opts = ("use_fp16_arithmetic", "fuse_ops_in_attention") if fp16 else ()
            out = run_model(oracle, d, inputs, opts)[0][out_name]
            np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), case + ".npz"), output=out,
                                **{"in_" + k: v for k, v in inputs.items()})
            print(case, out.shape, float(out.std()))
    pytest = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"]
    ids = subprocess.run(pytest + ["--collect-only", "tests"], cwd=ROOT, stdout=subprocess.PIPE, text=True).stdout.split()
    for test in sorted({i.split("[")[0] for i in ids if "::" in i}):
        subprocess.run(pytest + [test], env=dict(os.environ, OSB_RECORD_REFERENCE=oracle), cwd=ROOT)
