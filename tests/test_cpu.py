"""CPU-only suite (`-m "not gpu"`): the oracle against its pins, the host logic, and the C-ABI library surface.

Pinning of the oracle (SURVEY.md section 8c): the reference ships no tests or golden vectors, so
  (1) oracle/_ref = the reference's own sources compiled in place, i.e. outputs of the reference itself run here;
  (2) oracle/np_oracle.py = an independent numpy restatement;
(1) and (2) must agree on every tiny architecture, (2) must reproduce the committed golden vectors bit-for-bit, and
(1) must match torch on a Conv -> GroupNorm -> SiLU chain (the check the survey used to validate the XNNPACK build).
The outputs of (1) are stored under tests/golden/ (recorded by tests/golden/make_golden.py), so the suite runs without the
reference sources or oracle/_ref.
"""
import ctypes
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from onnxstream_b200 import emit
from util import golden_sample, reference_outputs, run_model, report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from np_oracle import NumpyOracle, parse_model  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE = os.path.join(ROOT, "oracle", "_ref", "liboracle_ref.so")


@pytest.fixture(scope="module")
def workdir():
    with tempfile.TemporaryDirectory(prefix="osb200_c_") as d:
        yield d


def _archs(workdir, wdtype="float32"):
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


@pytest.mark.parametrize("arch", ["unet", "sdxl_unet", "vae", "clip"])
def test_restatement_matches_reference_fp32(workdir, arch):
    d, inputs, out = _archs(workdir)[arch]
    ref = reference_outputs(arch + "32", lambda lib: run_model(lib, d, inputs, ())[0])[out]
    got = NumpyOracle(d).run(inputs)[out]
    assert report(golden_sample(got), ref)["rel_to_max"] <= 5e-5


def test_restatement_matches_reference_fp16(workdir):
    d, inputs, out = _archs(workdir, "float16")["unet"]
    ref = reference_outputs("unet16", lambda lib: run_model(lib, d, inputs, ("use_fp16_arithmetic", "fuse_ops_in_attention"))[0])[out]
    got = NumpyOracle(d, fp16=True).run(inputs)[out]
    assert report(golden_sample(got), ref)["rel_to_max"] <= 1e-2    # both round every node output to fp16; XNNPACK f16 elementwise differs in the last bit


def test_reference_matches_torch_conv_groupnorm_silu(workdir):
    import torch
    import torch.nn.functional as F
    g = emit.GraphBuilder(os.path.join(workdir, "cgs") + "/", "float32", seed=11, keep_in_memory=True)
    x = g.input("x", (1, 16, 12, 12))
    h = g.conv(x, 32, 3, stride=2, pad=1)
    h = g.silu(g.group_norm(h, 8, 1e-5))
    g.finish()
    xin = np.random.default_rng(1).standard_normal((1, 16, 12, 12)).astype(np.float32)
    ref = reference_outputs("conv_groupnorm_silu", lambda lib: run_model(lib, g.out_dir, {"x": xin}, ())[0])[h.name]
    names = list(g.blobs)
    w = torch.from_numpy(g.blobs[[n for n in names if n.endswith("_nhwc.bin")][0]][1]).permute(0, 3, 1, 2)
    vecs = [torch.from_numpy(g.blobs[n][1]) for n in names if not n.endswith("_nhwc.bin") and g.blobs[n][0] == "float32"]
    bias = vecs[0]
    gamma, beta = vecs[-2].reshape(-1), vecs[-1].reshape(-1)
    y = F.silu(F.group_norm(F.conv2d(torch.from_numpy(xin), w, bias, stride=2, padding=1), 8, gamma, beta, 1e-5)).numpy()
    assert report(ref, golden_sample(y))["max_abs"] <= 2e-5


def _index_graphs(workdir):
    """Small graphs for the op types outside the diffusion models: (dir, inputs, output name, exact?)."""
    rng = np.random.default_rng(7)
    out = []
    d = os.path.join(workdir, "g_maxpool") + "/"
    g = emit.GraphBuilder(d, "float32", seed=11)
    x = g.input("x", (1, 8, 12, 12))
    c = g.conv(x, 16, 3)
    g.node("MaxPool", [c], [(1, 16, 6, 6)], [("ceil_mode", "0"), ("dilations", "1,1"), ("kernel_shape", "2,2"), ("pads", "0,0,0,0"), ("strides", "2,2")], out_names=["poola"])
    g.node("MaxPool", [c], [(1, 16, 12, 12)], [("ceil_mode", "0"), ("dilations", "1,1"), ("kernel_shape", "5,5"), ("pads", "2,2,2,2"), ("strides", "1,1")], out_names=["poolb"])
    g.finish()
    xin = {"x": (rng.standard_normal((1, 8, 12, 12)) - 1.0).astype(np.float32)}
    out += [(d, xin, "poola", False), (d, xin, "poolb", False)]
    d = os.path.join(workdir, "g_trilu") + "/"
    g = emit.GraphBuilder(d, "float32", seed=12)
    m = g.input("m", (6, 7))
    t = g.node("Trilu", [m, g.const(np.asarray(1, dtype=np.int64))], [(6, 7)], [("upper", "1")])
    g.node("Mul", [t, g.scalar(2.0)], [(6, 7)], out_names=["tri"])
    g.finish()
    out.append((d, {"m": rng.standard_normal((6, 7)).astype(np.float32)}, "tri", True))
    d = os.path.join(workdir, "g_scatter") + "/"
    g = emit.GraphBuilder(d, "float32", seed=13)
    data = g.input("data", (4, 5))
    upd = g.input("upd", (2, 3))
    idx = np.asarray([[[0, 0], [1, 4], [3, 2]], [[2, 2], [0, 3], [3, 4]]], dtype=np.int64)
    sc = g.node("ScatterND", [data, g.const(idx), upd], [(4, 5)])
    g.node("Mul", [sc, g.scalar(1.0)], [(4, 5)], out_names=["scattered"])
    g.finish()
    out.append((d, {"data": rng.standard_normal((4, 5)).astype(np.float32), "upd": rng.standard_normal((2, 3)).astype(np.float32)}, "scattered", True))
    d = os.path.join(workdir, "g_argmax") + "/"
    g = emit.GraphBuilder(d, "float32", seed=14)
    v = g.input("v", (1, 9))
    g.node("ArgMax", [v], [(1,)], [("axis", "-1"), ("keepdims", "0")], out_names=["arg"])
    g.finish()
    out.append((d, {"v": np.asarray([[3, -1, 7, 7, 2, 7, 0, -5, 6]], dtype=np.int64)}, "arg", True))
    return out


def test_restatement_matches_reference_index_ops(workdir):
    """MaxPool / Trilu / ScatterND / ArgMax (src/onnxstream.cpp:8075, 7883, 7939, 6930): numpy restatement == the reference."""
    for d, inputs, name, exact in _index_graphs(workdir):
        ref = reference_outputs("index_" + os.path.basename(d.rstrip("/")), lambda lib: run_model(lib, d, inputs, ())[0])[name]
        got = NumpyOracle(d).run(inputs)[name]
        if exact:
            assert np.array_equal(np.asarray(got).ravel(), np.asarray(ref).ravel()), name
        else:
            assert report(golden_sample(got), ref)["rel_to_max"] <= 5e-5, name


def test_restatement_matches_reference_llama_decode(workdir):
    """BASELINE config[4] hot path at toy size (KV-cache decode step: Gather, rotary, RMSNorm, grouped-KV attention): numpy == reference."""
    cfg = emit.LlamaConfig.tiny()
    d = os.path.join(workdir, "llama_np") + "/"
    emit.emit_llama_decode(d, cfg, "float32")
    inputs = emit.llama_inputs(cfg)
    ref = reference_outputs("llama_tiny32", lambda lib: run_model(lib, d, inputs, ("use_scaled_dp_attn_op",))[0])["logits"]
    got = NumpyOracle(d).run(inputs)["logits"]
    assert report(got, ref)["rel_to_max"] <= 5e-5


def test_torch_exporter_block_matches_torch(workdir):
    """SURVEY section 8 f4: torch.nn.Module -> model.txt + blobs (onnxstream_b200/export_torch.py, no `onnx` package), executed by the
    reference itself, must reproduce torch: a UNet-style block with Conv, GroupNorm, SiLU, Gemm, LayerNorm, attention, GEGLU,
    Concat, nearest upsampling and a strided Conv."""
    import torch
    import torch.nn as nn
    import torch.nn.functional as F
    from onnxstream_b200.export_torch import export_module

    class Block(nn.Module):
        def __init__(s):
            super().__init__()
            s.c = nn.Conv2d(4, 32, 3, padding=1); s.g = nn.GroupNorm(8, 32); s.t = nn.Linear(16, 32); s.ln = nn.LayerNorm(32)
            s.q = nn.Linear(32, 32, bias=False); s.k = nn.Linear(32, 32, bias=False); s.v = nn.Linear(32, 32, bias=False); s.o = nn.Linear(32, 32)
            s.ff = nn.Linear(32, 256); s.ff2 = nn.Linear(128, 32); s.up = nn.Conv2d(64, 4, 3, padding=1); s.down = nn.Conv2d(4, 4, 3, stride=2, padding=1)

        def forward(s, x, temb):
            h = s.c(x)
            h = F.silu(s.g(h)) + s.t(F.silu(temb))[:, :, None, None]
            b, c, hh, ww = h.shape
            t = h.flatten(2).transpose(1, 2)
            n = s.ln(t)
            q, k, v = (f(n).view(b, -1, 4, 8).transpose(1, 2) for f in (s.q, s.k, s.v))
            t = t + s.o(F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(b, -1, 32))
            a1, gate = s.ff(t).chunk(2, dim=-1)
            t = t + s.ff2(a1 * F.gelu(gate))
            u = F.interpolate(torch.cat([t.transpose(1, 2).reshape(b, c, hh, ww), h], 1), scale_factor=2.0, mode="nearest")
            return s.down(s.up(u)) * 0.5

    torch.manual_seed(0)
    m = Block().eval()
    x, temb = torch.randn(1, 4, 6, 6), torch.randn(1, 16)
    ref = m(x, temb).detach().numpy()
    for wd, opts, tol in (("float32", (), 2e-5), ("float16", ("use_fp16_arithmetic", "fuse_ops_in_attention"), 2e-2)):
        d = os.path.join(workdir, "exp_block_" + wd) + "/"
        info = export_module(m, (x, temb), d, wd, input_names=["sample", "t_emb"], output_names=["out_sample"])
        assert info["inputs"] == ["sample", "t_5F_emb"] and info["outputs"] == ["out_5F_sample"]     # converter's name mangling
        feed = dict(zip(info["inputs"], [x.numpy(), temb.numpy()]))
        got = reference_outputs("export_block_" + wd, lambda lib: run_model(lib, d, feed, opts)[0])[info["outputs"][0]]
        assert got.shape == ref.shape and report(got, ref)["rel_to_max"] <= tol, wd
        if wd == "float16":
            # the exporter writes the attention block in the diffusers-export order: the engine's planner (host code, no GPU needed)
            # must claim it as one multi-head-attention group next to GroupNorm / LayerNorm / GEGLU
            from onnxstream_b200.model import plan_summary
            last = plan_summary(open(d + "model.txt").read()).splitlines()[-1]
            assert " MHA=1" in last and " GEGLU=1" in last and " GROUPNORM=1" in last and " LAYERNORM=1" in last, last
        # the numpy restatement agrees on the exported graph too
        if wd == "float32":
            npo = NumpyOracle(d).run(dict(zip(info["inputs"], [x.numpy(), temb.numpy()])))[info["outputs"][0]]
            assert report(npo, ref)["rel_to_max"] <= 2e-5


def test_torch_exporter_transformers_models(workdir):
    """Real library architectures with random weights: transformers' CLIPTextModel (causal-masked attention, quick-GELU) and
    LlamaForCausalLM (RMSNorm, rotary, grouped KV heads) exported without `onnx` and run by the reference: logits == torch."""
    import torch
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
        d = os.path.join(workdir, "exp_" + name) + "/"
        info = export_module(w, (ids,), d, "float32", input_names=["input_ids"], output_names=[out])
        ref = w(ids).detach().numpy()
        feed = {info["inputs"][0]: ids.numpy().astype(np.int64)}
        got = reference_outputs("export_%s_float32" % name, lambda lib: run_model(lib, d, feed)[0])
        assert got.shapes[info["outputs"][0]] == ref.shape and report(got[info["outputs"][0]], golden_sample(ref))["rel_to_max"] <= 2e-5, name
        # three-way: the numpy restatement agrees with torch (and hence with the reference) on the same export
        assert report(NumpyOracle(d).run(feed)[info["outputs"][0]], ref)["rel_to_max"] <= 2e-5, name
        # fp16 weights + fp16 arithmetic in the reference stays within the fp16 bar of torch's fp32 forward
        d16 = os.path.join(workdir, "exp16_" + name) + "/"
        info16 = export_module(w, (ids,), d16, "float16", input_names=["input_ids"], output_names=[out])
        got16 = reference_outputs("export_%s_float16" % name, lambda lib: run_model(lib, d16, feed, ("use_fp16_arithmetic", "fuse_ops_in_attention"))[0])[info16["outputs"][0]]
        assert report(got16, golden_sample(ref))["rel_to_max"] <= 2e-2, name


def test_planner_fusion_on_cpu(engine_lib, workdir):
    """The engine's planner is host code and runs without a GPU (model_b200_plan_summary): every diffusers-export pattern of a
    UNet-shaped graph must be claimed by a fusion group, and switching the fusions off must give one step per op."""
    from onnxstream_b200.model import plan_summary
    g = emit.emit_unet(None, emit.UNetConfig.tiny(16), "float16", keep_in_memory=True)
    text = g.text()
    rep = plan_summary(text, library_path=engine_lib)
    steps = [l.split(" ", 3) for l in rep.splitlines() if l and not l.startswith("#")]
    summary = dict(kv.split("=") for kv in rep.splitlines()[-1].split()[1:])
    n_ops = len([l for l in text.splitlines() if l])
    assert int(summary["ops"]) == n_ops and sum(int(s[1]) for s in steps) == n_ops       # the groups partition the op list
    blocks = int(summary["GEGLU"])                                                          # one GEGLU feed-forward per transformer block
    assert blocks > 0 and int(summary["MHA"]) == 2 * blocks and int(summary["LAYERNORM"]) == 3 * blocks
    # nothing that belongs to a pattern is left to run as a single op
    leftovers = {s[2] for s in steps if s[0] == "SINGLE"}
    assert not (leftovers & {"Softmax", "Erf", "InstanceNormalization", "Sigmoid", "Pow", "ReduceMean", "Sqrt", "Slice"}), leftovers
    # every resnet output conv takes its residual in the epilogue; every GroupNorm is one group (with or without SiLU)
    assert int(summary["CONV_ADD"]) > 0 and int(summary["GROUPNORM"]) > 0
    # fusion off: the reference's op-by-op schedule
    rep0 = plan_summary(text, fuse_nodes=False, fuse_attention=False, library_path=engine_lib)
    assert int(dict(kv.split("=") for kv in rep0.splitlines()[-1].split()[1:])["steps"]) == n_ops
    # an LLM decode graph: the ScaledDotProductAttention rewrite windows are found
    d = os.path.join(workdir, "llama_plan") + "/"
    emit.emit_llama_decode(d, emit.LlamaConfig.tiny(), "float32")
    repl = plan_summary(open(d + "model.txt").read(), fp16_arithmetic=False, use_scaled_dp_attn_op=True, library_path=engine_lib)
    assert "SDPA=%d" % emit.LlamaConfig.tiny().layers in repl.splitlines()[-1]
    # ... and so are the decode-block groups: RMSNorm (7 ops, 2 per layer + the final one), rotary embedding (7 ops, q and k), the grouped
    # q/k/v projections (3 MatMuls sharing their input), the gated MLP (MatMul, Sigmoid, Mul, MatMul, Mul) and the two bias-free
    # projections whose residual Add rides in the GEMV epilogue; the groups still partition the op list
    L = emit.LlamaConfig.tiny().layers
    suml = dict(kv.split("=") for kv in repl.splitlines()[-1].split()[1:])
    assert int(suml["RMSNORM"]) == 2 * L + 1 and int(suml["ROPE"]) == 2 * L and int(suml["GEMV_GROUP"]) == L and int(suml["SWIGLU"]) == L and int(suml["LINEAR"]) == 2 * L, suml
    stepsl = [l.split(" ", 3) for l in repl.splitlines() if l and not l.startswith("#")]
    assert sum(int(t[1]) for t in stepsl) == int(suml["ops"])
    assert {t[1] for t in stepsl if t[0] == "GEMV_GROUP"} == {"3"} and {t[1] for t in stepsl if t[0] == "SWIGLU"} == {"5"}
    assert not ({t[2] for t in stepsl if t[0] == "SINGLE"} & {"Pow", "ReduceMean", "Sqrt", "Slice", "Neg", "Sigmoid"})
    # a prompt-shaped graph (16 rows per MatMul) keeps plain MatMuls: the GEMV groups are for decode
    # (rows > 8 is checked on the static shapes of model.txt)
    with pytest.raises(Exception):
        plan_summary("not a model line", library_path=engine_lib)


def test_golden_vectors():
    """tests/golden/*.npz were produced by tests/golden/make_golden.py from oracle/_ref; the restatement, and the reference
    where oracle/_ref is built, must still reproduce them (guards the emitter, the oracle build and the restatement against
    silent drift)."""
    files = sorted(f for f in os.listdir(GOLDEN) if f.endswith(".npz"))
    assert files, "no golden fixtures committed"
    sys.path.insert(0, GOLDEN)
    import make_golden
    for f in files:
        z = np.load(os.path.join(GOLDEN, f))
        case = f[:-4]
        with tempfile.TemporaryDirectory() as d:
            d = d + "/"
            inputs, out_name, fp16 = make_golden.build_case(case, d)
            opts = ("use_fp16_arithmetic", "fuse_ops_in_attention") if fp16 else ()
            if os.path.exists(ORACLE):
                ref = run_model(ORACLE, d, inputs, opts)[0][out_name]
                assert report(ref, z["output"])["rel_to_max"] <= (2e-3 if fp16 else 1e-5), case
            got = NumpyOracle(d, fp16=fp16).run(inputs)[out_name]
            assert report(got, z["output"])["rel_to_max"] <= (1e-2 if fp16 else 5e-5), case


def test_quantizer_rule():
    """onnx2txt.ipynb cell 1 `quantize`: percentile range, zero point = floor(|lo| / scale), scalar special case."""
    a = np.linspace(-1.0, 3.0, 10001).astype(np.float32)
    q, scale, zp = emit.quantize_uint8(a)
    lo, hi = np.sort(a)[10], np.sort(a)[-11]
    assert abs(scale - (hi - lo) / 255.0) < 1e-7 and zp == int(abs(lo) / scale)
    assert q.dtype == np.uint8 and q.min() == 0 and q.max() >= 254
    q, scale, zp = emit.quantize_uint8(np.asarray(-0.5, np.float32))
    assert (float(q) - zp) * scale == -0.5


def test_parser_roundtrip(workdir):
    d, inputs, out = _archs(workdir)["unet"]
    ops = parse_model(open(d + "model.txt").read())
    assert ops[-1]["outputs"][0]["name"] == out
    conv = next(o for o in ops if o["type"] == "Conv")
    assert conv["inputs"][1]["name"].endswith("_nchw.bin") and os.path.exists(d + conv["inputs"][1]["name"].replace("_nchw", "_nhwc"))


def test_capi_exports_every_declared_symbol(engine_lib):
    lib = ctypes.CDLL(engine_lib)
    names = []
    for h in ("onnxstream_b200.h", "onnxstream_b200_kernels.h"):
        text = open(os.path.join(ROOT, "include", h)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names += re.findall(r"\b((?:model|osb)_[a-z0-9_]+)\s*\(", text)
    assert len(set(names)) >= 40
    missing = [n for n in sorted(set(names)) if not hasattr(lib, n)]
    assert not missing, missing


def test_no_cpu_fallback(engine_lib):
    """Without a CUDA device the library loads but model_new_2 must fail loudly -- there is no CPU path to fall back to."""
    code = ("import ctypes,sys; l=ctypes.CDLL(%r); l.model_new_2.restype=ctypes.c_void_p; "
            "h=l.model_new_2(0,b'nocache'); print('HANDLE', h)" % engine_lib)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert "HANDLE None" in r.stdout, r.stdout + r.stderr
    assert "no CUDA device" in r.stderr


def test_product_does_not_import_oracle():
    bad = []
    for base, _, files in os.walk(os.path.join(ROOT, "onnxstream_b200")):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".h", ".cuh")):
                t = open(os.path.join(base, f), errors="ignore").read()
                if re.search(r"(import\s+np_oracle|from\s+oracle|oracle/_ref|liboracle_ref|xnn_shim)", t):
                    bad.append(f)
    assert not bad, bad


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    import bench                                   # reads RANK / WORLD_SIZE from the environment at import

    class StubLib:                                 # the two comm entry points of the engine library, without a GPU
        def __init__(self):
            self.joined = None

        def osb_comm_unique_id(self, buf):
            buf.raw = bytes((7 * i + rank) % 256 for i in range(128))      # only rank 0's id may survive
            return 0

        def osb_comm_init(self, world_, rank_, uid):
            self.joined = (world_, rank_, bytes(uid))
            return 0x1234

    lib = StubLib()
    comm = bench.make_comm(lib, dist)
    agg_t = bench.dist_max(dist, 1.0 + rank)       # time = max over ranks
    arr = bench.dist_bcast_array(dist, np.arange(6, dtype=np.float32).reshape(2, 3) if rank == 0 else None)
    inputs = bench.make_workload("tiny_unet_fp16").inputs(rank)           # rank r = sample r
    q.put((rank, comm, lib.joined, agg_t, arr.tolist(), float(inputs["sample"].sum())))
    dist.destroy_process_group()


def test_multi_rank_host_logic_gloo():
    """world_size-2 gloo run of the host-side N > 1 logic of bench.py itself: the NCCL-id exchange that bootstraps the engine's communicator
    (make_comm -> onnxstream_b200/multi.py), max-over-ranks timing, the reference-output broadcast, rank -> sample mapping."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + os.getpid() % 1000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(60)
    rank0_id = bytes((7 * i) % 256 for i in range(128))
    for r, (rank, comm, joined, agg_t, arr, ssum) in enumerate(res):
        assert rank == r and comm == 0x1234
        assert joined == (2, r, rank0_id)                  # every rank joined with rank 0's id
        assert agg_t == pytest.approx(2.0)                 # max over ranks of (1 + rank)
        assert arr == [[0.0, 1.0, 2.0], [3.0, 4.0, 5.0]]
    assert res[0][5] != res[1][5]                           # different samples per rank


def test_qu8_restatement_bit_exact(tmp_path):
    """Pins oracle/np_oracle.py's uint8 restatement (percentile quantisation of the inputs, XNNPACK qu8 add / multiply / fully-connected,
    dequantisation) BIT-EXACT to the reference run: m_use_uint8_arithmetic on a graph of Add, Mul and MatMul with m_range_data.  The
    XNNPACK kernels behind these ops in oracle/_ref are the real library (not the shim)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import np_oracle as npo
    from onnxstream_b200 import emit
    d = str(tmp_path) + "/"
    g = emit.GraphBuilder(d, "uint8", seed=21)
    a_t, b_t = g.input("a", (1, 40, 48)), g.input("b", (1, 40, 48))
    s_t = g.node("Add", [a_t, b_t], [(1, 40, 48)], name="addop")
    p_t = g.node("Mul", [a_t, b_t], [(1, 40, 48)], name="mulop")
    y_t = g.linear(s_t, 32, bias=False, name="fcop")
    g.mark_output(p_t); g.mark_output(y_t)
    g.finish()
    rng = np.random.default_rng(1)
    a = rng.standard_normal((1, 40, 48)).astype(np.float32)
    b = (rng.standard_normal((1, 40, 48)) * 2 + 0.5).astype(np.float32)
    ranges = {"addop": (-5.0, 6.0), "mulop": (-8.0, 9.0), "fcop": (-7.0, 7.5)}
    out = reference_outputs("qu8_restatement", lambda lib: run_model(lib, d, {"a": a, "b": b}, ("use_uint8_arithmetic",), ranges=ranges, extra_outputs=[s_t.name])[0])
    sa, za = npo.qu8_range_to_scale(*npo.qu8_percentiles(a, 4))
    sb, zb = npo.qu8_range_to_scale(*npo.qu8_percentiles(b, 4))
    qa, qb = npo.qu8_quantize(a, sa, za), npo.qu8_quantize(b, sb, zb)
    so, zo = npo.qu8_range_to_scale(*ranges["addop"]); sm, zm = npo.qu8_range_to_scale(*ranges["mulop"]); sf, zf = npo.qu8_range_to_scale(*ranges["fcop"])
    qs = npo.qu8_add(qa, sa, za, qb, sb, zb, so, zo)
    assert np.array_equal(golden_sample(npo.qu8_dequantize(qs, so, zo)), out[s_t.name])
    assert np.array_equal(golden_sample(npo.qu8_dequantize(npo.qu8_mul(qa, sa, za, qb, sb, zb, sm, zm), sm, zm)), out[p_t.name])
    import re
    line = [l for l in open(d + "model.txt").read().splitlines() if l.startswith("fcop:")][0]
    m = re.search(r"(\w+\.bin)\(uint8\[([^,]+),(\d+)\]:48,32\)", line)
    qw = np.fromfile(d + m.group(1), np.uint8).reshape(48, 32)
    sw, zw = np.float32(float(m.group(2))), int(m.group(3))
    qy = npo.qu8_gemm(qs.reshape(40, 48), so, zo, qw, sw, zw, sf, zf)
    assert np.array_equal(golden_sample(npo.qu8_dequantize(qy, sf, zf).reshape(1, 40, 32)), out[y_t.name])


def test_planner_side_branch_and_gn_statistics(engine_lib, tmp_path):
    """Host-side planning of the two round-2 schedule changes, on the SD-UNet topology (no GPU needed):
      * side branch: the time-embedding MLP, every resnet's time_emb_proj chain and the cross-attention K / V projections do not depend on
        the latent (the graph input that starts the longest op chain) -> hoisted to the second stream;
      * GroupNorm statistics: every GroupNorm fed by the step right before it (conv, conv + residual, per-channel time-embedding add)
        gets them from that producer instead of a pass of its own."""
    from onnxstream_b200.model import plan_summary
    d = str(tmp_path) + "/"
    cfg = emit.UNetConfig.tiny(8)
    emit.emit_unet(d, cfg, "float16", seed=0)
    # the side-branch schedule is opt-in (OSB_SIDE_BRANCH=1, read once per process): plan in a child process
    code = ("import sys; sys.path.insert(0, %r); from onnxstream_b200.model import plan_summary; "
            "sys.stdout.write(plan_summary(open(%r).read(), library_path=%r))" % (ROOT, d + "model.txt", engine_lib))
    rep = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, OSB_SIDE_BRANCH="1"), stdout=subprocess.PIPE, text=True, check=True).stdout
    lines = rep.splitlines()
    summ = dict(kv.split("=") for kv in lines[-1].split()[1:])
    n_resnets = sum(1 for l in lines if l.startswith("SINGLE 1 Gemm") and "[side]" in l) - 2      # 2 = the time-embedding MLP itself
    assert n_resnets >= 6, rep[-2000:]
    assert int(summ["side"]) >= 3 * n_resnets                      # SiLU + Gemm + Unsqueeze(s) per resnet
    n_cross = sum(1 for l in lines if l.startswith("MHA") and "[kv-side]" in l)
    n_mha = sum(1 for l in lines if l.startswith("MHA"))
    assert n_mha >= 2 and n_cross == n_mha // 2, (n_mha, n_cross)   # every transformer block: one self- and one cross-attention
    assert not any("[side]" in l and l.startswith(("CONV_ADD", "GROUPNORM", "MHA")) for l in lines)
    n_gn = int(summ["GROUPNORM"])
    assert int(summ["gn_stats_producers"]) >= n_gn // 2, (summ, n_gn)
    # a graph with a single input has no side branch
    vd = str(tmp_path) + "/vae/"
    emit.emit_vae_decoder(vd, emit.VAEConfig.tiny(8), "float16")
    assert "side=" not in plan_summary(open(vd + "model.txt").read(), library_path=engine_lib).splitlines()[-1]


def test_tiled_vae_geometry_and_blend():
    """sd.cpp's tile walk (src/sd.cpp:1325-1340, 2478-2499) and feather blend (1296-1322) restated in onnxstream_b200/tiled_vae.py: the
    origins for the reference's three cases, and the blend against a direct transcription of the reference's scalar loop."""
    from onnxstream_b200 import tiled_vae as tv
    assert tv.tile_origins(64) == [0, 24, 32]                  # SD 1.5 512x512: 3 x 3 tiles
    assert tv.tile_origins(128) == [0, 24, 48, 72, 96]         # SDXL 1024x1024: 5 x 5 = 25 tiles
    assert tv.tile_origins(32) == [0] and tv.tile_origins(40) == [0, 8]
    rng = np.random.default_rng(0)
    canvas = rng.standard_normal((3, 96, 96)).astype(np.float32)
    ref = canvas.copy()
    tile = rng.standard_normal((3, 64, 64)).astype(np.float32)
    dx, dy, ramp = 32, 16, 8
    for c in range(3):
        for y in range(64):
            for x in range(64):
                f = np.float32(1)
                if dy and y < ramp:
                    f = np.float32(y) / np.float32(ramp)
                if dx and x < ramp:
                    f = f * (np.float32(x) / np.float32(ramp))
                ref[c, dy + y, dx + x] = tile[c, y, x] * f + ref[c, dy + y, dx + x] * (np.float32(1) - f)
    tv.blend_tile(canvas, tile, dx, dy, ramp)
    assert np.array_equal(canvas, ref)
