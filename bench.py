#!/usr/bin/env python
"""bench.py -- the BASELINE.json workloads of the B200 OnnxStream engine, one JSON line per run.

Default workload (what the driver runs): SD 1.5 UNet 512x512 bs=1 denoise-step throughput (BASELINE config[1] hot path).
One "step" = one UNet Model::run() on one 4x64x64 latent (the reference runs two per sampler step with CFG; the metric counts
UNet runs).  fp16 weights / fp16 arithmetic / attention fusion, i.e. what sd.cpp sets (src/sd.cpp:1616-1683).  Synthetic
graphs of the named architectures + seeded random weights (no checkpoints offline).

  value   : units/s with weights and inputs resident in HBM (one captured CUDA graph per step where the graph has no int64
            inputs), CUDA-event timed on the compute stream
  e2e     : the same metric through the reference-facing C ABI with HOST buffers: every step pushes the inputs from pinned host
            memory, streams ALL weights pinned-host -> HBM ring (the CUDA WeightsProvider; N>1: every rank uploads 1/N of each
            node over its own PCIe link and an NCCL all-gather over NVLink completes the ring slot) and reads the output back
  roofline: the dominant kernel (tcgen05 implicit-GEMM conv / GEMM) timed per launch with CUDA events in an eager pass
  cpu_baseline / --impl reference: the reference's own CPU path (oracle/_ref: unmodified reference sources + XNNPACK), FULL
            graph runs on the host cores (no prefix extrapolation for the default workload)
  parity  : every rank checks its streamed output against its resident-weights output, and one common sample against the
            reference's output (oracle/_ref, cached per box); the max over ranks is in the line

Other workloads (`--workload`): sdxl_unet_w8 (SDXL 1024x1024, uint8 weights; N=2 = the CFG cond/uncond pair), sdxl_turbo_w8
(512x512, one sample per GPU), vae_decoder_fp16, clip_text_fp32, sd15_pipeline (text encoder + 20 CFG steps + VAE decoder),
tinyllama_decode (seq 2048).  `--all-configs FILE` runs them all and writes one line each.

`--dump-outputs DIR` writes what the value arm computed in its last timed step -- every output tensor a caller of that
path receives -- as DIR/<tensor>.npy (float32, float64 for int64 outputs; sd15_pipeline: DIR/<workload>.<tensor>.npy), at
most 64 MB in all.  Inputs and weights are seeded, so two builds run on the same arguments can be compared output for output.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RANK = int(os.environ.get("RANK", "0"))
LOCAL_RANK = int(os.environ.get("LOCAL_RANK", "0"))
WORLD = int(os.environ.get("WORLD_SIZE", "1"))
if WORLD > 1 and "OSB_KEEP_VISIBLE" not in os.environ:
    # one process per GPU: each rank sees exactly its own device as device 0 (engine and torch alike)
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    devs = vis.split(",") if vis else [str(i) for i in range(64)]
    os.environ["CUDA_VISIBLE_DEVICES"] = devs[LOCAL_RANK]

# The contract is ONE JSON line on stdout: native libraries (NCCL prints its version banner) must not pollute it, so
# fd 1 points at stderr while the bench runs and the line is written to the saved descriptor at the end.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit_line(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


import numpy as np  # noqa: E402

from onnxstream_b200 import emit  # noqa: E402
from onnxstream_b200.model import Model, ENGINE_LIB  # noqa: E402

ORACLE_LIB = os.path.join(ROOT, "oracle", "_ref", "liboracle_ref.so")
HOST_CORES = os.cpu_count() or 1
# XNNPACK's pthreadpool with one worker per core is far slower than a moderate pool on many-core hosts (measured r01: 128
# workers -> 295 s per UNet run on the GPU box, vs 38 s with 8 on an 8-core host), so the reference gets min(cores, 32).
REF_THREADS = min(HOST_CORES, 32)
# torchrun exports OMP_NUM_THREADS=1 to every rank: ASSIGN (the oracle's shim loops are OpenMP; the engine does not use OpenMP)
os.environ["OMP_NUM_THREADS"] = str(REF_THREADS)
SHM = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
REF_CACHE = os.path.join(SHM, "osb200_ref_cache")

FP16 = ("use_fp16_arithmetic", "fuse_ops_in_attention")
DUMP_LIMIT_BYTES = 64 << 20


# =====================================================================================================================
# workloads
# =====================================================================================================================
class Workload:
    name = ""
    metric = ""
    unit = "steps/s"
    out_name = "out_5F_sample"
    options = FP16
    ref_options = ("fuse_ops_in_attention",)   # fp16 weights, fp32 XNNPACK arithmetic: the reference's --rpi mode (src/sd.cpp:1636-1638)
    dtype = "f16"
    tol = 3e-2            # |engine - reference| <= tol * max|reference| (fp16 arithmetic vs fp32 arithmetic on fp16 weights)
    describe = ""
    upcast = ()

    hbm_bound = False     # True: the step is weight-bandwidth bound (M = 1 GEMVs): the roofline is HBM GB/s over the whole step

    def emit(self, d):
        raise NotImplementedError

    def inputs(self, seed):
        raise NotImplementedError

    def engine_setup(self, m, resident):
        """Extra engine options for this workload (called before read_file)."""

    def later_inputs(self, inputs):
        """Inputs the host pushes on every run after the first (default: all of them)."""
        return inputs


class SD15UNet(Workload):
    name = "sd15_unet_fp16"
    metric = "SD1.5 UNet 512x512 bs=1 denoise steps/s (one UNet Model::run per step)"

    def __init__(self, latent=64):
        self.cfg = emit.UNetConfig.sd15(latent)
        self.describe = "SD1.5 UNet-shaped graph (BASELINE config[1] hot path), 4x%dx%d latent, 77x768 context, fp16 weights + fp16 arithmetic (fp32 accumulate)" % (latent, latent)

    def emit(self, d):
        return emit.emit_unet(d, self.cfg, "float16", seed=0)

    def inputs(self, seed):
        return emit.unet_inputs(self.cfg, seed=seed)


class SD15UNetFP32(SD15UNet):
    """BASELINE config[0]: the SD 1.5 UNet step in fp32 (fp32 blobs, fp32 arithmetic -- the reference's default CPU mode).  On the B200 engine
    every Conv / MatMul / Gemm runs on the tensor cores through the bf16 triple split (fp32-faithful); the reference arm is the same graph and
    blobs through XNNPACK f32."""
    name = "sd15_unet_fp32"
    metric = "SD1.5 UNet 512x512 bs=1 fp32 denoise steps/s (one UNet Model::run per step)"
    options = ("fuse_ops_in_attention",)
    ref_options = ("fuse_ops_in_attention",)
    dtype = "f32"
    tol = 2e-4

    def __init__(self, latent=64):
        super().__init__(latent)
        self.describe = "SD1.5 UNet-shaped graph (BASELINE config[0]), 4x%dx%d latent, 77x768 context, fp32 weights + fp32 arithmetic (tensor cores via bf16 triple split)" % (latent, latent)

    def emit(self, d):
        return emit.emit_unet(d, self.cfg, "float32", seed=0)


class TinyUNet(SD15UNet):
    name = "tiny_unet_fp16"
    metric = "tiny UNet steps/s (plumbing check)"

    def __init__(self):
        self.cfg = emit.UNetConfig.tiny(16)
        self.describe = "tiny SD-UNet-shaped graph, 16x16 latent"


class SDXLUNet(Workload):
    """SDXL base UNet, uint8 weights (the reference's W8A32 storage, onnx2txt percentile rule), sd.cpp's default arithmetic flags
    (m_use_fp16_arithmetic: blobs are dequantised on the device into fp16 operands, fp32 accumulate).  BASELINE config[2]:
    1024x1024, the CFG cond/uncond pair = 2 UNet runs per sampler step, one per GPU at N=2."""
    name = "sdxl_unet_w8"
    metric = "SDXL UNet 1024x1024 steps/s (one UNet Model::run per step; N=2 = the CFG cond/uncond pair)"
    tol = 4e-2

    def __init__(self, latent=128, name=None, metric=None):
        self.cfg = emit.UNetConfig.sdxl(latent)
        if name:
            self.name = name
        if metric:
            self.metric = metric
        px = latent * 8
        self.describe = "SDXL-UNet-shaped graph, 4x%dx%d latent (%dx%d px), 77x2048 context, time_ids/text_embeds add-embedding, uint8 weights dequantised on the device, fp16 arithmetic" % (latent, latent, px, px)

    def emit(self, d):
        return emit.emit_unet(d, self.cfg, "uint8", seed=0)

    def inputs(self, seed):
        return emit.unet_inputs(self.cfg, seed=seed)


class VAEDecoder(Workload):
    name = "vae_decoder_fp16"
    metric = "SD1.5 VAE decoder 64x64 -> 512x512 decodes/s"
    unit = "decodes/s"
    out_name = "outsample"
    options = FP16
    ref_options = ()

    def __init__(self):
        self.cfg = emit.VAEConfig()
        self.describe = "SD VAE-decoder-shaped graph, 4x64x64 latent -> 3x512x512, fp16 weights + fp16 arithmetic"

    def emit(self, d):
        return emit.emit_vae_decoder(d, self.cfg, "float16")

    def inputs(self, seed):
        return {"input_2E_1": np.random.default_rng(5 + seed).standard_normal((1, 4, self.cfg.latent, self.cfg.latent)).astype(np.float32)}


class CLIPText(Workload):
    name = "clip_text_fp32"
    metric = "CLIP text encoder (12 layers, 768 wide, 77 tokens) runs/s"
    unit = "runs/s"
    out_name = "last_5F_hidden_5F_state"
    options = ()
    ref_options = ()
    dtype = "f32"
    tol = 2e-4

    def __init__(self):
        self.cfg = emit.CLIPConfig()
        self.describe = "CLIP-text-encoder-shaped graph, fp32 (what sd.cpp runs the text encoder in)"

    def emit(self, d):
        return emit.emit_text_encoder(d, self.cfg, "float32")

    def inputs(self, seed):
        return {"input_5F_ids": np.random.default_rng(6 + seed).integers(0, self.cfg.vocab, (1, self.cfg.tokens)).astype(np.int64)}


class LlamaDecode(Workload):
    """TinyLlama-1.1B-shaped single-token decode at sequence 2048 (2047 cached positions), fp16 as llm.cpp ships it (src/llm.cpp:377)."""
    name = "tinyllama_decode"
    metric = "TinyLlama-1.1B decode tokens/s at seq 2048 (one Model::run per token)"
    unit = "tokens/s"
    out_name = "logits"
    options = ("use_fp16_arithmetic", "use_scaled_dp_attn_op")
    ref_options = ("use_scaled_dp_attn_op",)
    upcast = ("layernorm", "/norm/")
    hbm_bound = True
    wdtype = "float16"

    def __init__(self, tiny=False, w8=False):
        self.cfg = emit.LlamaConfig.tiny() if tiny else emit.LlamaConfig()
        if w8:
            self.wdtype = "uint8"
            self.name = "tinyllama_decode_w8"
            self.metric = "TinyLlama-1.1B decode tokens/s at seq 2048, uint8 weights (dequantised in registers, fp16 arithmetic)"
            self.tol = 5e-2
        self.describe = "Llama-shaped decode graph: %d layers, hidden %d, %d/%d heads, vocab %d, %d cached positions, %s weights; KV cache resident in HBM" % (
            self.cfg.layers, self.cfg.hidden, self.cfg.heads, self.cfg.kv_heads, self.cfg.vocab, self.cfg.past, self.wdtype)

    def emit(self, d):
        return emit.emit_llama_decode(d, self.cfg, self.wdtype)

    def engine_setup(self, m, resident):
        if resident:
            # the KV cache of a fixed-shape decode step lives in HBM: pushed once, reused by name; only logits come back
            m.lib.model_set_option(m.h, b"b200_keep_inputs", 1)
            m.lib.model_ext_add_output_convert(m.h, b"logits")
            m.lib.model_set_option(m.h, b"b200_drop_unconverted_outputs", 1)

    def later_inputs(self, inputs):
        return {k: v for k, v in inputs.items() if not k.startswith("pkv")}

    def inputs(self, seed):
        return emit.llama_inputs(self.cfg, seed=seed)


def make_workload(name):
    if name == "sd15_unet_fp16":
        return SD15UNet()
    if name == "sd15_unet_fp32":
        return SD15UNetFP32()
    if name == "tiny_unet_fp16":
        return TinyUNet()
    if name == "sdxl_unet_w8":
        return SDXLUNet(128)
    if name == "sdxl_turbo_w8":
        return SDXLUNet(64, "sdxl_turbo_w8", "SDXL Turbo UNet 512x512 1-step samples/s (one sample per GPU, shared streamed weights)")
    if name == "vae_decoder_fp16":
        return VAEDecoder()
    if name == "clip_text_fp32":
        return CLIPText()
    if name == "tinyllama_decode":
        return LlamaDecode()
    if name == "tinyllama_decode_w8":
        return LlamaDecode(w8=True)
    raise SystemExit(f"unknown workload {name}")


WORKLOADS = ["sd15_unet_fp16", "sd15_unet_fp32", "tiny_unet_fp16", "sdxl_unet_w8", "sdxl_turbo_w8", "vae_decoder_fp16", "clip_text_fp32", "tinyllama_decode", "tinyllama_decode_w8", "sd15_pipeline"]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1450.4), d.get("hbm_gbs", 6567.7), "measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def model_dir(workload: str) -> str:
    return os.path.join(SHM, f"osb200_bench_{workload}") + "/"


def ensure_model(w: Workload):
    """Emit the synthetic model directory once per box (rank 0), return (dir, meta)."""
    d = model_dir(w.name)
    meta = os.path.join(d, "meta.json")
    if not os.path.exists(meta):
        if RANK == 0:
            g = w.emit(d)
            json.dump({"flops": g.flops, "weight_bytes": g.weight_bytes, "params": g.weight_params, "ops": len(g.lines)}, open(meta + ".tmp", "w"))
            os.replace(meta + ".tmp", meta)
        else:
            while not os.path.exists(meta):
                time.sleep(0.5)
    return d, json.load(open(meta))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self):
        self.rows = []
        self.proc = None

    def start(self):
        try:
            q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0], f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# =====================================================================================================================
# torch.distributed plumbing (NCCL; one process per GPU)
# =====================================================================================================================
def dist_setup():
    if WORLD == 1:
        return None
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(0)
    import datetime
    # a rank that dies or skips a collective must not hold the others (and the GPU box) for NCCL's default 10 minutes
    dist.init_process_group("nccl", device_id=torch.device("cuda", 0), timeout=datetime.timedelta(seconds=int(os.environ.get("OSB_DIST_TIMEOUT_S", "300"))))
    return dist


def dist_device(dist) -> str:
    """Tensors of a collective live where the backend runs: NCCL on the GPU, gloo (the CPU tests of this host logic) on the host."""
    return "cuda" if str(dist.get_backend()).lower() == "nccl" else "cpu"


def dist_max(dist, x: float) -> float:
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=dist_device(dist))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def make_comm(lib, dist):
    """The engine library's own NCCL communicator (weight all-gather / broadcast), bootstrapped over the torch.distributed group:
    rank 0 creates the 128-byte ncclUniqueId, every rank receives it (onnxstream_b200/multi.py) and joins."""
    from onnxstream_b200 import multi

    def make_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        assert lib.osb_comm_unique_id(buf) == 0
        return bytes(buf.raw)

    uid = multi.exchange_unique_id(dist, RANK, make_id)
    comm = lib.osb_comm_init(WORLD, RANK, uid)
    assert comm, "ncclCommInitRank failed"
    return comm


def dist_barrier(dist):
    if dist is not None:
        import torch
        dist.barrier()
        torch.cuda.synchronize()


def dist_bcast_array(dist, arr, src=0):
    """Broadcast a float32 numpy array from rank `src` (shape known to every rank through `arr.shape` on src only)."""
    if dist is None:
        return arr
    obj = [arr if RANK == src else None]
    dist.broadcast_object_list(obj, src=src)
    return obj[0]


# =====================================================================================================================
# engine / reference drivers (both through the reference's C ABI)
# =====================================================================================================================
def make_engine_model(d, w: Workload, wp, resident, graph, comm=None):
    m = Model(ENGINE_LIB, 0, wp)
    for o in w.options:
        m.set_option(o, True)
    for p in w.upcast:
        m.add_upcast_pattern(p)
    m.lib.model_set_option(m.h, b"b200_resident_weights", 1 if resident else 0)
    m.lib.model_set_option(m.h, b"b200_cuda_graph", 1 if graph else 0)
    w.engine_setup(m, resident)
    if comm is not None:
        m.lib.model_b200_set_comm(m.h, comm, RANK, WORLD)
    m.read_file(d + "model.txt")
    return m


def step_api(m, inputs, out_name):
    m.clear_tensors()
    for k, v in inputs.items():
        m.add_tensor(k, v)
    m.run()
    return m.get_tensor(out_name) if out_name else None


def oracle_set_threads(n):
    lib = ctypes.CDLL(ORACLE_LIB)     # dlsym through the oracle's own dependencies reaches the libgomp it links
    lib.omp_set_num_threads(int(n))


def make_reference_model(d, w: Workload, model_file="model.txt"):
    oracle_set_threads(REF_THREADS)
    m = Model(ORACLE_LIB, REF_THREADS, "nocache")
    for o in w.ref_options:
        m.set_option(o, True)
    m.read_file(d + model_file)
    return m


def reference_output_cached(d, w: Workload, inputs, allow_compute=True):
    """One FULL run of the reference on `inputs`, cached per box (shared with tests/test_fullsize_gpu.py's cache layout).
    Returns (output, seconds or None when served from the cache)."""
    h = hashlib.sha1()
    h.update(open(d + "model.txt", "rb").read())
    for k in sorted(inputs):
        h.update(k.encode()); h.update(np.ascontiguousarray(inputs[k]).tobytes())
    h.update(repr((tuple(w.ref_options), w.out_name, "bench")).encode())
    os.makedirs(REF_CACHE, exist_ok=True)
    fn = os.path.join(REF_CACHE, h.hexdigest() + ".npy")
    if os.path.exists(fn):
        return np.load(fn), None
    if not allow_compute:
        raise RuntimeError("one full reference run of this graph takes minutes on the host cores: skipped here (this topology is checked at a smaller latent in tests/test_fullsize_gpu.py)")
    m = make_reference_model(d, w)
    t = time.time()
    out = step_api(m, inputs, w.out_name)
    dt = time.time() - t
    m.close()
    np.save(fn + ".tmp.npy", out)
    os.replace(fn + ".tmp.npy", fn)
    return out, dt


def model_lines_flops(d):
    """Per-line FLOPs of Conv / MatMul / Gemm ops of a model.txt (for bounded CPU samples of the large workloads)."""
    out = []
    for line in open(d + "model.txt").read().splitlines():
        if not line:
            continue
        typ = line.split("*", 1)[0].split(":")[1]
        fl = 0
        if typ in ("Conv", "MatMul", "Gemm"):
            ins = line.split("*input:")[1].split("*output:")[0].split(";")
            outs = line.split("*output:")[1].split("*")[0].split(";")

            def shape(t):
                s = t[t.index("(") + 1:-1]
                s = s.split(":")[-1]
                return [int(x) for x in s.split(",") if x]
            o = shape(outs[0])
            if typ == "Conv":
                wsh = shape(ins[1])
                fl = 2 * int(np.prod(o)) * wsh[1] * wsh[2] * wsh[3]
            else:
                a = shape(ins[0])
                fl = 2 * int(np.prod(o)) * a[-1]
        out.append((line, fl))
    return out


def time_reference(d, w: Workload, inputs, steps, warmup, budget_s):
    """FULL-graph runs of the reference CPU path: min(steps, what fits in budget_s) timed runs after min(warmup, 1) warm-up runs.
    When a single full run does not fit the budget (SDXL 1024x1024), a FLOP-weighted prefix of the graph is timed instead and the
    result is scaled -- stated in `sample`.  Returns (units_per_second, sample_text, seconds_per_run)."""
    m = make_reference_model(d, w)
    t = time.time(); step_api(m, inputs, None); t_first = time.time() - t      # warm-up run (also the calibration)
    if t_first <= budget_s / 2.5:
        n = int(max(1, min(steps, (budget_s - t_first) // max(t_first, 1e-3))))
        if warmup > 1 and t_first * (n + 1) < budget_s * 0.5:
            step_api(m, inputs, None)
        ts = []
        for _ in range(n):
            t = time.time(); step_api(m, inputs, None); ts.append(time.time() - t)
        m.close()
        per = float(np.mean(ts))
        return 1.0 / per, f"{n} full runs of the whole graph (all {len(open(d + 'model.txt').read().splitlines())} ops) after 1-2 warm-up runs; mean {per:.2f} s, min {min(ts):.2f} s, max {max(ts):.2f} s per run", per
    m.close()
    # too slow for full runs: prefix holding ~frac of the Conv/MatMul FLOPs
    lf = model_lines_flops(d)
    total = sum(f for _, f in lf)
    frac = max(0.02, min(0.5, budget_s / 3.0 / t_first))
    acc, n_ops = 0, 0
    for i, (_, f) in enumerate(lf):
        acc += f; n_ops = i + 1
        if acc >= frac * total:
            break
    fn = "model_prefix_ref.txt"
    open(d + fn, "w").write("\n".join(l for l, _ in lf[:n_ops]) + "\n")
    m = make_reference_model(d, w, fn)
    step_api(m, inputs, None)
    ts = []
    for _ in range(2):
        t = time.time(); step_api(m, inputs, None); ts.append(time.time() - t)
    m.close()
    per = float(np.mean(ts)) / (acc / total)
    return 1.0 / per, (f"one full run took {t_first:.1f} s (warm-up); timed sample = first {n_ops} of {len(lf)} graph ops = {100 * acc / total:.1f}% of the "
                       f"Conv/MatMul FLOPs, 2 runs, scaled to the whole graph"), per


# =====================================================================================================================
# the reference arm (--impl reference)
# =====================================================================================================================
def run_reference(args):
    if RANK != 0:
        return
    if args.workload == "sd15_pipeline":
        emit_line({"impl": "reference", "unavailable": "sd15_pipeline is a composite of three workloads: run their reference arms separately"})
        return
    w = make_workload(args.workload)
    if not os.path.exists(ORACLE_LIB):
        emit_line({"impl": "reference", "unavailable": "oracle/_ref/liboracle_ref.so missing (built from /root/reference by __graft_entry__.build())"})
        return
    d, meta = ensure_model(w)
    inputs = w.inputs(0)
    value, sample, per = time_reference(d, w, inputs, args.steps, args.warmup, budget_s=float(os.environ.get("OSB_REF_BUDGET_S", "170")))
    line = {
        "impl": "reference", "metric": w.metric, "value": value, "unit": w.unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.describe + " -- reference CPU path: same blobs, fp32 XNNPACK arithmetic, ONE sample on the host cores (per-sample throughput; it does not scale with --gpus)"},
        "cpu_baseline": {"value": value, "unit": w.unit, "cores": REF_THREADS, "host_cores": HOST_CORES, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": w.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(line)


# =====================================================================================================================
# the B200 arm
# =====================================================================================================================
def value_outputs(m):
    """Every output tensor of the last run of `m`, as a caller of Model::run receives it."""
    out = {}
    for n in m.get_all_tensor_names():
        t = m.get_tensor(n)
        out[n] = m.get_tensor_i64(n) if t is None else t
    return out


def write_outputs(d, outputs):
    """DIR/<name>.npy for every output, float32 (float64 for int64 / float64 tensors); an output larger than its share of
    DUMP_LIMIT_BYTES is replaced by a fixed, seeded sample of its elements."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_LIMIT_BYTES // max(len(outputs), 1)
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype in (np.int64, np.float64) else np.float32)
        if a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)


def measure(w: Workload, args, dist, clocks=None, outputs=None):
    """value / e2e / roofline / parity for one single-model workload; returns the JSON line (rank 0) or None.
    `outputs` (a dict): filled with what the value arm computed in its last timed step."""
    d, meta = ensure_model(w)
    dist_barrier(dist)
    inputs = w.inputs(RANK)   # rank r = sample r (seed + rank, src/sd.cpp:2671)
    peak_tf, peak_bw, peak_src = peaks()
    has_i64 = any(v.dtype == np.int64 for v in inputs.values())

    # ---------------- value arm: weights + inputs resident in HBM ----------------
    mv = make_engine_model(d, w, "ram+nocache", resident=True, graph=True)
    for _ in range(3):      # run 1 fills the HBM weight cache, run 2 warms scratch, run 3 captures the graph
        out_v = step_api(mv, inputs, w.out_name)
    later = w.later_inputs(inputs)
    if len(later) != len(inputs):
        for _ in range(3):  # fewer host inputs from now on (the rest stays in HBM): the graph is re-captured for that input set
            step_api(mv, later, w.out_name)
    st_v = mv.stats()
    launches_per_step = int(st_v["kernel_launches"])
    if clocks is None:
        clocks = ClockSampler(); clocks.start()      # sampled from the warm-up through both timed regions (value and e2e)
    graph_ok = True
    try:
        mv.run_resident(args.warmup)
    except Exception:
        graph_ok = False
    if graph_ok:
        dist_barrier(dist)
        gpu_ms = mv.run_resident(args.steps)
        value_mode = "HBM-resident weights + inputs, one captured CUDA graph per step" + (" (int64 inputs through device mirrors)" if has_i64 else "")
    else:
        # the graph reads int64 input VALUES on the host (shape arithmetic): eager runs, CUDA-event time of each run's stream work
        for _ in range(args.warmup):
            step_api(mv, later, None)
        dist_barrier(dist)
        gpu_ms = 0.0
        for _ in range(args.steps):
            step_api(mv, later, None)
            gpu_ms += mv.stats()["last_gpu_ms"]
        launches_per_step = int(mv.stats()["kernel_launches"])
        value_mode = "HBM-resident weights, eager launches (int64 input values are read on the host), CUDA-event time per run incl. the input upload"
    dist_barrier(dist)
    gpu_ms = dist_max(dist, gpu_ms)
    ms_per_step = gpu_ms / args.steps
    value = WORLD * 1000.0 / ms_per_step
    if outputs is not None:
        if graph_ok:
            # graph replays leave their outputs on the device: one more replay of the same graph on the same inputs returns them
            step_api(mv, later, None)
        outputs.update(value_outputs(mv))

    # ---------------- supplementary: host inputs / outputs through the C ABI every step, weights resident ----------------
    e2e_resident = None
    e2e_r_s, e2e_r_err = float("inf"), None
    try:                      # no collectives inside the try: a rank-local failure must not strand the other ranks at a barrier
        for _ in range(2):
            step_api(mv, inputs, w.out_name)
        t0r = time.perf_counter()
        for _ in range(args.steps):
            step_api(mv, inputs, w.out_name)
        e2e_r_s = time.perf_counter() - t0r
    except Exception as e:    # supplementary only: never take the bench down
        e2e_r_err = str(e)
    e2e_r_s = dist_max(dist, e2e_r_s)
    if e2e_r_err is None and e2e_r_s != float("inf"):
        e2e_resident = {"value": WORLD * args.steps / e2e_r_s, "unit": w.unit, "ms_per_step": 1000.0 * e2e_r_s / args.steps,
                        "note": "host inputs / outputs through the C ABI every step, weights resident in HBM (b200_resident_weights, the reference's --ram mode); ranks not barrier-aligned"}
    else:
        e2e_resident = {"value": None, "note": f"failed: {e2e_r_err}"}

    # ---------------- roofline leg: eager pass with per-launch CUDA events on the tcgen05 kernel ----------------
    mv.lib.model_set_option(mv.h, b"b200_cuda_graph", 0)
    step_api(mv, inputs, w.out_name)
    mv.lib.osb_tc_profile(1)
    step_api(mv, inputs, w.out_name)
    prof = (ctypes.c_double * 4)()
    mv.lib.osb_tc_profile_read(prof)
    if os.environ.get("OSB_TC_DUMP"):
        buf = ctypes.create_string_buffer(1 << 20)
        mv.lib.osb_tc_profile_dump.argtypes = [ctypes.c_char_p, ctypes.c_int]
        nb = mv.lib.osb_tc_profile_dump(buf, len(buf))
        open(os.environ["OSB_TC_DUMP"], "w").write(buf.raw[:max(nb, 0)].decode())
    mv.lib.osb_tc_profile(0)
    st_e = mv.stats()
    n_tc, tc_ms, tc_flops, tc_bytes = [float(x) for x in prof]
    achieved_tf = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "tc_gemm_kernel + tc_pair_kernel (tcgen05 implicit-GEMM conv / GEMM: single-CTA and CTA-pair tiles, all launches of one step)",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf if peak_tf else None,
                "peak_source": peak_src, "launches": int(n_tc), "kernel_ms_per_step": tc_ms, "flops_per_step": tc_flops,
                "algorithmic_bytes_per_step": tc_bytes,
                # share of the SAME eager, event-instrumented step (numerator and denominator carry the same per-launch event cost)
                "share_of_step": tc_ms / float(st_e["last_gpu_ms"]) if st_e.get("last_gpu_ms") else None, "traffic": None}
    if w.hbm_bound or n_tc == 0:
        # weight-bandwidth-bound step (decode GEMVs): algorithmic bytes = every weight once + every graph input once, over the whole step
        in_bytes = sum(int(v.nbytes) // (2 if v.dtype == np.float32 else 1) for v in inputs.values())     # activations live as fp16
        algo = float(meta["weight_bytes"] + in_bytes)
        ach = algo / (ms_per_step * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "whole step (grouped gemv_panel / gemv_w8_panel + attention_decode + elementwise): weights and KV cache streamed once per token",
                    "achieved": ach, "peak": peak_bw, "unit": "GB/s", "frac": ach / peak_bw, "peak_source": peak_src.replace("sustained bf16 cuBLAS", "STREAM-style copy"),
                    "algorithmic_bytes_per_step": algo, "traffic": None}
    # DRAM traffic of the same kernel from the committed ncu pass (scripts/ncu_traffic.py): per launch, like `achieved`
    for tname in ("r02_tc_traffic.json", "r01_tc_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if w.name == "sd15_unet_fp16" and os.path.exists(tpath) and n_tc:
            tj = json.load(open(tpath))
            roofline["traffic"] = tj.get("dram_bytes_per_launch")
            roofline["traffic_unit"] = "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, %d launches of one step; capture: profiles/%s%s)" % (
                tj.get("launches", 0), tname, (", taken at commit " + tj["commit"]) if tj.get("commit") else "")
            roofline["algorithmic_bytes_per_launch"] = tc_bytes / n_tc
            break
    mv.close()
    del mv

    # ---------------- e2e arm: host buffers through the C ABI, weights streamed every step ----------------
    comm = None
    me = Model(ENGINE_LIB, 0, "ram")
    if WORLD > 1:
        comm = make_comm(me.lib, dist)
    me.close()
    me = make_engine_model(d, w, "ram+nocache", resident=False, graph=False, comm=comm)
    for _ in range(max(2, args.warmup)):
        out_e = step_api(me, inputs, w.out_name)
    dist_barrier(dist)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out_e = step_api(me, inputs, w.out_name)
    dist_barrier(dist)
    e2e_s = dist_max(dist, time.perf_counter() - t0)
    clk = clocks.stop()
    st = me.stats()
    e2e_value = WORLD * args.steps / e2e_s
    h2d = int(st["weight_bytes_streamed"] + st["h2d_input_bytes"])
    d2h = int(st["d2h_output_bytes"])

    # ---------------- parity: EVERY rank, max over ranks in the line ----------------
    scale_v = float(np.abs(out_v).max())
    diff_sr = dist_max(dist, float(np.abs(out_e - out_v).max()) / max(scale_v, 1e-12))   # streamed (NCCL path at N>1) vs resident, own sample
    parity = {"streamed_vs_resident_rel_all_ranks": diff_sr, "ranks": WORLD}
    ref_s = None
    if os.path.exists(ORACLE_LIB) and not args.no_cpu_baseline:
        in0 = w.inputs(0)
        if RANK == 0:
            try:
                ref0, ref_s = reference_output_cached(d, w, in0, allow_compute=meta["flops"] <= 2.5e12)
            except Exception as e:    # the checker must never take the bench down
                ref0 = None
                parity["oracle_error"] = str(e)
        else:
            ref0 = None
        ref0 = dist_bcast_array(dist, ref0)
        if ref0 is not None:
            # sample 0 through THIS rank's streamed engine (NCCL-fed weights).  EVERY rank steps, rank 0 included: the weight stream's
            # all-gather is a collective, a rank that skipped the step would leave the others waiting in it
            got0 = step_api(me, in0, w.out_name)
            err = float(np.abs(got0 - ref0).max()) / max(float(np.abs(ref0).max()), 1e-12)
            parity["vs_reference_rel_all_ranks"] = dist_max(dist, err)
            parity["tol"] = w.tol
            parity["what"] = "max|engine - reference| / max|reference| on sample 0, every rank's streamed engine vs one full run of oracle/_ref (fp16 weights, fp32 XNNPACK arithmetic); max over ranks"
            parity["ok"] = bool(parity["vs_reference_rel_all_ranks"] <= w.tol and diff_sr <= 1e-2)   # run-to-run: atomics reorder fp32 sums
    me.close()

    line = {
        "metric": w.metric, "value": value, "unit": w.unit, "n_gpus": WORLD, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
        "config": {"workload": "%s: %d ops, %.0f M params, %.3f TFLOP/step; one sample per GPU" % (w.describe, meta["ops"], meta["params"] / 1e6, meta["flops"] / 1e12),
                   "weights": "value: " + value_mode + "; e2e: streamed pinned-host -> HBM ring every step",
                   "l2": "per-step weight stream = %.2f GB >> 126 MB L2, no flush needed" % (meta["weight_bytes"] / 1e9), "parallelism": f"dp{WORLD} (rank r = sample r)"},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": w.unit, "ms_per_step": 1000.0 * e2e_s / args.steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "weight_ring_bytes": int(st["weight_ring_bytes"]), "largest_node_bytes": int(st["weight_largest_node_bytes"]),
                "peak_hbm_resident_weight_bytes": int(st["weight_peak_live_bytes"]), "h2d_gbs": h2d / (e2e_s / args.steps) / 1e9,
                "weight_upload": ("every rank uploads 1/N of each node, ncclAllGather completes the slot" if WORLD > 1 else "cudaMemcpyAsync per node on the copy stream")},
        "e2e_resident_weights": e2e_resident,
        "parity": parity,
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step, "tcgen05_launches_per_step": int(st_e["tc_launches"]),
        "roofline": roofline,
    }

    if RANK == 0 and WORLD == 1 and not args.no_cpu_baseline and os.path.exists(ORACLE_LIB):
        try:
            # (DiskNoCache provider: every run re-reads the blobs and re-creates its operators, so the parity run above is a
            # representative run, not a cold outlier)
            if ref_s is not None and (ref_s >= 45 or getattr(args, "all_configs", None)):     # --all-configs: the parity run IS the sample (bounded total time)
                v, sample = 1.0 / ref_s, f"1 full run of the whole graph (the parity run), {ref_s:.1f} s"
            else:
                v, sample, per = time_reference(d, w, w.inputs(0), 2, 1, budget_s=100.0)
            line["cpu_baseline"] = {"value": v, "unit": w.unit, "cores": REF_THREADS, "host_cores": HOST_CORES, "kind": "reference",
                                    "sample": sample + " through the reference's Model::run (same blobs, fp32 XNNPACK arithmetic)"}
        except Exception as e:   # the baseline must never take the bench down
            line["cpu_baseline"] = {"value": None, "unit": w.unit, "cores": REF_THREADS, "kind": "reference", "sample": f"failed: {e}"}
    return line if RANK == 0 else None


def run_pipeline(args, dist, outputs=None):
    """BASELINE config[1]: text encoder (cond + uncond) + 20 sampler steps x 2 UNet runs (CFG) + VAE decoder = one 512x512 image.
    Each model is measured on its own (value / e2e as in `measure`); the image time is the sum over its calls."""
    parts = [("clip_text_fp32", 2), ("sd15_unet_fp16", 40), ("vae_decoder_fp16", 1)]
    clocks = ClockSampler(); clocks.start()
    lines, t_val, t_e2e, launches, h2d, d2h = {}, 0.0, 0.0, 0, 0, 0
    a2 = argparse.Namespace(**vars(args)); a2.no_cpu_baseline = True
    for name, calls in parts:
        part = None if outputs is None else {}
        ln = measure(make_workload(name), a2, dist, clocks=ClockSampler(), outputs=part)
        if part:
            outputs.update({f"{name}.{k}": v for k, v in part.items()})
        if RANK == 0:
            lines[name] = ln
            t_val += calls * ln["ms_per_step"]; t_e2e += calls * ln["e2e"]["ms_per_step"]
            launches += calls * ln["gpu_launches_per_step"]; h2d += calls * ln["e2e"]["h2d_bytes_per_step"]; d2h += calls * ln["e2e"]["d2h_bytes_per_step"]
    clk = clocks.stop()
    if RANK != 0:
        return None
    u = lines["sd15_unet_fp16"]
    return {
        "metric": "SD1.5 full pipeline 512x512 images/s (2 text-encoder runs + 20 steps x 2 UNet runs + 1 VAE decode)", "value": WORLD * 1000.0 / t_val, "unit": "images/s",
        "n_gpus": WORLD, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "BASELINE config[1]: CLIP-text (fp32) x2 + SD1.5 UNet fp16 x40 + VAE decoder fp16 x1, each timed over --steps runs; image time = sum of calls x per-call time (sampler host math excluded)",
                   "parts_ms": {k: v["ms_per_step"] for k, v in lines.items()}, "parts_e2e_ms": {k: v["e2e"]["ms_per_step"] for k, v in lines.items()}},
        "clocks": clk,
        "e2e": {"value": WORLD * 1000.0 / t_e2e, "unit": "images/s", "ms_per_step": t_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches, "roofline": u["roofline"], "parity": {k: v.get("parity") for k, v in lines.items()},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="sd15_unet_fp16", choices=WORKLOADS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--all-configs", default=None, help="run every BASELINE workload and append one JSON line each to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.all_configs or args.impl == "reference"):
        ap.error("--dump-outputs dumps the B200 path of one workload: it does not combine with --all-configs or --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    dist = dist_setup()
    if args.all_configs:
        for name in ["sd15_unet_fp16", "sd15_pipeline", "sdxl_unet_w8", "sdxl_turbo_w8", "vae_decoder_fp16", "clip_text_fp32", "tinyllama_decode", "tinyllama_decode_w8", "sd15_unet_fp32"]:
            a2 = argparse.Namespace(**vars(args)); a2.workload = name
            if name != "sd15_unet_fp16":
                a2.steps = min(args.steps, 10)
            try:
                line = run_pipeline(a2, dist) if name == "sd15_pipeline" else measure(make_workload(name), a2, dist)
            except Exception as e:
                line = {"workload": name, "error": str(e)} if RANK == 0 else None
            if RANK == 0 and line is not None:
                line["workload_key"] = name
                with open(args.all_configs, "a") as f:
                    f.write(json.dumps(line) + "\n")
                if name == "sd15_unet_fp16":
                    emit_line(line)
    else:
        outputs = {} if args.dump_outputs else None
        line = run_pipeline(args, dist, outputs) if args.workload == "sd15_pipeline" else measure(make_workload(args.workload), args, dist, outputs=outputs)
        if RANK == 0:
            if outputs is not None:
                write_outputs(args.dump_outputs, outputs)
            emit_line(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
