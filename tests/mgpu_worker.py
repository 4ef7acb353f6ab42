"""Worker of tests/test_multi_gpu.py: one process per GPU (torchrun), NCCL weight distribution through the engine's WeightStreamer.
Every rank runs ITS OWN sample (seed = rank) on the tiny fp16 UNet with all weights streamed through the HBM ring -- sharded upload
(1/N over this rank's PCIe link + ncclAllGather) by default, root upload + ncclBroadcast with OSB_SHARDED_H2D=0 -- and compares the
result with the reference's output for that sample (tests/golden/unet_tiny16_fp16_seed<rank>.npz).  Prints one MGPU_OK / MGPU_FAIL line per rank."""
import ctypes
import os
import sys

RANK = int(os.environ["RANK"]); WORLD = int(os.environ["WORLD_SIZE"]); LOCAL = int(os.environ.get("LOCAL_RANK", RANK))
vis = os.environ.get("CUDA_VISIBLE_DEVICES")
devs = vis.split(",") if vis else [str(i) for i in range(16)]
os.environ["CUDA_VISIBLE_DEVICES"] = devs[LOCAL]
os.environ["OMP_NUM_THREADS"] = "4"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from onnxstream_b200 import emit  # noqa: E402
from onnxstream_b200.model import Model, ENGINE_LIB  # noqa: E402

GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", f"unet_tiny16_fp16_seed{RANK}.npz"))
torch.cuda.set_device(0)
dist.init_process_group("nccl", device_id=torch.device("cuda", 0))
d = sys.argv[1]
cfg = emit.UNetConfig.tiny(16)
inputs = emit.unet_inputs(cfg, seed=RANK)
OPTS = ("use_fp16_arithmetic", "fuse_ops_in_attention")


def run(lib, comm=None, runs=1):
    m = Model(lib, 4, "ram+nocache" if lib == ENGINE_LIB else "nocache")
    for o in OPTS:
        m.set_option(o, True)
    if comm is not None:
        m.lib.model_b200_set_comm(m.h, comm, RANK, WORLD)
    m.read_file(d + "model.txt")
    out = None
    for _ in range(runs):
        m.clear_tensors()
        for k, v in inputs.items():
            m.add_tensor(k, v)
        m.run()
        out = m.get_tensor("out_5F_sample")
    return out, m


probe = Model(ENGINE_LIB, 0, "ram")
ident = ctypes.create_string_buffer(128)
if RANK == 0:
    assert probe.lib.osb_comm_unique_id(ident) == 0
obj = [bytes(ident.raw)]
dist.broadcast_object_list(obj, src=0)
comm = probe.lib.osb_comm_init(WORLD, RANK, obj[0])
assert comm, "ncclCommInitRank failed"
probe.close()
got, m = run(ENGINE_LIB, comm, runs=3)          # 3 runs: ring wrap-around and slot reuse across runs
st = m.stats()
assert all(np.array_equal(GOLDEN["in_" + k], v) for k, v in inputs.items()), "inputs differ from the stored case"
ref = GOLDEN["output"]
alone, _ = run(ENGINE_LIB, None)                # the same engine without NCCL: every byte over this rank's own link
err = float(np.abs(got - ref).max()) / max(float(np.abs(ref).max()), 1e-9)
self_err = float(np.abs(got - alone).max()) / max(float(np.abs(alone).max()), 1e-9)
ok = err <= 3e-2 and self_err <= 5e-3 and np.isfinite(got).all()
print(f"{'MGPU_OK' if ok else 'MGPU_FAIL'} rank {RANK}/{WORLD} vs_reference {err:.3e} vs_single_gpu {self_err:.3e} streamed_bytes {int(st['weight_bytes_streamed'])} sharded {os.environ.get('OSB_SHARDED_H2D', 'default')}", flush=True)
dist.barrier()
dist.destroy_process_group()
