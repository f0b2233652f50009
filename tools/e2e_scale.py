"""End-to-end (tb_step_host, pinned host buffers) throughput of G ranks stepping at once, with the PCIe traffic nvidia-smi
sees per GPU meanwhile: what bounds the end-to-end curve at 8 GPUs (VERDICT round 1, item 8).
    torchrun --nproc-per-node G tools/e2e_scale.py [n_envs] [mode: zero_copy|staging]
Rank 0 prints one JSON line."""
import json, os, subprocess, sys, threading, time
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, ".")
from tennisbot_rl_b200.batch import TennisBatch

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
mode = sys.argv[2] if len(sys.argv) > 2 else "zero_copy"
os.environ["TB_HOST_MODE"] = mode
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
b = TennisBatch("SwingRacket-v0", n, device=local, seed=0, env_id_offset=rank * n)
b.reset_host()
hb = b.host_buffers()
np.copyto(hb["actions"], np.random.default_rng(rank).uniform(-1, 1, hb["actions"].shape).astype(np.float32))
for _ in range(26):
    b.step_host(want_terminal=False, want_events=False)
rows = []
def dmon():
    p = subprocess.Popen(["nvidia-smi", "dmon", "-s", "t", "-d", "1", "-c", "4"], stdout=subprocess.PIPE, text=True)
    for line in p.stdout:
        f = line.split()
        if len(f) >= 3 and f[0].isdigit():
            rows.append((int(f[0]), float(f[1]), float(f[2])))  # gpu, rx MB/s, tx MB/s
th = threading.Thread(target=dmon) if rank == 0 else None
if world > 1:
    dist.barrier()
if th:
    th.start()
torch.cuda.synchronize()
t0 = time.perf_counter()
steps = 0
while time.perf_counter() - t0 < 4.0:
    for _ in range(26):
        b.step_host(want_terminal=False, want_events=False)
    steps += 26
dt = time.perf_counter() - t0
rate = torch.tensor([n * steps / dt], dtype=torch.float64, device="cuda")
if world > 1:
    dist.all_reduce(rate)
if th:
    th.join()
if rank == 0:
    per_gpu = {}
    for g, rx, tx in rows:
        per_gpu.setdefault(g, []).append((rx, tx))
    pcie = {g: {"rx_MBps": float(np.median([r for r, _ in v])), "tx_MBps": float(np.median([t for _, t in v]))} for g, v in per_gpu.items()}
    print(json.dumps({"gpus": world, "envs_per_gpu": n, "transport": mode, "e2e_env_steps_per_s": float(rate.item()),
                      "per_gpu_env_steps_per_s": float(rate.item()) / world, "host_cores": os.cpu_count(),
                      "bytes_per_env_step_over_pcie": 24 + 24 + 4 + 1,
                      "implied_pcie_GBps_total": float(rate.item()) * 53 / 1e9, "nvidia_smi_dmon_pcie": pcie}))
if world > 1:
    dist.destroy_process_group()
