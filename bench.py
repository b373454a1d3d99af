#!/usr/bin/env python
"""bench.py - video VAE encode+decode frames/sec (BASELINE.json metric), one JSON line.

    python bench.py --gpus 1 --steps K --warmup W          # this framework (CUDA engine through the C ABI), config c2
    python bench.py --config c3|c4|c5 ...                  # the other BASELINE.json configs through the same harness
    python bench.py --impl reference ...                   # the reference algorithm on the host CPU cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" = encode(x).latent_dist.mode() -> decode(z).sample of one synthetic clip (or clip batch) through the public
model API, wrapper tiling/chunking on.  Configs (BASELINE.json `configs[1..4]`):
  c2  17x3x576x1024 fp16, SD2.1 model (1 chunk x 2 tiles of 576x576); N GPUs: clip of 1+16N frames, frame-sharded,
      one chunk per rank (weak scaling), one NCCL halo frame per codec direction
  c3  33x3x512x512 bf16, SD3 model (2 chunks, un-tiled); N GPUs: 1+32N frames, two chunks per rank (weak)
  c4  129x3x720x1280 fp16 (8 chunks x 6 ragged tiles), the 8 chunks split over N ranks with the halo exchange (strong)
  c5  batch-32 of 17x3x256x256 fp16, 32/N clips per rank, no communication (strong)
Keys:
  value      frames/s, inputs resident in HBM when the timed region starts
  e2e        same through host buffers: pinned host clip -> H2D -> encode/decode -> D2H of the reconstruction, per step
  roofline   tensor bound of the dominant kernels (tcgen05 implicit-GEMM conv): algorithmic FLOPs of their launches /
             their CUDA-event time in the timed region, against MEASURED_PEAKS.json (sustained bf16 cuBLAS TF/s)
  cpu_baseline        the oracle (CPU restatement of the reference algorithm, fp32) on the host cores, on a bounded
             sample, scaled to the workload by network-input pixel count            (N = 1, rank 0)
  torch_cuda_baseline the reference ALGORITHM in the bench dtype on torch-CUDA library kernels (cuDNN / SDPA), eager,
             wrapper tiling on, cudnn.benchmark False and True - the north_star's ">= 4x" denominator (N = 1, c2/c3)
  parity_sharded      N > 1: rank 0 also runs the un-sharded clip and the gathered sharded result must be
             bit-identical (moments and reconstruction); the line carries the verdict
  dumped     with --dump-outputs DIR: shape and stored element count of each array written to DIR

--dump-outputs DIR writes what the last timed step computed (rank 0's share) as float32 .npy files: latent.npy, the
latent z = encode(x).latent_dist.mode() that is decoded, and recon.npy, decode(z).sample.  An array of more than
DUMP_MAX_ELEMS elements is stored as a fixed seeded sample of its flattened elements.  Weights and inputs are seeded,
so runs with the same arguments on two builds can be compared array for array.  bench.py writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only; imports must not leave __pycache__ behind

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "video VAE encode+decode frames/sec at 17x576x1024"
UNIT = "frames/s"

CONFIGS = {
    "c2": dict(variant="sd21", dtype="fp16", frames=17, height=576, width=1024, batch=1, scaling="weak", chunks_per_rank=1,
               metric=METRIC),
    "c3": dict(variant="sd3", dtype="bf16", frames=33, height=512, width=512, batch=1, scaling="weak", chunks_per_rank=2,
               metric="video VAE encode+decode frames/sec at 33x512x512 (SD3 model, bf16)"),
    "c4": dict(variant="sd21", dtype="fp16", frames=129, height=720, width=1280, batch=1, scaling="strong",
               metric="video VAE encode+decode frames/sec at 129x720x1280"),
    "c5": dict(variant="sd21", dtype="fp16", frames=17, height=256, width=256, batch=32, scaling="strong",
               metric="video VAE encode+decode frames/sec, batch-32 of 17x256x256"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-cuda"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--frames", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--dtype", default=None, choices=["fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the sharded == un-sharded check at N > 1")
    ap.add_argument("--shard", default="frame", choices=["frame", "unit"],
                    help="N > 1, batch-1 configs: 'frame' = clip sharded on the frame axis + halo exchange (default; c2/c3 grow the "
                         "clip with N), 'unit' = the FIXED clip resident on every rank, its (chunk x tile) work units dealt over "
                         "the ranks (strong scaling of a clip with fewer chunks than GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's latent and reconstruction to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    for k in ("frames", "height", "width", "dtype"):
        if getattr(args, k) is not None:
            cfg[k] = getattr(args, k)
    args.cfg = cfg
    args.frames, args.height, args.width, args.dtype = cfg["frames"], cfg["height"], cfg["width"], cfg["dtype"]
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("bf16_tflops_sustained", 1400.0)), "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"
    return 1400.0, "fallback 1.4 PFLOP/s sustained (of fallback)"


def source_hash(root=None):
    """sha256 over the CUDA sources + the C header with comments and whitespace removed: identifies the KERNELS a
    committed ncu capture belongs to (editing a comment does not make a capture stale, editing code does)."""
    import re
    root = root or ROOT
    h = hashlib.sha256()
    d = os.path.join(root, "cvvae_b200", "csrc")
    for f in sorted(os.listdir(d)) + ["../../include/cvvae_b200.h"]:
        with open(os.path.join(d, f), "r", encoding="utf-8", errors="replace") as fh:
            src = fh.read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)     # block comments
        src = re.sub(r"//[^\n]*", "", src)                  # line comments (no '//' occurs inside string literals here)
        src = re.sub(r"\s+", "", src)
        h.update(f.encode() + b"\0" + src.encode())
    return h.hexdigest()[:16]


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU baseline
def usable_cores():
    """Host threads this process can really run at once: min(cpu_count, affinity mask, cgroup CPU quota).
    (A 1-GPU box of this pool shows 128 CPUs but a 16-CPU cgroup quota; 128 threads there run 8x SLOWER than 16.)"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, -(-int(parts[0]) // int(parts[1]))))
            else:
                quota = int(parts[0])
                with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                    period = int(f.read())
                if quota > 0:
                    n = min(n, max(1, -(-quota // period)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def sample_shape(n_runs):
    """Bounded CPU sample per step, shrunk when many runs are asked for so that the arm ends within a few minutes."""
    side = 192 if n_runs <= 6 else (128 if n_runs <= 30 else 96)
    return (1, 3, 17, side, side)


def oracle_cfg(cfg, **wrap):
    from oracle import cvvae_oracle as O
    if cfg["variant"] == "sd21":
        return O.VAEConfig(variant="sd21", **wrap)
    return O.VAEConfig(variant="sd3", z_channels=16, **wrap)


def cpu_sample(cfg, steps=1, shape=None, warmup=0):
    """Reference algorithm (oracle port, fp32) on the host cores on a bounded sample."""
    from oracle import cvvae_oracle as O  # the one place bench.py executes oracle/: the CPU baseline
    cores = usable_cores()
    torch.set_num_threads(cores)
    ocfg = oracle_cfg(cfg, tile_spatial_size=None, en_de_n_frames_a_time=None)
    sd = O.make_state_dict(ocfg, 1234)
    x = O.synthetic_video(shape, 0)
    with torch.no_grad():
        O.decode(O.encode(O.synthetic_video((1, 3, 1, 32, 32), 0), sd, ocfg).mode(), sd, ocfg)  # page in oneDNN
        for _ in range(warmup):
            O.decode(O.encode(x, sd, ocfg).mode(), sd, ocfg)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.decode(O.encode(x, sd, ocfg).mode(), sd, ocfg)
        dt = (time.perf_counter() - t0) / steps
    return dt, cores


def tiles_1d(n, tile=576, stride=448):
    out, i = [], 0
    while True:
        out.append(min(tile, n - i))
        if i + tile >= n:
            break
        i += stride
    return out


def workload_pixels(frames, height, width, batch=1, chunk=16):
    """Pixels the wrapper actually pushes through the networks (tile overlap and the re-encoded chunk frames included)."""
    n_chunks = max(1, -(-(frames - 1) // chunk))
    net_frames = sum(min(chunk * (n + 1) + 1, frames) - chunk * n for n in range(n_chunks))
    return batch * net_frames * sum(tiles_1d(height)) * sum(tiles_1d(width))


def cpu_baseline_entry(args, steps=1, warmup=0):
    cfg = args.cfg
    shp = sample_shape(steps + warmup)
    dt, cores = cpu_sample(cfg, steps, shp, warmup)
    ratio = workload_pixels(args.frames, args.height, args.width, cfg["batch"]) / (shp[2] * shp[3] * shp[4])
    fps = cfg["batch"] * args.frames / (dt * ratio)
    return {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle fp32 ({cfg['variant']} nets) encode+decode of one {shp[2]}x{shp[3]}x{shp[4]} clip "
                      f"({dt:.2f} s), scaled x{ratio:.1f} by network-input pixel count to "
                      f"{cfg['batch']}x{args.frames}x{args.height}x{args.width} (tile overlap of the 576/448 tiling and the "
                      f"re-encoded chunk-boundary frames included)"}, dt


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    entry, dt = cpu_baseline_entry(args, steps, warm)
    line = {"impl": "reference", "metric": args.cfg["metric"], "value": entry["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": args.cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.cfg['batch']}x{args.frames}x3x{args.height}x{args.width} encode+decode ({args.config}), "
                                   f"bounded CPU sample per step"},
            "cpu_baseline": entry,
            "e2e": {"value": entry["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ output dump
DUMP_MAX_ELEMS = 4 << 20   # per array: 16 MB of float32, so latent + reconstruction stay within 64 MB


def dump_array(t, seed=0):
    """`t` as a float32 numpy array, or, above DUMP_MAX_ELEMS elements, the flattened elements at DUMP_MAX_ELEMS sorted
    positions drawn (with replacement) from a generator seeded with `seed`: the positions depend on the size alone."""
    n = t.numel()
    if n <= DUMP_MAX_ELEMS:
        return t.float().cpu().numpy()
    idx = torch.randint(0, n, (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(seed)).sort().values
    return t.reshape(-1)[idx.to(t.device)].float().cpu().numpy()


def dump_outputs(d, arrays):
    """Write each named tensor to d/<name>.npy; returns {name: {"shape", "stored"}} for the JSON line."""
    os.makedirs(d, exist_ok=True)
    info = {}
    for name, t in arrays.items():
        a = dump_array(t)
        np.save(os.path.join(d, name + ".npy"), a)
        info[name] = {"shape": list(t.shape), "stored": int(a.size)}
    return info


# ------------------------------------------------------------------------------------------ GPU arms
def build_model(cfg, dtype):
    from cvvae_b200 import CVVAEModel, CVVAESD3Model
    torch.manual_seed(1234)
    m = CVVAEModel() if cfg["variant"] == "sd21" else CVVAESD3Model()   # reference defaults: tile 576, chunks of 16(+1)
    g = torch.Generator().manual_seed(4321)
    for k, p in m.named_parameters():  # non-trivial affine/bias so nothing is skipped or degenerate
        if p.dim() == 1:
            p.data.copy_(torch.rand(p.shape, generator=g) * (0.4 if k.endswith("bias") else 1.0) + (-0.2 if k.endswith("bias") else 0.5))
    return m.to(dtype).cuda()


class TorchCudaReference:
    """The reference algorithm on torch-CUDA library kernels (cuDNN etc.): the north_star's '>= 4x the reference's own
    torch-cuda' denominator.  The reference is Python and /root/reference does not exist on the GPU box, so this runs its
    pinned restatement (oracle/, checked against the reference's own outputs in tests/test_oracle_golden.py) with the
    same state dict as the engine; kind = "port"."""

    def __init__(self, cfg, state_dict):
        from oracle import cvvae_oracle as O
        self.O = O
        self.cfg = oracle_cfg(cfg)
        self.sd = state_dict
        self.encode_n_frames_a_time = 16
        self.decode_n_frames_a_time = 4

    def tiled_encode(self, x):
        return self.O.tiled_encode(x, self.sd, self.cfg)

    def tiled_decode(self, z):
        return self.O.tiled_decode(z, self.sd, self.cfg)


def time_torch_cuda(ref, x, zc, warmup=3, reps=10):
    """frames/s of the torch-CUDA reference arm: CUDA events, `warmup` untimed passes, median of `reps`."""
    def step():
        with torch.no_grad():
            return ref.tiled_decode(ref.tiled_encode(x)[:, :zc])
    out = {}
    frames = x.shape[0] * x.shape[2]
    for bench_flag in (False, True):
        torch.backends.cudnn.benchmark = bench_flag
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            step()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        ts.sort()
        out["cudnn_benchmark_" + ("true" if bench_flag else "false")] = {"frames_per_s": frames / (ts[len(ts) // 2] * 1e-3),
                                                                          "ms_per_step_median": ts[len(ts) // 2]}
    torch.backends.cudnn.benchmark = False
    torch.cuda.empty_cache()
    return out


def main():
    args = parse()
    cfg = args.cfg
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    assert torch.cuda.is_available(), "bench.py needs a GPU (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local)
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dtype = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    zc = 4 if cfg["variant"] == "sd21" else 16

    from cvvae_b200 import _lib
    _lib.load()   # the library __graft_entry__.build() made; bench.py compiles nothing and raises if it is missing
    model = build_model(cfg, dtype)
    ops = model._engine().ops
    if args.impl == "torch-cuda":
        net = TorchCudaReference(cfg, dict(model.state_dict()))
        ops = None
    else:
        net = model

    # ---- this rank's share of the work
    from cvvae_b200.parallel import FrameShardedVAE, chunk_ranges, frame_range
    stride = 16
    F, B = args.frames, cfg["batch"]
    sharded, total_chunks = None, None
    unit = None
    if args.shard == "unit" and world > 1 and B == 1:
        from cvvae_b200.parallel import UnitShardedVAE
        unit = UnitShardedVAE(model)
        cfg["scaling"] = "strong"
        total_chunks = max(1, -(-(F - 1) // stride))
        total_frames = F
        ranges = [(0, total_chunks)] * world
        b_local = B
    elif cfg["scaling"] == "weak":          # c2 / c3: (F-1)/16 chunks per rank, clip of 1 + (F-1) N frames
        cpr = (F - 1) // stride
        total_chunks = cpr * world
        total_frames = 1 + (F - 1) * world
        ranges = [(r * cpr, (r + 1) * cpr) for r in range(world)]
        b_local = B
    elif B == 1:                            # c4: fixed clip, its chunks split over the ranks
        total_chunks = (F - 1) // stride
        total_frames = F
        ranges = chunk_ranges(total_chunks, world)
        b_local = B
    else:                                   # c5: fixed batch of clips, split over the ranks
        assert B % world == 0, "batch must divide over the ranks"
        total_frames = F
        ranges = [(0, (F - 1) // stride)] * world
        b_local = B // world
    if world > 1 and B == 1 and unit is None:
        assert args.impl == "ours"
        sharded = FrameShardedVAE(model)
    c0, c1 = ranges[rank]
    f0, f1 = (frame_range(c0, c1, stride) if (sharded is not None and c1 > c0) else (0, (F if sharded is None else 0)))

    def gen_chunk_frames(a, b, seed_base=0):
        """Frames [a, b) of the (virtual) whole clip: one seeded block per 16-frame chunk so that any rank can rebuild any part."""
        parts = []
        t = a
        while t < b:
            c = 0 if t == 0 else (t - 1) // stride
            lo, hi = frame_range(c, c + 1, stride)
            g = torch.Generator().manual_seed(1000 + seed_base + c)
            blk = (torch.rand((b_local, 3, hi - lo, args.height, args.width), generator=g) * 2 - 1).to(dtype)
            parts.append(blk[:, :, t - lo:min(b, hi) - lo])
            t = min(b, hi)
        return torch.cat(parts, dim=2) if len(parts) > 1 else parts[0]

    x_host = gen_chunk_frames(f0, f1, seed_base=(rank * 100 if (sharded is None and unit is None and world > 1) else 0)).pin_memory()
    x_dev = x_host.cuda()

    def step(x):
        """One encode -> decode of this rank's share; returns (latent z, reconstruction)."""
        with torch.no_grad():
            if sharded is not None:
                z = sharded.encode_local(x, total_chunks)[:, :zc].contiguous()
                return z, sharded.decode_local(z, total_chunks)
            if unit is not None:
                z = unit.encode(x)[:, :zc].contiguous()
                return z, unit.decode(z)
            z = net.tiled_encode(x)[:, :zc]
            return z, net.tiled_decode(z)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        sync()
        ms = torch.tensor([s.elapsed_time(e)], device="cuda")
        if world > 1:
            every = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(every, ms)
            timed.per_rank = [round(t.item() / steps, 2) for t in every]   # each rank's own device time per step
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # ---- N > 1: sharded result == un-sharded result of the same engine, checked on rank 0 before anything is timed
    parity = None
    if unit is not None and not args.no_parity:
        with torch.no_grad():
            mom_u = unit.encode(x_dev)
            rec_u = unit.decode(mom_u[:, :zc].contiguous())
            mom_f = model.tiled_encode(x_dev)
            rec_f = model.tiled_decode(mom_f[:, :zc].contiguous())
            parity = bool(torch.equal(mom_f, mom_u) and torch.equal(rec_f, rec_u))   # every rank holds the full result
            del mom_u, rec_u, mom_f, rec_f
        torch.cuda.empty_cache()
        flag = torch.tensor([1 if parity else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = bool(flag.item())
        if not parity:
            if rank == 0:
                print(json.dumps({"metric": cfg["metric"], "n_gpus": world, "parity_sharded": False,
                                  "error": "unit-sharded encode/decode differs from the un-sharded run of the same engine"}))
            dist.destroy_process_group()
            sys.exit(1)
    if sharded is not None and not args.no_parity:
        with torch.no_grad():
            mom_l = sharded.encode_local(x_dev, total_chunks)
            rec_l = sharded.decode_local(mom_l[:, :zc].contiguous(), total_chunks)
            lens_p = [frame_range(a, b, stride)[1] - frame_range(a, b, stride)[0] if b > a else 0 for a, b in ranges]
            lens_l = [frame_range(a, b, stride // 4)[1] - frame_range(a, b, stride // 4)[0] if b > a else 0 for a, b in ranges]
            mom_g = sharded.gather_frames(mom_l, lens_l)
            rec_g = sharded.gather_frames(rec_l, lens_p)
            if rank == 0:
                x_full = gen_chunk_frames(0, total_frames).cuda()
                mom_f = model.tiled_encode(x_full)
                rec_f = model.tiled_decode(mom_f[:, :zc].contiguous())
                parity = bool(torch.equal(mom_f, mom_g) and torch.equal(rec_f, rec_g))
                del x_full, mom_f, rec_f
            del mom_g, rec_g, mom_l, rec_l
        torch.cuda.empty_cache()
        flag = torch.tensor([1 if (parity or rank != 0) else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() == 0:
            if rank == 0:
                print(json.dumps({"metric": cfg["metric"], "n_gpus": world, "parity_sharded": False,
                                  "error": "sharded encode/decode differs from the un-sharded run of the same engine"}))
            dist.destroy_process_group()
            sys.exit(1)

    for _ in range(max(args.warmup, 3)):
        last = step(x_dev)
    sync()

    def timed_step():
        nonlocal last
        last = step(x_dev)

    # ---- device-resident timing (+ per-conv CUDA events for the roofline)
    launches0 = ops.launch_count() if ops else 0
    sampler = ClockSampler(local) if rank == 0 else None
    if ops:
        ops.start_profile()
    ms_total = timed(timed_step, args.steps)
    ms_per_rank = getattr(timed, "per_rank", None)
    prof = ops.stop_profile() if ops else None
    clocks = sampler.stop() if sampler else None
    launches = (ops.launch_count() - launches0) if ops else 0
    ms_step = ms_total / args.steps
    job_frames = B * total_frames
    value = job_frames / (ms_step * 1e-3)
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, {"latent": last[0], "recon": last[1]})
    out = last[1]

    # ---- end-to-end: pinned host clip -> H2D -> encode/decode -> D2H of the reconstruction, every step
    rec_host = torch.empty(out.shape, dtype=out.dtype).pin_memory()

    def e2e_step():
        xd = x_host.cuda(non_blocking=True)
        r = step(xd)[1]
        rec_host.copy_(r, non_blocking=True)

    if args.impl == "ours":
        model.enable_cuda_graphs(True)  # public option of the model: every network call replays a captured graph
    e2e_step()
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps) / args.steps
    e2e = {"value": job_frames / (ms_e2e * 1e-3), "unit": UNIT, "cuda_graphs": args.impl == "ours",
           "h2d_bytes_per_step": x_host.numel() * x_host.element_size(),
           "d2h_bytes_per_step": rec_host.numel() * rec_host.element_size()}
    if args.impl == "ours":
        model.enable_cuda_graphs(False)
    peak_hbm = round(torch.cuda.max_memory_allocated() / 1e9, 2)  # activations + weights + graph pools, this rank

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    roof = None
    if prof and prof["conv_tc"]["ms"] > 0:
        tc = prof["conv_tc"]
        achieved = tc["flops"] / (tc["ms"] * 1e-3) / 1e12
        traffic, traffic_src, traffic_stale = None, None, None
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp) and args.config == "c2":
            # ncu dram bytes (read + write) per conv launch of this command, from the committed capture; stamped with the
            # hash of the CUDA sources it was captured from - a mismatch means the kernels changed since (stale)
            with open(tp) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
            traffic_stale = tj.get("source_hash") != source_hash()
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel / conv_tc_psw_kernel / conv_stk_kernel (tcgen05 implicit-GEMM conv, all "
                                             "launches of the timed region)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "traffic_stale": traffic_stale,
                "algorithmic_bytes_per_launch": tc["bytes"] / max(tc["launches"], 1),
                "peak_source": peak_src, "algorithmic_tflop_per_step": tc["flops"] / args.steps / 1e12,
                "kernel_ms_per_step": tc["ms"] / args.steps, "launches_per_step": tc["launches"] / args.steps,
                "share_of_step": tc["ms"] / ms_total,
                # the up-sampling convs run as folded 2x2 phase kernels (2.25x fewer MACs than the reference issues);
                # `achieved` counts EXECUTED FLOPs, this is the same time against the reference's dense count
                "reference_dense_tflop_per_step": tc["ref_flops"] / args.steps / 1e12,
                "achieved_vs_reference_count": tc["ref_flops"] / (tc["ms"] * 1e-3) / 1e12,
                "conv_direct_ms_per_step": prof["conv_direct"]["ms"] / args.steps}
    n_tiles = len(tiles_1d(args.height)) * len(tiles_1d(args.width))
    par = (f"frame-shard x{world}" if sharded is not None else (f"(chunk x tile)-unit-shard x{world}" if unit is not None else
           (f"batch-shard x{world}" if world > 1 else "single GPU")))
    line = {"metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"name": args.config,
                       "workload": f"{B}x{total_frames}x3x{args.height}x{args.width} clip{'s' if B > 1 else ''}, encode(x).mode() -> "
                                   f"decode(z), wrapper tiling 576/448 + 16-frame chunks; {cfg['variant'].upper()}-variant model, "
                                   f"seeded random weights",
                       "per_gpu": f"{b_local} x {c1 - c0} chunk(s) of <= 17 frames x {n_tiles} spatial tile(s) (<= 576x576, stride 448)",
                       "parallelism": par,
                       "l2": "no explicit flush: every step streams far more than the 126 MB L2 (activations up to 1.4 GB each)"},
            "impl": args.impl, "gpu_launches": launches // args.steps if launches else 0, "clocks": clocks, "e2e": e2e,
            "peak_hbm_gb": peak_hbm, "source_hash": source_hash()}
    if parity is not None:
        line["parity_sharded"] = parity
    if ms_per_rank is not None:
        # `ms_per_step` is the MAX of these (the slowest GPU sets the pace of a weak-scaled job; power-capped B200s of one box
        # differ by a few per cent)
        line["ms_per_step_per_rank"] = ms_per_rank
    if roof:
        line["roofline"] = roof
    if dumped is not None:
        line["dumped"] = dumped
    if args.impl == "ours" and world == 1:
        if not args.no_torch_baseline and args.config in ("c2", "c3"):
            ref = TorchCudaReference(cfg, dict(model.state_dict()))
            tcb = time_torch_cuda(ref, x_dev, zc, warmup=3, reps=10)
            tcb.update({"kind": "port", "unit": UNIT, "dtype": args.dtype,
                        "what": "reference algorithm (oracle restatement pinned to the reference's outputs) on torch-CUDA library "
                                "kernels, eager, wrapper tiling/chunking on, same state dict and input; CUDA events, 3 warm-ups, "
                                "median of 10; the reference's own modules cannot travel to the GPU box (/root/reference absent)"})
            tcb["speedup_value_vs_cudnn_benchmark_false"] = value / tcb["cudnn_benchmark_false"]["frames_per_s"]
            tcb["speedup_value_vs_cudnn_benchmark_true"] = value / tcb["cudnn_benchmark_true"]["frames_per_s"]
            line["torch_cuda_baseline"] = tcb
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_entry(args, 1)[0]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
