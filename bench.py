#!/usr/bin/env python
"""Flagship benchmark: KV-block write+read throughput through the store's public API.

Metric (BASELINE.json): KV-block write/read GB/s, 128 KB paged-KV blocks, synthetic random
blocks.  Methodology mirrors the reference's own benchmark (infinistore/benchmark.py:
132-208): `--size-mb` of KV pages split into `--block-kb` blocks with fresh keys every
round, block allocation outside the timed region, writes then reads issued in `--layers`
batches, one `sync()` after each phase, read-back verified against the source.

One STEP = `--rounds` rounds of (write size-mb -> sync -> read it back -> sync), every round
with fresh keys (first-writer-wins would turn a re-write into a no-op).  Defaults: 4 GiB per
phase x 24 rounds = 192 GiB moved per GPU per step, so that K = 20 steps are a timed region
of ~1.4 s at N = 1 and ~6 s at N >= 2 (round 1 timed 0.02 s; 16 rounds gave 0.93 s at
N = 1).  The pool cannot hold a whole
run: it is purged and re-reserved between epochs, OUTSIDE the timed regions, whose
device-measured durations (CUDA events, barrier + synchronize on both sides) are summed.

Topology at N GPUs (one process per GPU, torchrun): every rank hosts one pool shard of
the store (server thread + HBM pool on its GPU) and is a client of the shard on GPU
(rank+1) % N, so for N >= 2 every byte crosses NVLink exactly once per direction and the
per-GPU work is fixed (weak scaling).  N = 1: the pool is on the same GPU (HBM to HBM).

One JSON line on rank 0.  `value` = aggregate (write+read) payload GB/s over all ranks,
max over ranks.  `e2e` = the same step through the public API including, per step, the
host->device copy of every round's pages from pinned (NUMA-local) host memory, overlapped
layer by layer with the writes, and a device->host read of the result.
`baselines` are measured in the same run on the same box and are EMULATIONS, labelled as
such: the reference itself cannot be built offline (DESIGN.md §5, `--impl reference`).
`extra` carries BASELINE.json configs 3, 4 and 5 and single-block latency percentiles.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "kv_block_write_read_GBps"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--size-mb", type=int, default=4096, help="KV bytes per phase (one round)")
    p.add_argument("--rounds", type=int, default=24, help="write+read rounds per step")
    p.add_argument("--block-kb", type=int, default=128)
    p.add_argument("--layers", type=int, default=32, help="batches per phase (reference --steps)")
    p.add_argument("--variant", default="auto", choices=["auto", "ldst", "tma", "ldst256"])
    p.add_argument("--max-ctas", type=int, default=0)
    p.add_argument("--streams", type=int, default=4, help="internal launch streams per connection")
    p.add_argument("--stage-kb", type=int, default=0, help="TMA pipeline slot size (0 = default)")
    p.add_argument("--ring-kb", type=int, default=0, help="TMA pipeline ring per CTA (0 = default)")
    p.add_argument("--host-lookup", action="store_true",
                   help="resolve read keys through the server instead of the HBM index")
    p.add_argument("--base-port", type=int, default=0)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip configs 3-5, latency, baselines")
    p.add_argument("--pool-gb", type=int, default=0, help="HBM pool per GPU (0 = auto: what fits)")
    p.add_argument("--ref-size-mb", type=int, default=1024,
                   help="reference arm: MB written+read per step (one round)")
    p.add_argument("--quick", action="store_true",
                   help="small shapes for a functional check (256 MB x 2 rounds, no extras)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps write a fixed, seeded sample of what the last "
                        "step read back (`dst`) to DIR/dst_sample.npy: float32, 32 MB in all "
                        "(dst_sample_rank<r>.npy per rank with several GPUs)")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        p.error("--dump-outputs needs --impl b200")
    return a


def reference_arm(args):
    """The UNMODIFIED reference, built by baseline/build_reference.sh into baseline/_ref (its
    own sources and Makefile; the missing system libraries are stood in for as that script
    documents) and driven through its own stock entry points, in clean interpreters that
    cannot see this repo: `python -m infinistore.server` and `python -m infinistore.benchmark`
    (infinistore/benchmark.py: fresh UUID keys per iteration, `--steps` batches per phase,
    one sync() per phase, host clock - the methodology this file mirrors).

    Only the reference's LOCAL_GPU data path can run here: its RDMA path needs an RDMA NIC,
    and the box has none (the verbs stand-in creates no queue pairs).  One server + one
    benchmark client per rank, client tensors on the rank's GPU, pool in pinned host memory
    (where the reference always keeps it).  A reference step is ONE round of `--ref-size-mb`
    written and read back (the b200 arm moves 16 x 4 GiB per step; at PCIe speed that would
    take minutes per step) - rates, not step times, are comparable."""
    import re
    import signal
    import socket
    import urllib.request

    ref = os.path.join(ROOT, "baseline", "_ref")
    so = [f for f in (os.listdir(os.path.join(ref, "infinistore"))
                      if os.path.isdir(os.path.join(ref, "infinistore")) else [])
          if f.startswith("_infinistore") and f.endswith(".so")]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    def unavailable(why):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": why[:300]}))

    bind_to_gpu_numa_node(local_rank)  # same placement help as the b200 arm; children inherit it
    if not so:
        return unavailable("baseline/_ref has no native module: run baseline/build_reference.sh "
                           "(needs uvloop's libuv, flashinfer's spdlog headers, nvcc toolchain)")
    env = dict(os.environ, PYTHONPATH=ref,
               PATH=os.path.join(ROOT, "baseline", "refshim", "bin") + os.pathsep +
               os.environ.get("PATH", ""))
    env.pop("PYTHONHOME", None)
    probe = subprocess.run([sys.executable, "-c", "import infinistore._infinistore, torch; "
                            "assert torch.cuda.is_available()"],
                           cwd="/tmp", env=env, capture_output=True, text=True, timeout=600)
    if probe.returncode != 0:
        last = (probe.stderr.strip().splitlines() or ["import failed"])[-1]
        return unavailable("reference module does not import / no GPU: " + last)

    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("gloo")  # host-side rendezvous only: no GPU work in this process

    def allmax(x):
        if dist is None:
            return x
        import torch

        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    size_mb, block_kb = args.ref_size_mb, args.block_kb
    rounds = max(args.steps, args.warmup, 1)
    base = args.base_port or (27000 + (int(os.environ.get("MASTER_PORT", "0")) % 2000))
    sport, mport = base + 2 * rank, base + 2 * rank + 1
    pool_gb = (rounds * size_mb + 1023) // 1024 + 2
    log = open(f"/tmp/ref_server_{rank}.log", "w")
    server = subprocess.Popen(
        [sys.executable, os.path.join(ROOT, "baseline", "ref_server_launch.py"),
         "--service-port", str(sport),
         "--manage-port", str(mport), "--prealloc-size", str(pool_gb),
         "--minimal-allocate-size", str(min(block_kb, 64)), "--log-level", "warning"],
        cwd="/tmp", env=env, stdout=log, stderr=subprocess.STDOUT, start_new_session=True)
    result = None
    try:
        deadline = time.time() + 300  # pinning tens of GB of host memory takes a while
        up = False
        while time.time() < deadline and server.poll() is None:
            try:
                urllib.request.urlopen(f"http://127.0.0.1:{mport}/kvmap_len", timeout=2).read()
                socket.create_connection(("127.0.0.1", sport), timeout=2).close()
                up = True
                break
            except Exception:  # noqa: BLE001
                time.sleep(0.5)
        if not up:
            log.flush()
            tail = open(log.name).read()[-300:].replace("\n", " | ")
            raise RuntimeError("reference server did not come up: " + tail)

        def bench(iterations):
            r = subprocess.run(
                [sys.executable, "-m", "infinistore.benchmark", "--service-port", str(sport),
                 "--size", str(size_mb), "--block-size", str(block_kb), "--iteration", str(iterations),
                 "--src-gpu", str(local_rank), "--dst-gpu", str(local_rank), "--steps", str(args.layers)],
                cwd="/tmp", env=env, capture_output=True, text=True, timeout=1800)
            m = re.search(r"write cache: ([0-9.]+) MB/s, read cache: ([0-9.]+) MB/s", r.stdout)
            if r.returncode != 0 or not m:
                raise RuntimeError("reference benchmark failed: " +
                                   (r.stderr.strip().splitlines() or r.stdout.strip().splitlines()
                                    or ["?"])[-1])
            return float(m.group(1)), float(m.group(2))

        if args.warmup:
            bench(args.warmup)
            urllib.request.urlopen(urllib.request.Request(f"http://127.0.0.1:{mport}/purge", method="POST"),
                                   timeout=60).read()
        if dist is not None:
            dist.barrier()
        w_mibs, r_mibs = bench(args.steps)
        mib = float(size_mb * args.steps)
        secs = mib / w_mibs + mib / r_mibs  # the benchmark's own write_sum + read_sum
        e2e = None
        if not args.no_e2e:
            urllib.request.urlopen(urllib.request.Request(f"http://127.0.0.1:{mport}/purge", method="POST"),
                                   timeout=60).read()
            if dist is not None:
                dist.barrier()
            r = subprocess.run(
                [sys.executable, os.path.join(ROOT, "baseline", "ref_e2e.py"), "--service-port", str(sport),
                 "--size-mb", str(size_mb), "--block-kb", str(block_kb), "--layers", str(args.layers),
                 "--steps", "2", "--gpu", str(local_rank)],
                cwd="/tmp", env=env, capture_output=True, text=True, timeout=1200)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if r.returncode == 0 and lines:
                e2e = json.loads(lines[-1])
        result = (secs, w_mibs, r_mibs, e2e)
    except Exception as e:  # noqa: BLE001
        result = e
    finally:
        try:
            os.killpg(server.pid, signal.SIGINT)
            server.wait(20)
        except Exception:  # noqa: BLE001
            try:
                os.killpg(server.pid, signal.SIGKILL)
            except Exception:  # noqa: BLE001
                pass
    failed = allmax(1.0 if isinstance(result, Exception) else 0.0)
    if failed:
        why = repr(result) if isinstance(result, Exception) else "another rank failed"
        unavailable("reference run failed: " + why)
    else:
        secs = allmax(result[0])
        bytes_per_step = 2 * (size_mb << 20)
        value = world * bytes_per_step * args.steps / secs / 1e9
        e2e_json = None
        have_e2e = allmax(0.0 if result[3] else 1.0) == 0.0
        if have_e2e:
            e_secs = allmax(result[3]["e2e_secs"])
            e2e_json = {"value": round(world * bytes_per_step * result[3]["steps"] / e_secs / 1e9, 3),
                        "unit": "GB/s", "h2d_bytes_per_step": result[3]["h2d_bytes_per_step"],
                        "d2h_bytes_per_step": result[3]["d2h_bytes_per_step"],
                        "steps": result[3]["steps"], "verified": result[3]["verified"],
                        "how": "baseline/ref_e2e.py: the reference's public API, pinned host pages "
                               "H2D per layer + synchronize before each write (its servers copy "
                               "on their own streams), D2H of the result"}
        if rank == 0:
            print(json.dumps({
                "metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(secs / args.steps * 1e3, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "fp32 pages (dtype-blind bytes)",
                "data": "synthetic random KV pages, fresh UUID keys per iteration",
                "impl": "reference",
                "config": {"model": "paged-KV blocks", "block_kb": block_kb,
                           "bytes_per_gpu_per_step": bytes_per_step, "layers_per_phase": args.layers,
                           "data_path": "LOCAL_GPU (TCP + CUDA IPC + per-block cudaMemcpyAsync to the "
                                        "pinned host pool): the only reference path that can run "
                                        "without an RDMA NIC",
                           "driver": "infinistore.server.main (stock; baseline/ref_server_launch.py "
                                     "tolerates the container's refusal of oom_score_adj) + "
                                     "python -m infinistore.benchmark (stock), one pair per GPU",
                           "clock": "the reference benchmark's own host clock around issue+sync",
                           "build": "unmodified sources, reference Makefile, stand-ins for missing "
                                    "system libraries: baseline/build_reference.sh"},
                "breakdown": {"write_MiBps_rank0": result[1], "read_MiBps_rank0": result[2]},
                "e2e": e2e_json, "gpu_launches": 0,
            }))
    if dist is not None:
        dist.destroy_process_group()


def bind_to_gpu_numa_node(index: int):
    """Pin this process (and the threads it starts later) to the CPUs of the NUMA node the
    GPU hangs off, so that pinned host buffers are first-touched on that node: with 8 ranks
    streaming from host memory at once, remote-node buffers cost ~20 % of the H2D rate
    (round 1: e2e scaling 0.80 at N = 8).  Returns the node or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = int(vis.split(",")[index]) if vis else index
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]  # 00000000:1b:00.0 -> 0000:1b:00.0
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:  # noqa: BLE001 - best effort (containers may hide sysfs)
        pass
    return None


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return
    if args.quick:
        args.size_mb, args.rounds, args.no_extra = min(args.size_mb, 256), min(args.rounds, 2), True

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa_node = bind_to_gpu_numa_node(local_rank)  # before any pinned allocation

    import numpy as np
    import torch

    import infinistore_b200 as ist
    from infinistore_b200 import _infinistore as native
    from infinistore_b200.utils import ClockSampler

    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (run it through gpurun)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(x: float, op) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def allmax(x):
        return allreduce(x, dist.ReduceOp.MAX) if dist else x

    def allmin(x):
        return allreduce(x, dist.ReduceOp.MIN) if dist else x

    def allsum(x):
        return allreduce(x, dist.ReduceOp.SUM) if dist else x

    block_bytes = args.block_kb * 1024
    size_bytes = args.size_mb << 20
    nblocks = size_bytes // block_bytes
    layers = args.layers
    while nblocks % layers != 0 and layers > 1:
        layers //= 2
    per_layer = nblocks // layers
    elems = block_bytes // 2  # bf16 KV pages
    rounds = max(1, args.rounds)
    e2e_steps = 0 if args.no_e2e else 2

    # ---- one pool shard per rank; sized to what the GPU has left after the page tensors
    free_b, _total_b = torch.cuda.mem_get_info(dev)
    reserve = 2 * size_bytes + (12 << 30)  # src + dst + CE roofline peer buffer + slack
    auto_pool = max(2 * size_bytes, min(112 << 30, free_b - reserve))
    pool_bytes = (args.pool_gb << 30) if args.pool_gb else auto_pool
    pool_rounds = max(1, (pool_bytes - (64 << 20)) // size_bytes - 1)  # rounds per epoch
    base_port = args.base_port or (23000 + (int(os.environ.get("MASTER_PORT", "0")) % 2000))
    scfg = native.ServerConfig()
    scfg.service_port = base_port + rank
    scfg.host = "127.0.0.1"
    scfg.pool_backend = "hbm"
    scfg.pool_devices = [local_rank]
    scfg.minimal_allocate_size = max(16, min(args.block_kb, 64))
    scfg.prealloc_bytes = (pool_rounds + 1) * size_bytes + (64 << 20)
    scfg.log_level = "warning"
    server = native.Server(scfg)
    server.start()
    barrier()

    peer = (rank + 1) % world
    ccfg = ist.ClientConfig(host_addr="127.0.0.1", service_port=base_port + peer,
                            connection_type=ist.TYPE_RDMA, log_level="warning",
                            device=local_rank, device_lookup=not args.host_lookup,
                            copy_variant=args.variant, max_ctas=args.max_ctas,
                            streams=args.streams, pipe_stage_kb=args.stage_kb,
                            pipe_ring_kb=args.ring_kb)
    conn = ist.InfinityConnection(ccfg)
    conn.connect()

    # ---- synthetic KV pages (bf16), far larger than L2 (126 MB): nothing is served from cache
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    src = torch.empty(nblocks * elems, device=dev, dtype=torch.bfloat16)
    chunk = 64 << 20
    for a in range(0, src.numel(), chunk):  # fp32 randn of the whole tensor would not fit twice
        n = min(chunk, src.numel() - a)
        src[a:a + n] = torch.randn(n, device=dev, dtype=torch.float32, generator=gen).to(torch.bfloat16)
    dst = torch.zeros_like(src)
    conn.register_mr(src)
    conn.register_mr(dst)
    offsets = [i * elems for i in range(nblocks)]
    offsets_np = np.asarray(offsets, dtype=np.int64)
    stream = torch.cuda.Stream(device=dev)
    key_rng = random.Random(1234 + rank)  # same keys every run with the same arguments

    def fresh_round():
        """Keys, reserved pool blocks and the (key, offset) list of one round (untimed)."""
        tag = f"{key_rng.getrandbits(128):032x}"
        keys = [f"{tag}-{i:07d}" for i in range(nblocks)]
        remote = conn.allocate_rdma(keys, block_bytes)
        return remote, list(zip(keys, offsets))

    host_t = {"issue_write": 0.0, "sync_write": 0.0, "issue_read": 0.0, "sync_read": 0.0}

    def run_round(remote, blocks, record=False):
        t0 = time.perf_counter()
        for l in range(layers):
            a, b = l * per_layer, (l + 1) * per_layer
            conn.rdma_write_cache(src, offsets_np[a:b], elems, remote[a:b])
        t1 = time.perf_counter()
        conn.sync()
        t2 = time.perf_counter()
        for l in range(layers):
            a, b = l * per_layer, (l + 1) * per_layer
            conn.read_cache(dst, blocks[a:b], elems)
        t3 = time.perf_counter()
        conn.sync()
        t4 = time.perf_counter()
        if record:
            host_t["issue_write"] += t1 - t0
            host_t["sync_write"] += t2 - t1
            host_t["issue_read"] += t3 - t2
            host_t["sync_read"] += t4 - t3

    def new_epoch(nrounds):
        """Empty this rank's pool shard and reserve blocks for `nrounds` rounds (untimed)."""
        barrier()          # nobody is still reading the shard we are about to purge
        server.purge()
        barrier()
        return [fresh_round() for _ in range(nrounds)]  # allocation is outside the timing

    def run_rounds(total_rounds, record):
        """Returns the summed device time (ms) of the timed regions: each epoch's rounds are
        bracketed by barrier + synchronize on both sides and timed with CUDA events."""
        total_ms = 0.0
        remaining = total_rounds
        while remaining > 0:
            n_ep = min(remaining, pool_rounds)
            prepared = new_epoch(n_ep)
            dst.zero_()
            torch.cuda.synchronize()
            barrier()
            ev0 = torch.cuda.Event(enable_timing=True)
            ev1 = torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for r in range(n_ep):
                run_round(*prepared[r], record=record)
            ev1.record(stream)
            torch.cuda.synchronize()
            barrier()
            total_ms += ev0.elapsed_time(ev1)
            remaining -= n_ep
            del prepared
        return total_ms

    with torch.cuda.stream(stream):
        run_rounds(args.warmup * rounds, record=False)
        torch.cuda.synchronize()
        assert args.warmup == 0 or torch.equal(src, dst), "read-back mismatch after warm-up"
        launches0 = conn.stats()["kernel_launches"]
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms = run_rounds(args.steps * rounds, record=True)
        clocks = sampler.stop()
        launches = conn.stats()["kernel_launches"] - launches0
        nr = args.steps * rounds
        w_ms = (host_t["issue_write"] + host_t["sync_write"]) / nr * 1e3
        r_ms = (host_t["issue_read"] + host_t["sync_read"]) / nr * 1e3
        breakdown = {"write_phase_ms": round(w_ms, 3), "read_phase_ms": round(r_ms, 3),
                     "write_phase_GBps": round(size_bytes / w_ms / 1e6, 1),
                     "read_phase_GBps": round(size_bytes / r_ms / 1e6, 1),
                     **{"host_" + k + "_ms_per_round": round(v / nr * 1e3, 3)
                        for k, v in host_t.items()},
                     "cpus": len(os.sched_getaffinity(0)), "numa_node": numa_node,
                     "epochs": -(-nr // pool_rounds), "rounds_per_epoch": int(pool_rounds)}
    ok = bool(torch.equal(src, dst))
    if args.dump_outputs:
        # one position per stride, drawn from a fixed seed: the same sample for the same arguments
        stride = -(-dst.numel() // ((32 << 20) // 4 // world))
        n = -(-dst.numel() // stride)
        pos = np.arange(n) * stride + np.random.default_rng(rank).integers(0, stride, n)
        pos = np.minimum(pos, dst.numel() - 1)
        sample = dst.index_select(0, torch.from_numpy(pos).to(dev)).float().cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "dst_sample.npy" if world == 1 else f"dst_sample_rank{rank}.npy"
        np.save(os.path.join(args.dump_outputs, name), sample)

    ms_max = allmax(ms)
    ms_per_step = ms_max / args.steps
    bytes_per_step = 2 * size_bytes * rounds  # write + read, per GPU
    value = world * bytes_per_step / (ms_per_step * 1e-3) / 1e9

    # ---- independent rooflines, measured now on this box by the COPY ENGINE (no kernel of
    #      this repo): every rank copies 1 GiB to its ring peer at the same time
    roof = {"nominal_nvlink_GBps_per_dir_per_gpu": 900}
    try:
        ce_bytes = 1 << 30
        a = torch.empty(ce_bytes, dtype=torch.uint8, device=dev)
        tgt = torch.device("cuda", (local_rank + 1) % world) if world > 1 else dev
        b = torch.empty(ce_bytes, dtype=torch.uint8, device=tgt)
        for _ in range(2):
            b.copy_(a, non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(8):
            b.copy_(a, non_blocking=True)
        e1.record()
        e1.synchronize()
        ce = 8 * ce_bytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
        barrier()
        ce_min = allmin(ce)
        del a, b
        if world == 1:
            roof.update({"ce_local_copy_GBps": round(ce_min, 1),
                         "what": "cudaMemcpyAsync D2D on the same GPU, payload GB/s (each byte "
                                 "read once + written once)"})
        else:
            roof.update({"ce_ring_GBps_per_gpu": round(ce_min, 1),
                         "what": "cudaMemcpyPeerAsync to the ring peer, all ranks at once (every "
                                 "link busy in both directions), min over ranks"})
        roof["fraction_of_copy_engine"] = round(value / (world * ce_min), 3)
    except Exception as e:  # noqa: BLE001
        roof["ce_error"] = repr(e)[:200]
    if world > 1:
        roof["fraction_of_nominal_900"] = round(value / (world * 900.0), 3)
    else:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:  # noqa: BLE001
            pass
        hbm = peaks.get("hbm_gbs", 6650.0)
        roof["measured_hbm_copy_GBps"] = hbm
        roof["fraction_of_measured_hbm_copy"] = round(value / (hbm / 2), 3)

    # ---- end to end: pinned host pages -> H2D (layer-wise, overlapped) -> write -> sync ->
    #      read -> sync, every round; D2H of the result at the end of the step
    e2e = None
    if e2e_steps:
        host_src = torch.empty(nblocks * elems, dtype=torch.bfloat16).pin_memory()
        host_src.copy_(src.cpu())
        host_out = torch.empty(elems + 1, dtype=torch.bfloat16).pin_memory()
        h2d_bytes = size_bytes * rounds
        d2h_bytes = (elems + 1) * 2

        # The inputs of round r+1 stream in over PCIe (their own stream, one event per layer)
        # while round r is read back: `src` is free as soon as the write phase has been
        # sync()ed.  Without this the link idles for the whole read phase of every round
        # (7 ms of 88 at N >= 2: the store's time then shows up 1:1 in the end-to-end number).
        copy_stream = torch.cuda.Stream(device=dev)
        layer_ready = [torch.cuda.Event() for _ in range(layers)]

        def h2d_round():
            copy_stream.wait_stream(stream)      # whatever still reads `src` has been issued
            with torch.cuda.stream(copy_stream):
                for l in range(layers):
                    a, b = l * per_layer, (l + 1) * per_layer
                    src[a * elems:b * elems].copy_(host_src[a * elems:b * elems], non_blocking=True)
                    layer_ready[l].record(copy_stream)

        def e2e_step(prepared):
            with torch.cuda.stream(stream):
                h2d_round()
                for i, (remote, blocks) in enumerate(prepared):
                    for l in range(layers):
                        a, b = l * per_layer, (l + 1) * per_layer
                        stream.wait_event(layer_ready[l])   # the page mover waits for `stream`
                        conn.rdma_write_cache(src, offsets_np[a:b], elems, remote[a:b])
                    conn.sync()
                    if i + 1 < len(prepared):
                        h2d_round()
                    for l in range(layers):
                        a, b = l * per_layer, (l + 1) * per_layer
                        conn.read_cache(dst, blocks[a:b], elems)
                    conn.sync()
                same = (dst[-elems:] == src[-elems:]).all().to(torch.bfloat16).reshape(1)
                host_out[:elems].copy_(dst[:elems], non_blocking=True)
                host_out[elems:].copy_(same, non_blocking=True)
                stream.synchronize()
            return float(host_out[elems].item())

        good = 1.0
        dt = 0.0
        e2e_step(new_epoch(1))  # warm-up: one round
        done = 0
        while done < e2e_steps:
            # an epoch holds pool_rounds rounds: run as many whole steps as fit, else split a step
            prepared = new_epoch(min(pool_rounds, rounds))
            need = rounds
            barrier()
            t0 = time.perf_counter()
            while need > 0:
                take = prepared[:need]
                good = min(good, e2e_step(take))
                need -= len(take)
                if need > 0:
                    torch.cuda.synchronize()
                    dt += time.perf_counter() - t0
                    prepared = new_epoch(min(pool_rounds, need))
                    barrier()
                    t0 = time.perf_counter()
            torch.cuda.synchronize()
            dt += time.perf_counter() - t0
            done += 1
        dt_max = allmax(dt)
        ok = ok and good == 1.0
        e2e = {"value": round(world * bytes_per_step * e2e_steps / dt_max / 1e9, 2), "unit": "GB/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
               "steps": e2e_steps, "ms_per_step": round(dt_max / e2e_steps * 1e3, 3),
               "pinned_numa_node": numa_node,
               "how": "per round: pinned host pages -> H2D layer by layer on a copy stream, each "
                      "layer written as soon as it has landed; sync; read back; sync - the next "
                      "round's H2D runs under the read phase; D2H of one page + the check flag "
                      "at the end of the step"}
        del host_src

    # ---- extras: latency percentiles, emulated baselines, BASELINE.json configs 3-5
    extra, baselines, vs_baseline = None, None, None
    if not args.no_extra:
        import importlib.util

        # bench/ is a directory next to this file (bench.py): load the module by path
        spec = importlib.util.spec_from_file_location(
            "istore_bench_configs", os.path.join(ROOT, "bench", "configs.py"))
        xc = importlib.util.module_from_spec(spec)
        sys.modules["istore_bench_configs"] = xc  # dataclasses resolve annotations through it
        spec.loader.exec_module(xc)

        ctx = xc.Ctx(dist=dist, rank=rank, world=world, local=local_rank, dev=dev,
                     base_port=base_port + 100, barrier=barrier, allmax=allmax, allsum=allsum,
                     allmin=allmin)
        extra = {}
        barrier()
        server.purge()
        barrier()
        try:
            extra["latency_us"] = xc.latency(ctx, base_port + peer)
        except Exception as e:  # noqa: BLE001
            extra["latency_us"] = {"error": repr(e)[:300]}
        try:
            baselines = xc.baselines(ctx, block_bytes)
            ref_gbps = baselines.get("reference_localgpu_pattern", {}).get("aggregate_GBps")
            if ref_gbps:
                vs_baseline = round(value / ref_gbps, 1)
        except Exception as e:  # noqa: BLE001
            baselines = {"error": repr(e)[:300]}
    all_ok = allsum(0.0 if ok else 1.0) == 0.0
    total_launches = int(allsum(float(launches)))
    conn.close()
    barrier()
    server.stop()
    del src, dst
    torch.cuda.empty_cache()
    if extra is not None and world >= 2:
        for name, fn in (("config3_fanin", xc.fanin), ("config5_fp8_ring", xc.fp8_ring),
                         ("config4_nvls_bcast", xc.nvls_bcast)):
            try:
                extra[name] = fn(ctx)
            except Exception as e:  # noqa: BLE001
                extra[name] = {"error": repr(e)[:300]}
            barrier()

    if rank == 0:
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": vs_baseline,
            "dtype": "bf16", "data": "synthetic random KV pages, fresh keys every round",
            "verified": all_ok, "impl": "b200",
            "config": {"model": "paged-KV blocks", "block_kb": args.block_kb,
                       "bytes_per_gpu_per_step": bytes_per_step, "rounds_per_step": rounds,
                       "phase_bytes": size_bytes, "global_batch": nblocks * world,
                       "seq_len": None, "layers_per_phase": layers,
                       "parallelism": f"{world} pool shards, ring placement (rank r -> GPU (r+1)%N)",
                       "l2": f"working set {2 * size_bytes >> 20} MiB per GPU per round >> 126 MB L2 "
                             "(no flush needed)",
                       "variant": args.variant, "streams": args.streams,
                       "pipe_stage_kb": args.stage_kb or "default", "pipe_ring_kb": args.ring_kb or "default",
                       "lookup": "host" if args.host_lookup else "device-index",
                       "phase_sync": True, "timed_region_s": round(ms_max / 1e3, 3)},
            "roofline": roof,
            "clocks": clocks, "gpu_launches": total_launches, "e2e": e2e,
            "breakdown": breakdown, "baselines": baselines, "extra": extra,
        }
        if vs_baseline is not None:
            out["vs_baseline_note"] = ("value / (aggregate GB/s of the reference's LOCAL_GPU "
                                       "data-movement pattern EMULATED with library calls in "
                                       "this run); the reference itself is not buildable offline")
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
