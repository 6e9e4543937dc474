#!/usr/bin/env python
"""bench.py -- the measurement contract of this repository.

    python bench.py --gpus N --steps K --warmup W              (N = 1: plain python; N > 1: torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py ... --dump-outputs DIR                     (also writes what the last timed step computed)

Workload (BASELINE.json `metric`: "Mpix/s encode+decode 8K RGB q75"):  one STEP = encode one 7680x4320
RGB 4:4:4 frame at q75, restart interval 36, non-interleaved, then decode the JPEG just produced.
Frames are synthetic "S-photo" images (SURVEY.md section 8d), one distinct frame per rank.

  value   : Mpix/s with every input already resident in HBM: the raw frame for the encoder, the JPEG BYTES for the
            decoder (its marker scan K0 runs inside the timed region; nothing the host derived from the entropy-coded
            bytes is reused except the scan extents of the header walk).  Timed with CUDA events on the coder's stream
            around exactly K steps of every GPU stage; max over ranks; aggregate over ranks (weak scaling).
  e2e     : the same metric through the reference-facing C API (gpujpeg_encoder_encode /
            gpujpeg_decoder_decode) with HOST buffers, strictly SERIAL calls on one coder pair (the reference's own
            method: `gpujpegtool -n`, README.md:93-100): pinned host RGB in, host JPEG out, host JPEG in, host RGB out
            -- H2D/D2H and the host codestream writer/reader inside the timed region.  `e2e.pipelined_*` is the same
            loop from several host threads / coder pairs / streams (PCIe full duplex), reported beside it.
  roofline: for the slowest GPU stage: algorithmic bytes of SURVEY.md section 8d (9 B/pixel for the
            transform kernels, 6+c for the Huffman kernels) / its CUDA-event time / measured HBM peak.
  cpu_baseline / --impl reference : the CPU oracle (oracle/liboracle.so, a port of the reference's CPU
            path, byte-identical to the reference's own gpujpeg_huffman_cpu_* code) on all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, QUALITY, RST = 7680, 4320, 75, 36
WORKLOADS = {"8k": (7680, 4320, 36), "4k": (3840, 2160, 24), "hd": (1920, 1080, 24), "16k": (15360, 8640, 36)}
DUMP_VALUES = 1 << 22   # values kept per dumped array: three arrays of at most 16 MiB each in float32


def dump_outputs(directory, arrays):
    """--dump-outputs: each array as DIR/<name>.npy in float32 (exact for the u8 / i16 outputs of the codec).  An array of more
    than DUMP_VALUES values is reduced to the values at DUMP_VALUES positions drawn by a fixed seed, so that two builds run
    with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a).reshape(-1)
        if a.size > DUMP_VALUES:
            a = a[np.sort(np.random.default_rng(0).integers(0, a.size, DUMP_VALUES))]
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float32))


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions (B200_PROFILING.md clocks line).  NVML in a thread
    of this process (the counters nvidia-smi prints; ~2 ms period, so even a 10 ms timed region is covered);
    falls back to an `nvidia-smi -lms` child when the NVML binding is missing."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.samples, self.proc, self.index, self.run, self.thread, self.src = [], None, index, False, None, None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            bits = [nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                    nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap]
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while self.run:
                    try:
                        r = get_reasons(h)
                        self.samples.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx)] +
                                            ["Active" if r & b else "Not Active" for b in bits])
                    except Exception:
                        pass
                    time.sleep(0.002)

            self.run, self.src = True, "nvml"
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.run = False
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.src = "nvidia-smi"
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def stop(self):
        self.run = False
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        reasons = sorted({self.NAMES[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": self.src}


def bind_to_gpu_numa_node(local):
    """Pins this rank's host threads (and, by first touch, its pinned buffers) to the NUMA node its GPU hangs off: with
    8 ranks each moving 2 x 100 MB per step through one host, remote-node memory traffic was the end-to-end limiter of
    round 1 (VERDICT weak item 7).  Returns a short description for the record, or None when sysfs does not say."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"gpu": bus, "node": node, "cpus": len(cpus)}
    except Exception:
        return None


def host_cores():
    """cores this process may actually use: min(affinity mask, cgroup CPU quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(quota) // int(period)))
    except Exception:
        pass
    return n


def cpu_baseline(width, height, rst, seconds, threads):
    """Times the oracle port (encode + decode) on the host cores for about `seconds` of CPU work (whole frames);
    returns Mpix/s, the elapsed time and the number of frames."""
    import _oracle as o
    img = o.gen_image("photo", width, height)
    jpeg = o.encode(img, QUALITY, rst, threads=threads)  # warm (page faults, tables)
    frames = 0
    t0 = time.perf_counter()
    while frames < 4 or time.perf_counter() - t0 < seconds:
        jpeg = o.encode(img, QUALITY, rst, threads=threads)
        o.decode(jpeg, threads=threads)
        frames += 1
    dt = time.perf_counter() - t0
    return frames * width * height / dt / 1e6, dt, frames


def cpu_frames(width, height, rst, frames, threads):
    """the oracle port over exactly `frames` whole frames (encode + decode each); returns Mpix/s and the elapsed time"""
    import _oracle as o
    img = o.gen_image("photo", width, height)
    t0 = time.perf_counter()
    for _ in range(frames):
        jpeg = o.encode(img, QUALITY, rst, threads=threads)
        o.decode(jpeg, threads=threads)
    dt = time.perf_counter() - t0
    return frames * width * height / dt / 1e6, dt


def reference_gpu(kind, width, height, rst, iters=10):
    """'The kernel to beat': the reference's own GPU library (compiled in place into oracle/_ref by `make -C oracle refgpu`,
    its CUDA kernels recompiled for sm_100) on the same box, same frame, pinned host buffers obtained through its own
    gpujpeg_image_load_from_file, serial calls, perf_stats on -- in a child process, so that its gpujpeg_* symbols never
    meet the product's.  An extra of the record, not part of any timed region of this benchmark."""
    so = os.path.join(ROOT, "oracle", "_ref", "libgpujpeg_refgpu.so")
    if not os.path.exists(so):
        return {"unavailable": "oracle/_ref/libgpujpeg_refgpu.so not built"}
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_refgpu.py"), "bench", kind, str(width), str(height),
                              str(QUALITY), str(rst), str(iters)], capture_output=True, text=True, timeout=300)
        r = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as exc:   # the extra must never take the benchmark down
        return {"unavailable": repr(exc)[:200]}
    npix = width * height
    for k in ("encode_ms_e2e", "encode_ms_gpu", "decode_ms_e2e", "decode_ms_gpu"):
        if r.get(k):
            r[k.replace("_ms_", "_mpix_s_")] = round(npix / (r[k] * 1e-3) / 1e6, 1)
    if r.get("encode_ms_e2e") and r.get("decode_ms_e2e"):
        r["e2e_mpix_s"] = round(npix / ((r["encode_ms_e2e"] + r["decode_ms_e2e"]) * 1e-3) / 1e6, 1)
    if r.get("encode_ms_gpu") and r.get("decode_ms_gpu"):
        r["in_gpu_mpix_s"] = round(npix / ((r["encode_ms_gpu"] + r["decode_ms_gpu"]) * 1e-3) / 1e6, 1)
    return r


def run_reference(args):
    """--impl reference: the CPU path on this box's host cores.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    width, height, rst = WORKLOADS[args.size]
    cores = host_cores()
    for _ in range(max(0, args.warmup)):
        cpu_frames(width, height, rst, 1, cores)
    mpix, dt = cpu_frames(width, height, rst, args.steps, cores)
    line = {
        "impl": "reference", "metric": "Mpix/s encode+decode %s RGB q75" % args.size, "value": round(mpix, 2), "unit": "Mpix/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+i32", "data": "synthetic",
        "config": {"workload": "%dx%d RGB 4:4:4 q%d rst%d non-interleaved, encode+decode per step (S-photo)" % (width, height, QUALITY, rst)},
        "cpu_baseline": {"value": round(mpix, 2), "unit": "Mpix/s", "cores": cores, "kind": "port",
                         "sample": "%d full frames, oracle port (bit-identical to the reference's gpujpeg_huffman_cpu_* + "
                                   "gpujpeg_idct_cpu; restated colour/FDCT), OpenMP over segments/blocks" % args.steps},
        "e2e": {"value": round(mpix, 2), "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def nccl_transport_line(path):
    """What carries the peer traffic, for the record: the GPU0 row of `nvidia-smi topo -m` (NV<n> = n NVLink links through
    the NVSwitch fabric).  (NCCL_DEBUG=INFO would say it in NCCL's own words, but it also prints to stdout, which must
    carry exactly one JSON line; the measured scatter rate next to this entry -- ~700 GB/s, eleven times PCIe gen5 -- is
    the evidence that the path is NVLink peer-to-peer and not a bounce through the host.)"""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout.splitlines()
        row = [ln for ln in out if ln.startswith("GPU0")]
        return " ".join(row[0].replace("\x1b[4m", "").replace("\x1b[0m", "").split()[:9]) if row else None
    except Exception:
        return None


def scatter_gather_extra(g, torch, dist, rank, world, dev, enc, dec, frame_dev, width, height, rst, steps, nccl_log):
    """SURVEY.md section 8e "scattered from GPU 0": rank 0 holds one raw frame per rank on ITS GPU, sends them to their
    owners (NCCL point-to-point, gpujpeg_b200/batch.py), every rank encodes and decodes its frame through the C API with
    device buffers, and the JPEG streams are gathered (gather-v) on rank 0.  Timed on the device, max over ranks."""
    from gpujpeg_b200 import batch as bt
    npix = width * height
    frames = [frame_dev.clone() for _ in range(world)] if rank == 0 else None
    d_out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)

    def once():
        mine = bt.scatter_frames(frames, world, (height, width, 3), src=0, device=dev)
        streams = []
        for f in mine:
            j = enc.encode(f, QUALITY, rst)
            dec.decode(j, out=d_out)
            streams.append(torch.from_numpy(j).to(dev))
        return bt.gather_streams(streams, world, dst=0, device=dev)

    def timed_transfer(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier(); torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        dist.barrier(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    for _ in range(2):
        got = once()
    ms = timed_transfer(once, steps)
    # the scatter alone: what the transport gives (bytes leaving rank 0 / time)
    ms_scatter = timed_transfer(lambda: bt.scatter_frames(frames, world, (height, width, 3), src=0, device=dev), steps)
    out = None
    if rank == 0:
        out = {"value": round(world * npix / (ms * 1e-3) / 1e6, 1), "unit": "Mpix/s", "ms_per_step": round(ms, 3),
               "what": "one %dx%d frame per rank: NCCL send/recv of the raw frames from rank 0's GPU to their owners, encode + "
                       "decode through the C API with device buffers, gather-v of the JPEG streams to rank 0" % (width, height),
               "scatter_ms": round(ms_scatter, 3),
               "scatter_gbs": round((world - 1) * npix * 3 / (ms_scatter * 1e-3) / 1e9, 1),
               "gathered_stream_bytes": [int(x.numel()) for x in got],
               "peer_path": nccl_transport_line(nccl_log)}
    return out


def run_batch(args, g, o, torch, dist, rank, world, local, dev, numa, nccl_log):
    """BASELINE.json config 5 (`--size 16k --batch 32`): a FIXED batch of frames, frame f on rank f mod N (strong scaling).
    Two numbers per run, both whole-batch Mpix/s, device-timed, max over ranks:
      value            frames resident on their owners' GPUs: gpujpeg_encoder_encode (GPU image in, JPEG to the host) +
                       gpujpeg_decoder_decode (JPEG from the host, pixels into a CUDA buffer) per frame
      scattered.value  all raw frames on rank 0's GPU first: NCCL scatter to the owners, the same coding, gather-v of
                       the streams on rank 0"""
    import numpy as np
    from gpujpeg_b200 import batch as bt
    width, height, rst = WORKLOADS[args.size]
    npix, n_frames = width * height, args.batch
    mine = bt.my_frames(n_frames, world, rank)
    base = [torch.from_numpy(o.gen_image(args.kind, width, height, seed=12345 + k)) for k in range(min(4, n_frames))]
    stream = torch.cuda.current_stream().cuda_stream
    enc = g.Encoder(stream=stream, pinned_output=True)
    dec = g.Decoder(stream=stream)
    d_frames = [base[f % len(base)].to(dev) for f in mine]
    d_out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    sizes = []

    import ctypes
    p_enc = g.api.default_parameters(QUALITY, rst)
    p_img = g.api.image_parameters(width, height)

    def code(f):
        """encode a device-resident frame, decode the stream into a device buffer; returns the stream as a zero-copy view"""
        addr, size = enc.encode_raw(f, p_enc, p_img, device=True)
        dec.decode_raw(addr, size, g.api.GPUJPEG_DECODER_OUTPUT_CUSTOM_CUDA_BUFFER, d_out.data_ptr())
        return np.ctypeslib.as_array((ctypes.c_uint8 * size).from_address(addr))

    def step_resident():
        del sizes[:]
        for f in d_frames:
            sizes.append(code(f).size)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    ms = timed(step_resident, args.steps)
    value = n_frames * npix / (ms * 1e-3) / 1e6

    scattered = None
    if world > 1:
        all_frames = [base[f % len(base)].to(dev) for f in range(n_frames)] if rank == 0 else None

        def step_scattered():
            got = bt.scatter_frames(all_frames, n_frames, (height, width, 3), src=0, device=dev)
            streams = []
            for f in got:
                streams.append(torch.from_numpy(code(f)).to(dev))   # the copy to the device takes the bytes before the next encode reuses the buffer
            return bt.gather_streams(streams, n_frames, dst=0, device=dev)

        for _ in range(max(1, args.warmup - 1)):
            step_scattered()
        ms_sc = timed(step_scattered, args.steps)
        ms_only = timed(lambda: bt.scatter_frames(all_frames, n_frames, (height, width, 3), src=0, device=dev), args.steps)
        sent = (n_frames - len(bt.my_frames(n_frames, world, 0))) * npix * 3
        scattered = {"value": round(n_frames * npix / (ms_sc * 1e-3) / 1e6, 1), "unit": "Mpix/s", "ms_per_step": round(ms_sc, 3),
                     "scatter_ms": round(ms_only, 3), "scatter_gbs": round(sent / (ms_only * 1e-3) / 1e9, 1),
                     "peer_path": nccl_transport_line(nccl_log)}
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        emit({
            "metric": "Mpix/s encode+decode %s RGB q75, batch of %d frames" % (args.size, n_frames), "value": round(value, 1),
            "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32+i32 (u8 in, i16 coefficients)",
            "data": "synthetic",
            "config": {"workload": "%dx%d RGB 4:4:4 q%d rst%d non-interleaved, batch of %d S-%s frames (%d distinct), frame f on rank "
                                   "f mod %d, encode+decode per frame through the C API with device buffers, JPEG via the host"
                                   % (width, height, QUALITY, rst, n_frames, args.kind, len(base), world),
                       "l2": "inputs larger than L2 (%.0f MB raw per frame)" % (npix * 3 / 1e6),
                       "sharding": "frames round-robin over ranks, no data-path collective; `scattered`: NCCL send/recv of raw "
                                   "frames from rank 0 + gather-v of the streams"},
            "scattered": scattered, "jpeg_bytes_per_frame": int(np.mean(sizes)) if sizes else None,
            "gpu_launches": 6 * len(mine) * args.steps, "clocks": clocks, "numa": numa})
    enc.close()
    dec.close()
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """the ONE JSON line of the contract, on the process's real stdout"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def quiet_stdout():
    """libraries (NCCL, the CUDA runtime, child processes) may print to file descriptor 1; stdout must carry exactly one
    JSON line, so everything else is sent to stderr and the JSON line is written to a saved copy of the real stdout"""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", default="8k", choices=sorted(WORKLOADS))
    ap.add_argument("--kind", default="photo", choices=["photo", "random", "gradient"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    # the headline workload is 4:4:4 non-interleaved (BASELINE.json); these two select the SURVEY 8f rank-2 variants
    ap.add_argument("--subsampling", default="4:4:4", choices=["4:4:4", "4:2:2", "4:2:0", "4:4:0"])
    ap.add_argument("--interleaved", type=int, default=0, choices=[0, 1])
    # end-to-end arm: number of coder pairs driven concurrently, each by its own host thread on its own CUDA stream
    # (the reference's contract: one coder = one stream, instances are independent).  1 = strictly serial calls.
    ap.add_argument("--e2e-workers", type=int, default=3)
    # BASELINE.json config 5: a fixed batch of frames sharded round-robin over the ranks (strong scaling); with --batch the
    # step is the whole batch.  `--size 16k --batch 32` is the configuration the reference's north star names.
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step of each timed path "
                    "computed (rank 0's frame): the encoder's quantised coefficients and the decoded pixels of the resident "
                    "path, the JPEG stream of the end-to-end path; float32 .npy files, large ones as a fixed seeded sample")
    args = ap.parse_args()
    if args.dump_outputs and (args.batch or args.impl != "b200"):
        ap.error("--dump-outputs applies to the single-frame workload of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None   # before any pinned allocation (first touch)
    nccl_log = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import gpujpeg_b200 as g
    import _oracle as o  # synthetic frame generator only (the checker is never timed here)

    if args.batch > 0:
        return run_batch(args, g, o, torch, dist, rank, world, local, dev, numa, nccl_log)

    width, height, rst = WORKLOADS[args.size]
    npix = width * height
    frame = o.gen_image(args.kind, width, height, seed=12345 + rank)
    h_raw = torch.from_numpy(frame).pin_memory()
    d_raw = h_raw.to(dev, non_blocking=True)
    stream = torch.cuda.current_stream().cuda_stream
    enc = g.Encoder(stream=stream, pinned_output=True)
    dec = g.Decoder(stream=stream)

    # one reference-facing call each: sets up geometry/tables and leaves the decoder's inputs on the device
    headline = args.subsampling == "4:4:4" and args.interleaved == 0
    lh, lv = g.api.SUBSAMPLING[args.subsampling]
    if not headline:
        # RESTART_AUTO of the reference for this mode [ref: src/gpujpeg_encoder.c:290-317]
        rst = 12 * 3 if not args.interleaved else (12 if args.subsampling == "4:4:4" else 6)
    coef_bpp = 2.0 * (1.0 + 2.0 / (lh * lv))   # int16 coefficients per image pixel, all components
    jpeg = enc.encode(d_raw, QUALITY, rst, args.interleaved, subsampling=args.subsampling)
    c_bpp = (jpeg.size - 700) / npix
    h_jpeg = torch.from_numpy(jpeg).pin_memory()
    d_out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    h_out = torch.empty((height, width, 3), dtype=torch.uint8).pin_memory()
    dec.decode(h_jpeg.numpy(), out=d_out)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        enc.run_resident(d_raw, 3)      # K1 + K2 (encode, offsets, compaction)
        dec.run_resident(d_out, 7)      # K0 (marker list + clean stream from the JPEG bytes) + K3 + K4

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident throughput (headline `value`) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()   # runs until the end of the e2e loop: covers every timed region
    for _ in range(args.warmup):
        step_resident()
    ms_total = timed(step_resident, args.steps)
    ms_step = ms_total / args.steps
    outputs = {}
    if args.dump_outputs and rank == 0:   # before the per-stage timings below run the kernels again
        outputs["coefficients"] = enc.coefficients(width, height, (lh, lv), args.interleaved)
        outputs["pixels"] = d_out.cpu().numpy()
    value = world * npix / (ms_step * 1e-3) / 1e6

    # ---- per-stage times for the roofline (same stream, CUDA events, inputs > L2) ----
    stages = {}
    for name, fn in (("k1_fdct", lambda: enc.run_resident(d_raw, 1)), ("k2_huffman_encode", lambda: enc.run_resident(d_raw, 2)),
                     ("k0_marker_scan", lambda: dec.run_resident(d_out, 4)), ("k3_huffman_decode", lambda: dec.run_resident(d_out, 1)),
                     ("k4_idct", lambda: dec.run_resident(d_out, 2))):
        for _ in range(2):
            fn()
        stages[name] = timed(fn, max(5, args.steps // 2)) / max(5, args.steps // 2)

    # ---- end to end through the C API with host buffers ----
    host_img = h_raw.numpy()

    def step_e2e():
        p = g.api.default_parameters(QUALITY, rst, args.interleaved, args.subsampling)
        addr, size = enc.encode_raw(host_img, p, g.api.image_parameters(width, height), device=False)
        dec.decode_raw(addr, size, g.api.GPUJPEG_DECODER_OUTPUT_CUSTOM_BUFFER, h_out.data_ptr())
        return addr, size

    for _ in range(args.warmup):
        jpeg_addr, jpeg_size = step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        jpeg_addr, jpeg_size = step_e2e()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_sync_ms = float(dt.item()) / args.steps * 1e3
    if args.dump_outputs and rank == 0:   # the encoder's JPEG buffer stays valid until its next call
        import ctypes
        outputs["jpeg"] = np.ctypeslib.as_array((ctypes.c_uint8 * jpeg_size).from_address(jpeg_addr)).copy()
        dump_outputs(args.dump_outputs, outputs)

    # ---- the same calls from several host threads, one coder pair + one CUDA stream each: step n+1's H2D overlaps
    #      step n's kernels and step n-1's D2H (PCIe is full duplex).  Every step still copies its 99.5 MB in and its
    #      99.5 MB out inside the timed region; nothing is cached between steps. ----
    workers = max(1, args.e2e_workers)
    e2e_pipe_ms = None
    if workers > 1:
        pool = []
        for _ in range(workers):
            st = torch.cuda.Stream(device=dev)
            pool.append((g.Encoder(stream=st.cuda_stream, pinned_output=True), g.Decoder(stream=st.cuda_stream),
                         torch.empty((height, width, 3), dtype=torch.uint8).pin_memory(), st))
        counter = {"next": 0, "limit": 0}
        lock = threading.Lock()
        failed = []

        def work(slot):
            e, d, out, _ = pool[slot]
            try:
                torch.cuda.set_device(local)
                while True:
                    with lock:
                        if counter["next"] >= counter["limit"]:
                            return
                        counter["next"] += 1
                    p = g.api.default_parameters(QUALITY, rst, args.interleaved, args.subsampling)
                    addr, size = e.encode_raw(host_img, p, g.api.image_parameters(width, height), device=False)
                    d.decode_raw(addr, size, g.api.GPUJPEG_DECODER_OUTPUT_CUSTOM_BUFFER, out.data_ptr())
            except Exception as exc:   # a worker must never die silently: the number would look better than it is
                failed.append(exc)

        def run(n):
            counter["next"], counter["limit"] = 0, n
            ts = [threading.Thread(target=work, args=(i,)) for i in range(workers)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
            assert not failed, failed

        run(max(args.warmup, workers))
        barrier()
        t0 = time.perf_counter()
        run(args.steps)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_pipe_ms = float(dt.item()) / args.steps * 1e3
        for e, d, out, _ in pool:
            assert np.array_equal(out.numpy(), h_out.numpy()), "pipelined and serial end-to-end results disagree"
            e.close()
            d.close()
    # ONE rule for the headline: strictly serial calls (the reference's published method); the pipelined figure is
    # reported under its own keys
    e2e_ms = e2e_sync_ms
    used_workers = 1
    e2e_value = world * npix / (e2e_ms * 1e-3) / 1e6
    clocks = sampler.stop() if rank == 0 else None
    assert np.array_equal(h_out.numpy(), d_out.cpu().numpy()), "e2e and resident paths disagree"
    sg_extra = None
    if world > 1 and headline:
        sg_extra = scatter_gather_extra(g, torch, dist, rank, world, dev, enc, dec, d_raw, width, height, rst, max(3, args.steps // 4),
                                        nccl_log)

    if rank == 0:
        peak, peak_kind = hbm_peak()
        alg = {"k1_fdct": 3.0 + coef_bpp, "k2_huffman_encode": coef_bpp + c_bpp, "k3_huffman_decode": coef_bpp + c_bpp,
               "k4_idct": 3.0 + coef_bpp, "k0_marker_scan": 2.0 * c_bpp}
        worst = max((k for k in stages if k != "k0_marker_scan"), key=lambda k: stages[k])
        # DRAM traffic of that kernel from the committed ncu --set full capture of the same workload (per launch)
        traffic = None
        try:
            if args.size == "8k" and args.kind == "photo" and headline:
                tj = json.load(open(os.path.join(ROOT, "profiles", "traffic_8k_photo.json")))["kernels"]
                # the kernels of the stage (K2 = two launches: the coder and k_huff_place; its time above covers both)
                names = {"k1_fdct": ("k_fdct_rgb444",), "k2_huffman_encode": ("k_huff_encode", "k_huff_place"),
                         "k3_huffman_decode": ("k_huff_decode",), "k4_idct": ("k_idct_rgb444",)}[worst]
                hits = [v for k, v in tj.items() if k.startswith(names)]
                if hits:
                    traffic = int(sum(v["dram_bytes_read"] + v["dram_bytes_write"] for v in hits))
        except Exception:
            traffic = None
        roof = {k: alg[k] * npix / (stages[k] * 1e-3) / 1e9 for k in stages}
        path_gbs = (6.0 + 4 * coef_bpp + 2 * c_bpp) * npix / (ms_step * 1e-3) / 1e9
        line = {
            "metric": "Mpix/s encode+decode %s RGB q75" % args.size, "value": round(value, 1), "unit": "Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32+i32 (u8 in, i16 coefficients)", "data": "synthetic",
            "config": {"workload": "%dx%d RGB %s q%d rst%d %s, encode+decode per step, S-%s frame per rank, "
                                   "c=%.3f B/pixel" % (width, height, args.subsampling, QUALITY, rst,
                                                       "interleaved" if args.interleaved else "non-interleaved", args.kind, c_bpp),
                       "l2": "inputs larger than L2 (%.1f MB raw + %.0f MB coefficients per direction)"
                             % (npix * 3 / 1e6, npix * coef_bpp / 1e6),
                       "sharding": "one coder instance per GPU, independent frames, no data-path collective"},
            "stage_ms": {k: round(v, 4) for k, v in stages.items()},
            "roofline": {"bound": "hbm", "kernel": worst, "achieved": round(roof[worst], 1), "peak": peak, "unit": "GB/s",
                         "frac": round(roof[worst] / peak, 4), "traffic": traffic, "peak_source": peak_kind,
                         "all_stages_gbs": {k: round(v, 1) for k, v in roof.items()},
                         "path_achieved_gbs": round(path_gbs, 1), "path_frac": round(path_gbs / peak, 4)},
            "e2e": {"value": round(e2e_value, 1), "unit": "Mpix/s", "ms_per_step": round(e2e_ms, 3),
                    "h2d_bytes_per_step": int(npix * 3 + jpeg_size), "d2h_bytes_per_step": int(jpeg_size + npix * 3),
                    "workers": used_workers,
                    "how": "gpujpeg_encoder_encode + gpujpeg_decoder_decode with pinned host buffers, strictly serial calls on "
                           "one coder pair (the reference's `gpujpegtool -n` method); pipelined_* = the same calls from %d "
                           "host threads, one coder pair and one CUDA stream each.  Inside a call the library moves the frame in "
                           "8 stripes and runs its kernels stripe by stripe behind the copy (DESIGN.md section 5)" % workers,
                    "serial_value": round(world * npix / (e2e_sync_ms * 1e-3) / 1e6, 1), "serial_ms_per_step": round(e2e_sync_ms, 3),
                    "pipelined_value": round(world * npix / (e2e_pipe_ms * 1e-3) / 1e6, 1) if e2e_pipe_ms else None,
                    "pipelined_ms_per_step": round(e2e_pipe_ms, 3) if e2e_pipe_ms else None, "pipelined_workers": workers},
            # per step: K1, K2 (encode, offsets, compaction), K0 (count, scan, write), K3, K4 -- plus one 32-byte memset node
            "gpu_launches": 6 * args.steps,
            "clocks": clocks,
        }
        if not args.no_reference_gpu and world == 1:
            line["extras"] = {"reference_gpu": reference_gpu(args.kind, width, height, rst)}
        if sg_extra is not None:
            line.setdefault("extras", {})["scatter_gather"] = sg_extra
        if numa is not None:
            line["numa"] = numa
        if not args.no_cpu_baseline and world == 1:
            cores = host_cores()
            mpix, sec, nframes = cpu_baseline(width, height, rst, 12.0, cores)
            line["cpu_baseline"] = {"value": round(mpix, 2), "unit": "Mpix/s", "cores": cores, "kind": "port",
                                    "sample": "%d full %dx%d frames encode+decode, %.1f s, OpenMP %d threads (= cgroup CPU quota of the box)" % (nframes, width, height, sec, cores)}
        emit(line)
    enc.close()
    dec.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
