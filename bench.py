#!/usr/bin/env python3
"""bench.py -- decoded cimbar frames/s (1024x1024 mode B) on N B200s, with roofline and CPU baseline.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                      (the CPU restatement of the reference on the host cores)
    python bench.py ... --dump-outputs DIR                     (also write the last timed step's results to DIR/*.npy)

One "step" = one pass of the decode hot path over one batch of synthetic frames resident in HBM:
  K1 fused preprocess+ahash+colour -> K1x exact-walk check -> bit pack -> RS(155,125) -> fountain-chunk masks,
  then (N>1) one NCCL gather of the decoded chunk records to rank 0.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions of every field."""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "decoded cimbar frames/sec (1024x1024 mode-B)"
UNIT = "frames/s"
MODE_NAMES = {68: "B", 67: "Bm", 66: "Bu", 4: "4C", 8: "8C"}


def metric_name(mode_val):
    return METRIC if mode_val == 68 else "decoded cimbar frames/sec (mode %s)" % MODE_NAMES[mode_val]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=10000, help="frames per GPU per step (BASELINE config: 10k)")
    ap.add_argument("--workload", default="clean", choices=["clean", "errors1pct", "noise1pct"],
                    help="clean = BASELINE configs[1] frames; errors1pct = configs[2] (1%% wrong tiles, RS repairs); "
                         "noise1pct = 1%% of the cells replaced by random pixels (forces the exact flood-walk kernel)")
    ap.add_argument("--mode", type=int, default=68, choices=[68, 67, 66, 4, 8],
                    help="cimbar mode_val: 68 = B (headline), 4 = legacy 4C (BASELINE configs[4]), 8 = 8C, 67 = Bm, 66 = Bu")
    ap.add_argument("--sharpen", action="store_true",
                    help="decode with should_preprocess=true (CimbReader.cpp:17-46: 3x3 sharpen + block-7 threshold, inside K1)")
    ap.add_argument("--color-correction", type=int, default=0, choices=[0, 1, 2],
                    help="the reference's color_correction argument (0 = headline configuration; 1 = per-frame von Kries; "
                         "2 = per-frame header fit, the payload then carries consecutive fountain headers)")
    ap.add_argument("--gather", default="window", choices=["window", "window-direct", "nccl", "torch"],
                    help="N > 1: how the chunk records reach rank 0 -- window = a window in rank 0's HBM mapped by every rank over NVLink "
                         "(CUDA IPC), filled by copy-engine pushes on a side stream (cb200_gather_push / wait / release); window-direct = "
                         "the RS kernels store straight into that window (cb200_gather_slot / publish); nccl = cb200_gather_chunks "
                         "(ncclSend/Recv on a side stream, double buffered); torch = torch.distributed.gather on the decode stream "
                         "(round-1 behaviour)")
    ap.add_argument("--camera", action="store_true",
                    help="the camera path: photographs -> scan -> deskew -> decode (libcimbar_b200/camera_bench.py); one GPU")
    ap.add_argument("--fountain", action="store_true",
                    help="BASELINE configs[3]: fountain-encoded file, frames sharded over the ranks, records to rank 0, wirehair "
                         "reassembly checked by SHA-256 (libcimbar_b200/fountain_bench.py)")
    ap.add_argument("--file-mb", type=float, default=30.0, help="--fountain: file size in MB (30 = the config)")
    ap.add_argument("--e2e-frames", type=int, default=256)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-sample", type=int, default=0, help="frames per step for --impl reference (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed (rank 0) as DIR/<name>.npy: the chunk records of "
                         "a fixed, seeded sample of frames, and every frame's chunk mask and frame flags (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.camera or args.fountain):
        ap.error("--dump-outputs applies to the decode path (not to --impl reference, --camera or --fountain)")
    return args


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, chunks, mask, fflags):
    """The last step's results as float32 .npy files.  chunks is (frames, data_bytes) uint8; its rows go out for a sorted
    sample of frames drawn with a fixed seed (all of them when they fit), so that two builds run with the same arguments
    can be compared file by file.  mask (int32, < 2^24) and fflags (uint8) are exact in float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    B, row = chunks.shape
    small = 4 * 3 * B + 4 * 4096                                        # chunk_mask, frame_flags, the row index; .npy headers
    n = min(B, (DUMP_LIMIT_BYTES - small) // (4 * row))
    rows = np.sort(np.random.default_rng(0xD0).choice(B, n, replace=False)) if n < B else np.arange(B)
    sel = torch.from_numpy(rows).to(chunks.device)
    arrays = {"chunks": chunks.index_select(0, sel), "chunks_rows": rows, "chunk_mask": mask, "frame_flags": fflags}
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def k1_traffic_bytes():
    """dram bytes per K1 launch from the committed ncu capture, scaled per frame; None until one exists."""
    p = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def bind_to_gpu_numa_node(index):
    """pin this process (and therefore its pinned staging buffers, first touched after this call) to the CPUs that are local to
    GPU `index`: the end-to-end leg is PCIe-bound, and on a two-socket box half of the GPUs hang off the other socket"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d cpus local to GPU %d" % (len(cpus), index)
    except Exception as e:
        return "not bound (%s)" % type(e).__name__
    return "not bound"


# ------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import libcimbar_b200 as cb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the decode path has no CPU fallback)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B, K, W = args.frames, args.steps, max(args.warmup, 0)

    MV = args.mode
    ctx = cb.Context(MV, max_frames=max(B, args.e2e_frames), device=local)
    info = ctx.info
    K1_ALGO_BYTES = info.frame_bytes + info.total_cells      # the RGB8 frame read once + one result byte per cell
    stream = torch.cuda.Stream(device=dev)           # a real (non-default) stream: handle 0 would mean "context's own"
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # ---- synthetic input, generated on the device: payload -> RS(155,125) -> interleaved cells -> RGB8 frames
    g = torch.Generator(device=dev)
    g.manual_seed(0xC1B4 + rank)
    payload = torch.randint(0, 256, (B, info.data_bytes), dtype=torch.uint8, device=dev, generator=g)
    cc_flags = {0: 0, 1: cb.FLAG_CC_SIMPLE, 2: cb.FLAG_CC_FIT}[args.color_correction]
    if args.sharpen:
        cc_flags |= cb.FLAG_SHARPEN
    if args.color_correction == 2:
        # a fountain stream: every 625-byte chunk starts with FountainMetadata(encode_id, size, block_id) and the block ids
        # of a frame are consecutive (fountain/FountainMetadata.h:16-31) -- that is what CimbReader::init_ccm predicts from
        cpf, cs = info.chunks_per_frame, info.data_bytes // info.chunks_per_frame
        pv = payload.view(B, cpf, cs)
        size = 625 * 4000                                                # a multiple of the chunk size: no "radioactive" block id
        bid = (torch.arange(B, device=dev).view(B, 1) * cpf + torch.arange(cpf, device=dev).view(1, cpf)) % 65536
        pv[:, :, 0] = (1 & 0x7F) | ((size >> 17) & 0x80)
        pv[:, :, 1] = (size >> 16) & 0xFF
        pv[:, :, 2] = (size >> 8) & 0xFF
        pv[:, :, 3] = size & 0xFF
        pv[:, :, 4] = (bid >> 8).to(torch.uint8)
        pv[:, :, 5] = (bid & 0xFF).to(torch.uint8)
    cells = torch.empty((B, info.total_cells), dtype=torch.uint8, device=dev)
    ctx.encode_cells_dev(payload.data_ptr(), B, cells.data_ptr())
    if args.workload == "errors1pct":
        # replace 1 % of the cells (124 per frame) by a different valid tile/colour: RS must repair them
        k = info.total_cells // 100
        pos = torch.rand((B, info.total_cells), device=dev, generator=g).argsort(dim=1)[:, :k]
        nvals = 1 << (info.symbol_bits + info.color_bits)
        delta = torch.randint(1, nvals, (B, k), dtype=torch.uint8, device=dev, generator=g)
        cells.scatter_(1, pos, (cells.gather(1, pos) + delta) % nvals)
    frames = torch.empty((B, info.image_size_y, info.image_size_x, 3), dtype=torch.uint8, device=dev)
    ctx.render_frames_dev(cells.data_ptr(), B, frames.data_ptr())
    if args.workload == "noise1pct" and MV != 68:
        raise SystemExit("bench.py: --workload noise1pct is only wired for mode 68")
    if args.workload == "noise1pct":
        # overwrite 124 cells per frame with uniform-noise 8x8 tiles: the centre-wins proof fails, K1x decodes the frame
        k = info.total_cells // 100
        idx = cb.interleave_indices(68)          # any permutation of the cells will do for picking positions
        cx = torch.tensor([(62 + 9 * (c % 100), 8 + 9 * (c // 100)) if c < 600 else
                           ((8 + 9 * ((c - 600) % 112), 62 + 9 * ((c - 600) // 112)) if c < 11800 else
                            (62 + 9 * ((c - 11800) % 100), 962 + 9 * ((c - 11800) // 100))) for c in range(info.total_cells)],
                          device=dev)
        for f0 in range(0, B, 256):
            nb = min(256, B - f0)
            pos = torch.rand((nb, info.total_cells), device=dev, generator=g).argsort(dim=1)[:, :k]
            xy = cx[pos]                                             # (nb, k, 2)
            noise = torch.randint(0, 256, (nb, k, 8, 8, 3), dtype=torch.uint8, device=dev, generator=g)
            fi = torch.arange(nb, device=dev).view(nb, 1, 1, 1).expand(nb, k, 8, 8) + f0
            yy = (xy[:, :, 1].view(nb, k, 1, 1) + torch.arange(8, device=dev).view(1, 1, 8, 1)).expand(nb, k, 8, 8)
            xx = (xy[:, :, 0].view(nb, k, 1, 1) + torch.arange(8, device=dev).view(1, 1, 1, 8)).expand(nb, k, 8, 8)
            frames[fi, yy, xx] = noise
    chunks = torch.empty((B, info.data_bytes), dtype=torch.uint8, device=dev)
    mask = torch.empty(B, dtype=torch.int32, device=dev)
    fflags = torch.empty(B, dtype=torch.uint8, device=dev)
    gather_chunks = gather_mask = None
    exchange, gather_kind = None, None
    if world > 1:
        from libcimbar_b200.dist import RecordExchange
        gather_kind = args.gather
        if gather_kind in ("window", "window-direct"):
            # every rank must agree on the path: fall back to NCCL everywhere if any rank cannot map the window
            try:
                exchange = RecordExchange(ctx, gather_kind, B, rank, world)
                okw = 1
            except cb.Cb200Error as e:
                print("bench.py: rank %d cannot use the NVLink window (%s); falling back to --gather nccl" % (rank, e), file=sys.stderr)
                okw = 0
            t = torch.tensor([okw], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t.item()) == 0:
                exchange, gather_kind = None, "nccl"
        if gather_kind == "nccl":
            exchange = RecordExchange(ctx, "nccl", B, rank, world)
        if gather_kind == "torch" and rank == 0:
            gather_chunks = [torch.empty_like(chunks) for _ in range(world)]
            gather_mask = [torch.empty_like(mask) for _ in range(world)]
    torch.cuda.synchronize()
    step_no = [0]

    def step():
        # the one exchange of the path: decoded fountain chunk records -> rank 0 (wirehair ingest side)
        if exchange is None:
            ctx.decode_chunks_dev(frames.data_ptr(), B, chunks.data_ptr(), mask.data_ptr(), fflags.data_ptr(), flags=cc_flags)
            if world > 1:
                dist.gather(chunks, gather_chunks, dst=0)
                dist.gather(mask, gather_mask, dst=0)
            return
        step_no[0] += 1
        sidx = step_no[0]
        pc, pm = exchange.begin(sidx)          # window: this rank's slot in rank 0's HBM; nccl: a local send buffer
        ctx.decode_chunks_dev(frames.data_ptr(), B, pc, pm, fflags.data_ptr(), flags=cc_flags)
        exchange.end(sidx)
        if rank == 0 and sidx > 1:             # the records of the previous step: complete while this step decodes
            exchange.collect(sidx - 1)
            exchange.release(sidx - 1)

    def drain():
        if exchange is not None and rank == 0 and step_no[0] > 0:
            exchange.collect(step_no[0])
            exchange.release(step_no[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx.set_timing(False)
    for _ in range(max(W, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ctx.set_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = cb.launch_count()
    e0.record()
    for _ in range(K):
        step()
    drain()                                          # rank 0: the last step's records have arrived too
    e1.record()
    launches = cb.launch_count() - launches0         # counted by the library at every launch site
    barrier()
    sampler.stop_flag = True
    elapsed_ms = e0.elapsed_time(e1)
    k_ms = [ctx.get_timing(i) for i in range(min(K, 64))]          # per launch, launch order [K1, K1x, pack, RS, mask]
    ctx.set_timing(False)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    sampler.join(timeout=1.0)

    # ---- parity of what was just timed (outside the timed region): every chunk decoded, bytes == payload
    gathered_ok = None
    if exchange is not None:
        import ctypes
        cudart = ctypes.CDLL("libcudart.so.12")          # the copy torch already loaded

        def dev_copy(ptr, nbytes):
            """nbytes at raw device address `ptr` (a window slot / a library-owned buffer) into a fresh torch tensor"""
            t = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            torch.cuda.synchronize()
            rc = cudart.cudaMemcpy(ctypes.c_void_p(t.data_ptr()), ctypes.c_void_p(ptr), ctypes.c_size_t(nbytes), 3)   # cudaMemcpyDeviceToDevice
            assert rc == 0, "cudaMemcpy failed: %d" % rc
            return t

        last = step_no[0]
        payloads = [torch.empty_like(payload) for _ in range(world)] if rank == 0 else None
        dist.gather(payload, payloads, dst=0)
        if rank == 0:
            # what arrived on rank 0 for the last step, rank by rank, against that rank's payload
            if gather_kind in ("window", "window-direct"):
                ctx.gather_status()
            got = []
            for r in range(world):
                if gather_kind in ("window", "window-direct"):
                    pc, pm = ctx.gather_slot(last & 1, r)
                    got.append((dev_copy(pc, B * info.data_bytes).view(B, info.data_bytes), dev_copy(pm, 4 * B).view(torch.int32)))
                else:
                    got.append((exchange.recv[last & 1][0][r], exchange.recv[last & 1][1][r]))
            chunks, mask = got[0]
            if args.workload == "clean":
                full = (1 << info.chunks_per_frame) - 1
                gathered_ok = all(bool((m_ == full).all().item()) and bool(torch.equal(c_, p_)) for (c_, m_), p_ in zip(got, payloads))
        elif exchange.send is not None:
            chunks, mask = exchange.send[last & 1]
        else:   # a peer's records live in rank 0's HBM: decode once more into local buffers for this rank's own parity line
            ctx.decode_chunks_dev(frames.data_ptr(), B, chunks.data_ptr(), mask.data_ptr(), fflags.data_ptr(), flags=cc_flags)
            torch.cuda.synchronize()
    ok_mask = bool((mask == (1 << info.chunks_per_frame) - 1).all().item())
    ok_data = bool(torch.equal(chunks, payload))
    n_fallback = int((fflags & 1).sum().item())
    ok_flags = not bool(fflags.any().item())
    if ok_mask and ok_data:
        parity = "bit-exact: %d frames/rank, all %d chunks/frame == payload" % (B, info.chunks_per_frame)
        if gathered_ok is not None:
            parity += "; records of all %d ranks as gathered on rank 0 == their payloads: %s" % (world, "yes" if gathered_ok else "NO (MISMATCH)")
    elif args.workload == "clean":
        parity = "MISMATCH mask_ok=%s data_ok=%s" % (ok_mask, ok_data)
    else:
        # damaged input: RS may legitimately give up on a chunk (the reference would too; exactness against the oracle is
        # what tests/test_gpu_parity.py checks) -- report how many chunks came through and that every one of those is right
        cpf, cs = info.chunks_per_frame, info.data_bytes // info.chunks_per_frame
        bits = ((mask.view(B, 1) >> torch.arange(cpf, device=dev, dtype=torch.int32).view(1, cpf)) & 1).bool()
        same = (chunks.view(B, cpf, cs) == payload.view(B, cpf, cs)).all(dim=2)
        good = int(bits.sum().item())
        wrong = int((bits & ~same).sum().item())
        parity = "%d of %d chunks decoded, %d frames complete; decoded chunks != payload: %d" % (
            good, B * cpf, int(bits.all(dim=1).sum().item()), wrong)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, chunks.view(B, info.data_bytes), mask.view(B), fflags)

    # ---- end to end through the host-pointer C ABI: pinned host frames -> cb200_decode_fountain -> host chunks
    e2e = None
    if not args.no_e2e:
        ne = min(args.e2e_frames, B)
        host_frames = torch.empty((ne, info.image_size_y, info.image_size_x, 3), dtype=torch.uint8, pin_memory=True)
        host_frames.copy_(frames[:ne])
        torch.cuda.synchronize()
        hf = host_frames.numpy()
        ctx.set_stream(None)
        ctx.decode_fountain(hf, flags=cc_flags)      # warm-up (allocates the staging buffers)
        barrier()
        t0 = time.perf_counter()
        esteps = max(3, min(K, 10))
        for _ in range(esteps):
            ch, cnt, mk, ff = ctx.decode_fountain(hf, flags=cc_flags)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        if args.workload == "clean":
            e2e_ok = bool((cnt == info.chunks_per_frame).all()) and np.array_equal(ch.reshape(ne, -1), payload[:ne].cpu().numpy())
        else:   # damaged input: the host path must return what the device path returned for the same frames
            e2e_ok = np.array_equal(mk, mask[:ne].cpu().numpy().astype(np.uint32))
        e2e = {"value": world * ne * esteps / dt, "unit": UNIT,
               "h2d_bytes_per_step": ne * info.frame_bytes,
               "d2h_bytes_per_step": ne * (info.data_bytes + 4 + 1),
               "frames_per_step": ne, "steps": esteps, "api": "cb200_decode_fountain (host pointers, pinned input)",
               "h2d_gbytes_per_s_per_gpu": ne * info.frame_bytes * esteps / dt / 1e9,
               "bound": "the host-to-device copy of the frames (3.1 MB each) over PCIe; the decode of a step takes ~1 % of the step",
               "numa": numa,
               "parity": "ok" if e2e_ok else "MISMATCH"}

    # ---- the drop-in call shape: ONE frame per call (Decoder::decode_fountain(img, sink)), pinned and pageable host memory
    e2e_single = None
    if not args.no_e2e and rank == 0:
        ns = min(64, host_frames.shape[0])
        pageable = np.array(hf[:ns])                      # an ordinary (pageable) allocation, like a cv::Mat
        def one_by_one(arr):
            lat = []
            for i in range(ns):
                t0 = time.perf_counter()
                ctx.decode_fountain(arr[i:i + 1], flags=cc_flags)
                lat.append(time.perf_counter() - t0)
            lat.sort()
            return {"median_ms": lat[len(lat) // 2] * 1e3, "p90_ms": lat[(9 * len(lat)) // 10] * 1e3, "frames_per_s": len(lat) / sum(lat)}
        one_by_one(hf)                                    # warm-up
        e2e_single = {"api": "cb200_decode_fountain with n = 1 per call (3.1 MB H2D + band-split K1 + RS + D2H, synchronous)",
                      "calls": ns, "pinned": one_by_one(hf), "pageable": one_by_one(pageable)}
        if MV == 68 and args.workload == "clean" and args.color_correction == 0:
            # the same call on a frame that needs the exact flood walk (one noise tile, as a camera frame would have many): the walk
            # is ONE warp per frame -- its throughput comes from thousands of frames in flight, a lone frame pays its whole latency
            nw = 8
            walk = np.array(hf[:nw])
            walk[:, 8:16, 512:520, :] = np.random.default_rng(5).integers(0, 256, (nw, 8, 8, 3), dtype=np.uint8)     # cell 50 of the top row
            lat, used = [], 0
            for i in range(nw + 1):
                t0 = time.perf_counter()
                _, _, _, ffw = ctx.decode_fountain(walk[i % nw:i % nw + 1])
                if i:
                    lat.append(time.perf_counter() - t0)
                    used += int(ffw[0]) & 1
            lat.sort()
            e2e_single["exact_walk_frame"] = {"median_ms": lat[len(lat) // 2] * 1e3, "calls": len(lat), "frames_through_the_walk": used,
                                              "note": "latency of one frame through K1x; batches: see --workload noise1pct"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    k1_ms = sum(r[0] for r in k_ms) / len(k_ms)
    stage_ms = [sum(r[i] for r in k_ms) / len(k_ms) for i in range(len(k_ms[0]))]
    peak, peak_src = measured_peak_gbs()
    achieved = B * K1_ALGO_BYTES / (k1_ms * 1e-3) / 1e9
    traffic = k1_traffic_bytes()
    out = {
        "metric": metric_name(MV), "value": world * B * K / (elapsed_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(W, 3),
        "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (integer/bitwise; float32 only in the colour classifier, bit-exact vs reference)",
        "data": "synthetic (device-generated: random payload -> RS(155,125) -> interleaved tiles -> RGB8 frames)",
        "config": {"workload": ({"clean": "BASELINE configs[1]", "errors1pct": "BASELINE configs[2] (1% wrong tiles)", "noise1pct": "1% noise tiles (exact-walk path)"}[args.workload]) +
                   (" with should_preprocess=true (sharpen + block-7 threshold inside K1)" if args.sharpen else "") +
                   ": %d synthetic %dx%d mode-%s frames per GPU per step through the full decode "
                   "(K1 fused threshold+ahash+colour, K1x exact-walk check, RS(%d,%d) with fused de-interleave, chunk masks)" % (
                       B, info.image_size_x, info.image_size_y, MODE_NAMES[MV], info.ecc_block_size, info.ecc_block_size - info.ecc_bytes),
                   "mode": "%s (%d)" % (MODE_NAMES[MV], MV), "frames_per_gpu_per_step": B, "color_correction": args.color_correction, "sharpen": bool(args.sharpen),
                   "l2": "input %.1f GB per step >> 126 MB L2 (no flush needed)" % (B * info.frame_bytes / 1e9),
                   "parallelism": "frames sharded one-per-GPU (dp%d); chunk records to rank 0 by %s" % (world, {
                       None: "nothing (one GPU)", "window": "copy-engine pushes into a window in rank 0's HBM (CUDA IPC peer mapping over NVLink, device-side epochs, side stream: overlaps the next decode)",
                       "window-direct": "direct NVLink stores of the RS kernels into rank 0's HBM (CUDA IPC window, device-side epochs)",
                       "nccl": "ncclSend/ncclRecv on a side stream (cb200_gather_chunks), double buffered",
                       "torch": "torch.distributed.gather on the decode stream"}[gather_kind])},
        "parity": parity + ("" if ok_flags else " (%d of %d frames/rank went through the exact flood-walk kernel)" % (n_fallback, B)),
        # kernels of this library launched inside the timed region, all ranks (counted at the launch sites, cb200_launch_count)
        "gpu_launches": launches,
        "kernel_ms_per_step": {"k1_decode": stage_ms[0], "k1x_flood_check": stage_ms[1], "pack": stage_ms[2], "rs": stage_ms[3], "chunk_mask": stage_ms[4]},
        "roofline": {"kernel": "k1_decode_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": B * K1_ALGO_BYTES,
                     "traffic": (traffic["dram_bytes_per_frame"] * B if traffic else None),
                     "traffic_source": (traffic["source"] if traffic else None),
                     "note": "K1 is bound by instruction issue and dependency latency, not by HBM: the same TMA pipeline with the decode "
                             "switched off (CB200_K1_L2_AHEAD=4096, tools/k1_sweep.py) copies at 7.4-7.5 TB/s on this GPU "
                             "(profiles/r02_results.md)"},
        "clocks": sampler.summary(),
    }
    if e2e:
        out["e2e"] = e2e
    if e2e_single:
        out["e2e_single_frame"] = e2e_single
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_from_device_frames(frames, info, MV, stage_ms[3] / B)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def usable_cores():
    """threads the CPU arms may use: the affinity mask, clamped by the cgroup CPU quota when there is one"""
    cores = len(os.sched_getaffinity(0))
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cores = max(1, min(cores, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        pass
    return cores


def best_thread_count(ora, host, cores, mode_val=68):
    """the CPU arm gets the thread count it runs fastest with on this box (oversubscribed or throttled hosts
    run slower with one thread per logical core), probed on a small sample"""
    probe = host[:min(host.shape[0], max(64, 2 * cores))]
    best, best_fps = cores, 0.0
    for t in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
        ora.bench_decode(mode_val, probe[:t], t, 1)
        secs, _ = ora.bench_decode(mode_val, probe, t, 1)
        fps = probe.shape[0] / secs
        if fps > best_fps * 1.03:
            best, best_fps = t, fps
    return best


def host_description():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"cpu_model": model, "logical_cpus": os.cpu_count(), "usable_cores": usable_cores()}


def cpu_stage_split(ora, mode_val, host):
    """single-thread per-stage split of the CPU restatement (BASELINE.md section 3): ms per frame"""
    import ctypes as C
    import numpy as np
    L = ora.lib
    L.cbo_stage_timing.argtypes = [C.c_int]
    L.cbo_stage_times.argtypes = [C.POINTER(C.c_double)]
    m = ora.mode(mode_val)
    n = min(host.shape[0], 24)
    ora.decode(m, host[0])
    L.cbo_stage_timing(1)
    t0 = time.perf_counter()
    for f in range(n):
        ora.decode(m, host[f])
    total = time.perf_counter() - t0
    st = (C.c_double * 4)()
    L.cbo_stage_times(st)
    L.cbo_stage_timing(0)
    out = {"frames": n, "threads": 1, "total_ms_per_frame": total / n * 1e3,
           "preprocess_ms": st[0] / n * 1e3, "symbol_walk_ms": st[1] / n * 1e3, "colour_ms": st[2] / n * 1e3,
           "rs_ms": st[3] / n * 1e3, "wirehair_ms": None}
    try:   # what OpenCV itself (the library the reference calls for this stage) needs on this host, one thread
        import cv2
        cv2.setNumThreads(1)
        def pre(img):
            return cv2.adaptiveThreshold(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY), 255, cv2.ADAPTIVE_THRESH_MEAN_C, cv2.THRESH_BINARY, 5, 0)
        pre(host[0])
        t0 = time.perf_counter()
        for f in range(n):
            pre(host[f])
        out["opencv_cvtColor_adaptiveThreshold_ms"] = (time.perf_counter() - t0) / n * 1e3
    except Exception:
        out["opencv_cvtColor_adaptiveThreshold_ms"] = None
    return out


def rs_standalone(ora, mode_val, host, k2_ms_per_frame):
    """the reference's own libcorrect (oracle/_ref, compiled unmodified) on exactly the RS blocks K2 gets, next to K2"""
    import ctypes as C
    import numpy as np
    try:
        from oracle_lib import Ref, _ptr
        ref = Ref()
    except Exception as e:
        return {"unavailable": str(e)[:80]}
    m = ora.mode(mode_val)
    n = min(host.shape[0], 16)
    raws = [ora.decode_raw(m, host[f]) for f in range(n)]
    cap_sym = ora.capacity(m, m.symbol_bits) if not m.legacy_mode else ora.capacity(m)
    out = np.zeros(16384, np.uint8)
    def run():
        for r in raws:
            ref.lib.ref_rs_stream(m.ecc_bytes, m.ecc_block_size, _ptr(r[:cap_sym]), cap_sym, _ptr(out))
            if r.size > cap_sym:
                tail = np.ascontiguousarray(r[cap_sym:])
                ref.lib.ref_rs_stream(m.ecc_bytes, m.ecc_block_size, _ptr(tail), tail.size, _ptr(out))
    run()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        run()
    cpu_ms = (time.perf_counter() - t0) / (reps * n) * 1e3
    return {"libcorrect_reference_ms_per_frame_1thread": cpu_ms, "k2_ms_per_frame": k2_ms_per_frame,
            "frames": n, "what": "reed_solomon_stream over the frame's symbol + colour streams (oracle/_ref = libcorrect compiled unmodified)"}


def cpu_baseline_from_device_frames(frames, info, mode_val=68, k2_ms_per_frame=None):
    """the oracle (CPU port of the reference decode) timed on the host cores on a bounded sample of the same frames"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    ora = Oracle()
    cores = usable_cores()
    S = int(min(frames.shape[0], max(64, 16 * cores)))
    host = frames[:S].cpu().numpy()
    cores = best_thread_count(ora, host, cores, mode_val)
    ora.bench_decode(mode_val, host[:cores], cores, 1)      # warm the per-thread malloc arenas
    secs, _ = ora.bench_decode(mode_val, host, cores, 1)
    n1 = max(8, S // cores)
    secs1, _ = ora.bench_decode(mode_val, host[:n1], 1, 1)
    return {"value": S / secs, "unit": UNIT, "cores": cores, "kind": "port",
            "single_thread_value": n1 / secs1,
            "sample": "%d of the same synthetic frames, full decode incl. RS, %d threads (one decoder per thread); "
                      "single thread: %.1f frames/s" % (S, cores, n1 / secs1),
            "build": "gcc -O3 -march=x86-64-v3 (AVX2), fused SIMD-friendly gray/box-threshold (oracle/Makefile)",
            "host": host_description(),
            "stages": cpu_stage_split(ora, mode_val, host),
            "rs_standalone": rs_standalone(ora, mode_val, host, k2_ms_per_frame)}


# ------------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    ora = Oracle()
    MV = args.mode
    m = ora.mode(MV)
    cores = usable_cores()
    S = args.ref_sample or int(max(64, 8 * cores))
    rng = np.random.default_rng(0xC1B4)
    base = min(S, 64)
    nbytes = (ora.capacity(m) // m.ecc_block_size) * (m.ecc_block_size - m.ecc_bytes)
    uniq = np.stack([ora.render_frame(m, ora.payload_to_cells(m, rng.integers(0, 256, nbytes, dtype=np.uint8))) for _ in range(base)])
    frames = np.concatenate([uniq] * ((S + base - 1) // base))[:S]
    K, W = args.steps, max(args.warmup, 1)
    cores = best_thread_count(ora, frames, cores, MV)
    for _ in range(W):
        ora.bench_decode(MV, frames, cores, 1)
    t0 = time.perf_counter()
    for _ in range(K):
        ora.bench_decode(MV, frames, cores, 1)
    dt = time.perf_counter() - t0
    value = S * K / dt
    out = {
        "impl": "reference", "metric": metric_name(MV), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic (same generator family: random payload -> RS -> tiles -> RGB8 frames)",
        "config": {"workload": "BASELINE configs[1]: synthetic %dx%d mode-%s frames through the full CPU decode "
                               "(threshold, flood walk, colour, RS) -- bounded sample of %d frames per step" % (
                                   m.image_size_x, m.image_size_y, MODE_NAMES[MV], S),
                   "mode": "%s (%d)" % (MODE_NAMES[MV], MV), "frames_per_step": S},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d frames per step, %d threads, one decoder per thread (the reference's own threading model); "
                                   "the reference's ./cimbar cannot be built here (needs C++ OpenCV), this is its CPU restatement "
                                   "pinned to its SHA-256 goldens" % (S, cores),
                         "build": "gcc -O3 -march=x86-64-v3 (AVX2), fused SIMD-friendly gray/box-threshold (oracle/Makefile)",
                         "host": host_description(),
                         "stages": cpu_stage_split(ora, MV, frames)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.camera:
        from libcimbar_b200 import camera_bench
        camera_bench.run(args, ClockSampler, measured_peak_gbs)
    elif args.fountain:
        from libcimbar_b200 import fountain_bench
        fountain_bench.run(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
