#!/usr/bin/env python
"""bench.py — attribute-transform throughput of the B200-native RAHT path.

    python bench.py --gpus N --steps K --warmup W            (our arm)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): one ~1M-point synthetic LiDAR ring cloud
(Ford_01-shaped, 64 lasers, seed 2 + rank), RGB + reflectance, octree-raht
lossy-attrs CTC settings (qp 34, chroma offset -2, prediction + sub-node
prediction on, search range 2500).  One step = the attribute coder's RAHT hot
path over one frame: for colour (A=3) and for reflectance (A=1), Morton key +
sort, gather, forward transform (RDOQ + quantisation + reconstruction), clip
and write back.  A step processes --frames (default 160) independent frames of
that shape per GPU in ONE batch call (pccb200_attr_raht_encode_multi_batch: the
library codes them in gangs, many dependency chains in flight; intra-coded frames,
slices and attributes are independent work units in the reference,
tmc3/encoder.cpp:545-568,1052); frames shard across GPUs (weak scaling, no
data-path collective; NCCL only broadcasts the parameter PODs).

Prints ONE JSON line (rank 0).  `value` = points/s with inputs resident in
HBM (CUDA events on the library's stream); `e2e` = the same through the
host-pointer C ABI with pinned host buffers (H2D + D2H inside the timed
region).  The oracle / compiled reference is only used for the reported
`cpu_baseline` and for `--impl reference`."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

# one hardware work queue per lane: with the default of 8, more than 8 streams
# alias and a long dataflow kernel of one call blocks the short kernels of
# another (must be set before the CUDA context exists)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# stdout carries the single JSON line and nothing else: libraries that write to
# file descriptor 1 (NCCL prints its version banner there) are sent to stderr
# once main() has claimed it; emit_json() writes to the saved descriptor
_JSON_FD = 1


def claim_stdout():
    global _JSON_FD
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit_json(line):
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "mpeg-pcc-tmc13_b200"))

N_POINTS = 1_000_000
QP = 34
CHROMA_OFFSET = -2
SEARCH_RANGE = 2500
METRIC = "attribute-transform Mpoints/s (RAHT forward: Morton sort + transform, RGB + reflectance)"
ALG_BYTES_PER_POINT = (16 + 12 * 3) + (16 + 12 * 1)  # SURVEY.md 8(d): 52 (RGB) + 28 (reflectance)


FRAMES_PER_STEP = 160  # frames in flight per GPU: one batch call, coded in gangs (DESIGN.md 6)
DISTINCT_FRAMES = 16   # distinct synthetic frames (geometry + attributes) the step cycles through


def workload_config(frames=FRAMES_PER_STEP):
    """identical for both arms (the driver compares the dicts)"""
    return {
        "workload": "configs[1]: octree-raht lossy-attrs, ~1M-point synthetic LiDAR ring cloud "
                    "(Ford_01-shaped), RGB + reflectance, single slice",
        "points_per_frame": N_POINTS,
        "attributes": "RGB (A=3) + reflectance (A=1), 8-bit",
        "attribute_model": f"smooth field + per-point texture of +-{TEXTURE_RGB} (RGB) / "
                           f"+-{TEXTURE_REFL} (reflectance): about a quarter of the RGB and a "
                           f"sixth of the reflectance coefficient positions quantise to 1 or 2 "
                           f"at qp {QP} (the zero-run / RDOQ chain is exercised on every block)",
        "qp": QP,
        "raht": "prediction + sub-node prediction, rahtExtension, RDOQ, search range 2500",
        "frames_per_step_per_gpu": frames,
        "distinct_frames": min(frames, DISTINCT_FRAMES),
        "parallelism": "frames shard across GPUs, no data-path collective",
        "l2": "512 MiB written between steps (excluded from timing) to flush L2",
    }


TEXTURE_RGB = 16    # +- amplitude of the per-point texture of the headline frame
TEXTURE_REFL = 24


def make_frame(seed, textured=True):
    """One frame of configs[1].  textured=False is round 1's smooth attribute
    field (0.1 % of the coefficients non-zero at qp 34); textured=True adds
    per-point texture so that the quantiser and the RDOQ zero-run chain are
    exercised like on real content (SURVEY section 6: 12-27 % of the positions
    quantise to 1 or 2)."""
    from pcc_attr_b200.synth import cloud_lidar, texture

    xyz, rgb = cloud_lidar(N_POINTS, seed=seed, a=3)
    rng = np.random.default_rng(seed + 1000)
    # reflectance: range-dependent intensity + noise
    r = np.linalg.norm(xyz.astype(np.float64), axis=1)
    refl = np.clip(200.0 * np.exp(-r / (r.max() + 1)) + rng.integers(-6, 7, size=r.shape), 0, 255)
    rgb = rgb.astype(np.int32)
    refl = np.rint(refl).astype(np.int32)[:, None]
    if textured:
        rgb = texture(rgb, TEXTURE_RGB, seed + 2000)
        refl = texture(refl, TEXTURE_REFL, seed + 3000)
    return xyz, rgb, refl


def make_pods(pb):
    p = pb.default_params()
    p.prediction_search_range = SEARCH_RANGE
    q = pb.QpSet()
    q.num_layers = 1
    q.layers[0][0] = QP
    q.layers[0][1] = CHROMA_OFFSET
    q.max_qp = 51
    q.fixed_point_qp_offset = 0
    q.num_ac_coeff_qp_layers = 0
    return p, q


# ---------------------------------------------------------------------------
# clocks sampling (nvidia-smi) during the timed region

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "1000"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                clk, mxv, util = float(f[0]), float(f[1]), float(f[6])
            except ValueError:
                continue
            mx = mxv
            if util > 0:
                sm.append(clk)
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            sm = [float(x.split(",")[0]) for x in self.lines if x and x.split(",")[0].strip().replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(self.lines)}


# ---------------------------------------------------------------------------
# reference / oracle on the host cores

def load_cpu_impl():
    """(callable, kind): the compiled unmodified reference if it travelled with
    the snapshot (oracle/_ref), else the oracle port."""
    ref = os.path.join(ROOT, "oracle", "_ref", "libtmc13_ref.so")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import pcc_testlib as tl

    if os.path.exists(ref):
        lib = C.CDLL(ref)
        lib.tmc13ref_attr_raht.restype = C.c_double

        def run(params, qpset, xyz, attrs):
            a = attrs.copy()
            coef = np.zeros((a.shape[1], a.shape[0]), dtype=np.int32)
            lib.tmc13ref_attr_raht(
                C.c_int(1), C.byref(params), C.byref(qpset), None,
                xyz.ctypes.data_as(C.POINTER(C.c_int32)), a.ctypes.data_as(C.POINTER(C.c_int32)),
                C.c_int(a.shape[1]), C.c_int(a.shape[0]), C.c_int(8),
                coef.ctypes.data_as(C.POINTER(C.c_int32)))
            return a, coef

        return run, "reference"

    def run(params, qpset, xyz, attrs):
        mort, a_s, order = tl.sort_cloud(xyz, attrs)
        rec, coef = tl.oracle_raht(1, params, qpset, mort, a_s)
        out = np.empty_like(rec)
        out[order] = np.clip(rec, 0, 255)
        return out, coef

    return run, "port"


def cpu_frame_seconds(run, params, qpset, frame):
    xyz, rgb, refl = frame
    t0 = time.perf_counter()
    run(params, qpset, xyz, rgb)
    run(params, qpset, xyz, refl)
    return time.perf_counter() - t0


def physical_cores():
    """number of physical cores of the host (hyper-threads counted once)"""
    try:
        seen, phys, core = set(), None, None
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("physical id"):
                phys = ln.split(":")[1].strip()
            elif ln.startswith("core id"):
                core = ln.split(":")[1].strip()
            elif not ln.strip():
                if phys is not None and core is not None:
                    seen.add((phys, core))
                phys = core = None
        if seen:
            return len(seen)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def bind_to_gpu_numa_node(torch, local):
    """Bind this rank's threads to the CPUs of its GPU's NUMA node (the launch
    and staging threads of 8 ranks otherwise wander over both sockets)."""
    try:
        pr = torch.cuda.get_device_properties(local)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (
            pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def host_cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def coefficient_histogram(coefs):
    """zero / soft (sum |q| in {1,2}) / hard positions of a list of [A, N] planes"""
    out = {}
    for name, c in coefs:
        sm = np.abs(c.astype(np.int64)).sum(axis=0)
        n = float(sm.size)
        out[name] = {"zero": float((sm == 0).sum() / n), "soft": float(((sm > 0) & (sm < 3)).sum() / n),
                     "hard": float((sm >= 3).sum() / n)}
    return out


def run_reference_arm(args):
    """The reference's own CPU implementation of the path (oracle/_ref: the
    unmodified sources compiled here; else the oracle port) on the host's
    physical cores: each step = one frame of the workload per thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import pcc_testlib as tl

    run, kind = load_cpu_impl()
    params = tl.make_params(search_range=SEARCH_RANGE)
    qpset = tl.make_qpset(qp=QP, chroma_offset=CHROMA_OFFSET)
    cores = physical_cores()
    if kind == "port":
        cores = 1  # the oracle port is driven through numpy here: one thread
    frames = [make_frame(sd) for sd in frame_seeds(0, min(4, cores))]

    def one_step():
        ts = [threading.Thread(target=cpu_frame_seconds, args=(run, params, qpset, frames[i % len(frames)]))
              for i in range(cores)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    one_core = cpu_frame_seconds(run, params, qpset, frames[0])
    for _ in range(args.warmup):
        one_step()
    total = 0.0
    for _ in range(args.steps):
        total += one_step()
    n = frames[0][0].shape[0]
    value = cores * n * args.steps / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mpoints/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(args.frames),
        "cpu_baseline": {
            "value": value, "unit": "Mpoints/s", "cores": cores, "kind": kind,
            "value_one_core": n / one_core / 1e6,
            "sample": f"each step: one frame of the workload ({n} points, RGB + reflectance) per "
                      f"host thread, {cores} threads = the physical cores ({len(frames)} distinct "
                      f"frames; the reference itself is single-threaded); host: {host_cpu_model()}"},
        "e2e": {"value": value, "unit": "Mpoints/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    emit_json(line)


# ---------------------------------------------------------------------------
# sharding helpers (also exercised on CPU with the gloo backend, tests/test_multiprocess.py)

def frame_seeds(rank, frames):
    """Distinct synthetic frames per rank: the path shards over frames with no
    exchange (SURVEY.md 8e)."""
    return [2 + rank * 100 + f for f in range(frames)]


def broadcast_pods(blob, dist, device):
    """Rank 0 owns the flattened parameter PODs; everyone else receives the
    bytes (the only collective of the path)."""
    import torch

    t = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(device)
    dist.broadcast(t, src=0)
    return bytes(t.cpu().numpy().tobytes())


def reduce_timing(values, dist, device):
    """max over ranks of per-rank elapsed times"""
    import torch

    t = torch.tensor(values, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


DUMP_BYTES = 60_000_000  # what --dump-outputs writes in all (npy headers aside)


def dump_outputs(out_dir, torch, dv, n):
    """The outputs of the last timed step, for comparing two builds: for every
    frame, the reconstructed colour and reflectance at a fixed, seeded sample of
    points and the colour and reflectance coefficients at the same positions of
    the coefficient planes (coding order), as float32 (attributes) and float64
    (coefficients).  The sample is sized to keep the files under DUMP_BYTES."""
    k = min(n, DUMP_BYTES // (len(dv) * (4 * 4 + 4 * 8)))
    idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    ti = torch.from_numpy(idx).to(dv[0]["rgb"].device)
    planes = {"rgb": (lambda d: d["rgb"][ti], np.float32),
              "reflectance": (lambda d: d["refl"][ti], np.float32),
              "coef_rgb": (lambda d: d["crgb"][:, ti], np.float64),
              "coef_reflectance": (lambda d: d["crefl"][:, ti], np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, (take, dtype) in planes.items():
        a = torch.stack([take(d) for d in dv]).cpu().numpy().astype(dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------
# our arm

def run_ours(args):
    import torch
    import torch.distributed as dist
    from concurrent.futures import ThreadPoolExecutor

    import pcc_attr_b200 as pb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_to_gpu_numa_node(torch, local)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pb.lib()
    pb.set_device(local)

    # parameter PODs: rank 0 owns them, NCCL broadcasts the bytes
    params, qpset = make_pods(pb)
    if distributed:
        if rank != 0:  # only rank 0's values count
            params, qpset = pb.RahtParams(), pb.QpSet()
        raw = broadcast_pods(bytes(params) + bytes(qpset), dist, dev)
        params = pb.RahtParams.from_buffer_copy(raw[:C.sizeof(pb.RahtParams)])
        qpset = pb.QpSet.from_buffer_copy(raw[C.sizeof(pb.RahtParams):])
    qpsets = [qpset, qpset]

    F = args.frames
    D = min(F, DISTINCT_FRAMES)
    pool = ThreadPoolExecutor(max_workers=8)
    frames = list(pool.map(make_frame, frame_seeds(rank, D)))
    n = frames[0][0].shape[0]

    # ---- device-resident inputs: F units cycling through the D distinct frames
    def to_dev(fr):
        src = [(torch.from_numpy(xyz).to(dev), torch.from_numpy(rgb).to(dev),
                torch.from_numpy(refl).to(dev)) for xyz, rgb, refl in fr]
        out = []
        for u in range(F):
            x, r, l = src[u % len(src)]
            out.append({"xyz": x, "rgb0": r, "refl0": l, "rgb": torch.empty_like(r),
                        "refl": torch.empty_like(l),
                        "crgb": torch.empty((3, n), dtype=torch.int32, device=dev),
                        "crefl": torch.empty((1, n), dtype=torch.int32, device=dev)})
        return out

    dv = to_dev(frames)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def dev_jobs(subset):
        # ONE call for all frames of the step: colour and reflectance of a frame in
        # one pass, the frames in gangs
        return [lambda: pb.attr_raht_multi_batch_dev(
            True, params, qpsets, [d["xyz"].data_ptr() for d in subset],
            [[d["rgb"].data_ptr(), d["refl"].data_ptr()] for d in subset],
            [[d["crgb"].data_ptr(), d["crefl"].data_ptr()] for d in subset],
            [n] * len(subset), [3, 1])]

    def run_jobs(jobs):
        for f in [pool.submit(j) for j in jobs]:
            f.result()

    def prepare(subset):
        flush.fill_(1)
        for d in subset:
            d["rgb"].copy_(d["rgb0"])
            d["refl"].copy_(d["refl0"])
        torch.cuda.synchronize()

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_device_step(subset):
        prepare(subset)
        pb.time_begin()
        run_jobs(dev_jobs(subset))
        return pb.time_end()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        timed_device_step(dv)

    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = pb.kernel_launch_count()
    step_ms = [timed_device_step(dv) for _ in range(args.steps)]
    total_ms = float(sum(step_ms))
    launches = pb.kernel_launch_count() - launches0
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, dv, n)

    # latency of one frame alone
    single_ms = min(timed_device_step(dv[:1]) for _ in range(3))

    # the dominant kernel timed alone: one call at a time, CUDA events around
    # every launch
    pb.profile_reset()
    pb.profile_enable(True)
    prof_steps = 2
    for _ in range(prof_steps):
        prepare(dv[:1])
        for j in dev_jobs(dv[:1]):
            j()
    pb.profile_enable(False)
    prof = pb.profile_read()
    # ... and inside a whole step (all gangs in flight): CUDA events around every launch
    pb.profile_reset()
    pb.profile_enable(True)
    prepare(dv)
    for j in dev_jobs(dv):
        j()
    pb.profile_enable(False)
    prof_step = pb.profile_read()
    gpu_frame0 = {k: dv[0][k].cpu().numpy() for k in ("rgb", "refl", "crgb", "crefl")}

    # the decoder on the same frame (extra key): coefficients in, attributes out
    dec = None
    if rank == 0:
        try:
            d0 = dv[0]
            drgb, drefl = torch.empty_like(d0["rgb"]), torch.empty_like(d0["refl"])
            k = len(qpsets)

            def dec_call():
                QP_ = C.POINTER(pb.QpSet) * k
                VP = C.c_void_p * k
                pb._check(pb.lib().pccb200_attr_raht_decode_multi_dev(
                    C.byref(params), C.c_int32(k), QP_(*[C.pointer(q) for q in qpsets]),
                    C.c_void_p(d0["xyz"].data_ptr()), VP(drgb.data_ptr(), drefl.data_ptr()),
                    (C.c_int32 * k)(3, 1), (C.c_int32 * k)(8, 8), C.c_int32(n),
                    VP(d0["crgb"].data_ptr(), d0["crefl"].data_ptr())))

            dec_call()
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                pb.time_begin()
                dec_call()
                ts.append(pb.time_end())
            ok = bool(torch.equal(drgb, d0["rgb"]) and torch.equal(drefl, d0["refl"]))
            dec = {"single_frame_ms": min(ts), "mpoints_per_s": n / min(ts) / 1e3,
                   "reproduces_encoder_reconstruction": ok}
            # all frames of the step through the batch entry (gangs, wavefront order)
            outs = [(torch.empty_like(d["rgb"]), torch.empty_like(d["refl"])) for d in dv]

            def dec_batch():
                pb.attr_raht_multi_batch_dev(
                    False, params, qpsets, [d["xyz"].data_ptr() for d in dv],
                    [[o[0].data_ptr(), o[1].data_ptr()] for o in outs],
                    [[d["crgb"].data_ptr(), d["crefl"].data_ptr()] for d in dv], [n] * F, [3, 1])

            dec_batch()
            torch.cuda.synchronize()
            tb = []
            for _ in range(2):
                flush.fill_(1)
                torch.cuda.synchronize()
                pb.time_begin()
                dec_batch()
                tb.append(pb.time_end())
            okb = bool(all(torch.equal(o[0], d["rgb"]) and torch.equal(o[1], d["refl"])
                           for o, d in zip(outs, dv)))
            dec["batch"] = {"frames": F, "ms_per_step": min(tb), "mpoints_per_s": F * n / min(tb) / 1e3,
                            "reproduces_encoder_reconstruction": okb}
            del outs
        except Exception as e:
            dec = {"error": str(e)[:200]}

    # the smooth attribute field of round 1 (zero runs thousands of coefficients
    # long, RDOQ nearly idle), same geometry: extra key, not the headline
    smooth = None
    if rank == 0 and not args.no_smooth:
        sframes = list(pool.map(lambda sd: make_frame(sd, textured=False), frame_seeds(rank, min(D, 8))))
        sdv = to_dev(sframes)
        for _ in range(2):
            timed_device_step(sdv)
        sm = [timed_device_step(sdv) for _ in range(max(3, args.steps // 2))]
        s1 = min(timed_device_step(sdv[:1]) for _ in range(3))
        smooth = {"value": F * n / (sum(sm) / len(sm)) / 1e3, "unit": "Mpoints/s (this GPU)",
                  "ms_per_step": sum(sm) / len(sm), "single_frame_ms": s1,
                  "attribute_model": "smooth field + noise of +-8 (round 1's frame): 0.1 % of the "
                                     "coefficient positions non-zero at qp 34"}
        del sdv, sframes

    # ---- end to end: host-pointer C ABI, pinned host buffers ---------------
    hsrc = [(torch.from_numpy(xyz).pin_memory(), torch.from_numpy(rgb).pin_memory(),
             torch.from_numpy(refl).pin_memory()) for xyz, rgb, refl in frames]
    hv = []
    for u in range(F):
        x, r, l = hsrc[u % D]
        hv.append({"xyz": x, "rgb0": r, "refl0": l,
                   "rgb": torch.empty(r.shape, dtype=r.dtype, pin_memory=True),
                   "refl": torch.empty(l.shape, dtype=l.dtype, pin_memory=True),
                   "crgb": torch.empty((3, n), dtype=torch.int32, pin_memory=True),
                   "crefl": torch.empty((1, n), dtype=torch.int32, pin_memory=True)})

    def host_jobs():
        return [lambda: pb.attr_raht_encode_multi_batch_into(
            params, qpsets, [h["xyz"] for h in hv], [[h["rgb"], h["refl"]] for h in hv],
            [[h["crgb"], h["crefl"]] for h in hv])]

    def host_prepare():
        flush.fill_(1)
        for h in hv:
            h["rgb"].copy_(h["rgb0"])
            h["refl"].copy_(h["refl0"])
        torch.cuda.synchronize()

    for _ in range(2):
        host_prepare()
        run_jobs(host_jobs())
    barrier()
    e2e_s = 0.0
    checksum = 0
    for _ in range(args.steps):
        host_prepare()
        t0 = time.perf_counter()
        run_jobs(host_jobs())
        checksum = int(hv[0]["crgb"].numpy()[0, :1024].astype(np.int64).sum())  # result read on the host
        e2e_s += time.perf_counter() - t0
    barrier()
    xyz, rgb, refl = frames[0]
    h2d = F * (xyz.nbytes + rgb.nbytes + refl.nbytes)
    d2h = F * 2 * (rgb.nbytes + refl.nbytes)
    e2e_equal_dev = bool(np.array_equal(hv[0]["crgb"].numpy(), gpu_frame0["crgb"])
                         and np.array_equal(hv[0]["crefl"].numpy(), gpu_frame0["crefl"]))

    extras = run_extras(args, pb, rank, world, params, qpset, frames[0], run_jobs)

    per_rank = [total_ms / args.steps]
    if distributed:
        g = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([total_ms, e2e_s], dtype=torch.float64, device=dev))
        per_rank = [float(x[0]) / args.steps for x in g]
        total_ms, e2e_s = max(float(x[0]) for x in g), max(float(x[1]) for x in g)
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        blk_ms, blk_launches = prof["block_transform"]
        blk_ms_per_frame = blk_ms / prof_steps
        # the dominant kernel inside a step: every launch carries one descent step of
        # the frames of a gang; per launch: algorithmic bytes / duration, averaged
        sblk_ms, sblk_launches = prof_step["block_transform"]
        achieved = ALG_BYTES_PER_POINT * n * F / (sblk_ms * 1e-3) / 1e9
        step_wall_ms = total_ms / args.steps  # (max over ranks; every rank codes F frames)
        aggregate = ALG_BYTES_PER_POINT * n * F / (step_wall_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("block_transform_dram_bytes_per_frame")
        line = {
            "metric": METRIC,
            "value": world * F * n * args.steps / (total_ms * 1e-3) / 1e6,
            "unit": "Mpoints/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": workload_config(F),
            "e2e": {"value": world * F * n * args.steps / e2e_s / 1e6, "unit": "Mpoints/s",
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * e2e_s / args.steps, "result_checksum": checksum,
                    "equals_device_resident_result": e2e_equal_dev},
            "concurrency": f"{F} frames per GPU in one batch call (colour and reflectance of a frame "
                           f"in one pass; frames coded in gangs: the top-down passes of a gang share "
                           f"their kernel launches)",
            "per_rank_ms_per_step": {"min": min(per_rank), "median": float(np.median(per_rank)),
                                     "max": max(per_rank), "all": per_rank},
            "numa_bound_cpus": numa_cpus,
            "single_frame": {"ms": single_ms, "mpoints_per_s": n / single_ms / 1e3,
                             "note": "one frame alone (RGB + reflectance in one pass)"},
            "decoder": dec,
            "smooth_frame": smooth,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {
                "bound": "hbm",
                "kernel": "k_block_warp_gang (top-down block transform; one launch = one descent "
                          "step of the frames of a gang, RGB + reflectance in one pass)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_frame": ALG_BYTES_PER_POINT * n,
                "launches_per_step": sblk_launches,
                "algorithmic_bytes_per_launch": ALG_BYTES_PER_POINT * n * F / max(1, sblk_launches),
                "avg_launch_ms": sblk_ms / max(1, sblk_launches),
                "launches_in_flight": "one per gang; the gangs of a step run side by side, so the "
                                      "per-launch figure is that of a kernel sharing the machine",
                "step_aggregate": {"achieved": aggregate, "frac": aggregate / peak,
                                   "note": "algorithmic bytes of all frames of a step / the step's "
                                           "device time (sort, tree build and tail included)"},
                "kernel_ms_per_frame_alone": blk_ms_per_frame,
                "kernel_launches_per_frame_alone": blk_launches / prof_steps,
                "note": "serial dependency chain per frame (RDOQ zero-run state in coding order + "
                        "sub-node prediction), latency bound; throughput comes from the number of "
                        "chains in flight; see DESIGN.md 5"},
            "phase_ms_per_frame_alone": {k: v[0] / prof_steps for k, v in prof.items()},
        }
        line.update(extras)
        # reported CPU baseline + parity: single N=1 run only (bounded: one frame)
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import pcc_testlib as tl

            run, kind = load_cpu_impl()
            cp, cq = tl.make_params(search_range=SEARCH_RANGE), tl.make_qpset(qp=QP, chroma_offset=CHROMA_OFFSET)
            t0 = time.perf_counter()
            c_rgb_rec, c_rgb = run(cp, cq, frames[0][0], frames[0][1])
            c_refl_rec, c_refl = run(cp, cq, frames[0][0], frames[0][2])
            secs = time.perf_counter() - t0
            line["cpu_baseline"] = {
                "value": n / secs / 1e6, "unit": "Mpoints/s", "cores": 1, "kind": kind,
                "sample": f"1 frame of the same workload ({n} points, RGB + reflectance), "
                          f"{secs:.2f} s on one host core; host: {host_cpu_model()}"}
            # the same frame: the GPU's coefficients and reconstruction against the CPU's
            parity = bool(np.array_equal(gpu_frame0["crgb"], c_rgb)
                          and np.array_equal(gpu_frame0["crefl"], c_refl)
                          and np.array_equal(gpu_frame0["rgb"], c_rgb_rec)
                          and np.array_equal(gpu_frame0["refl"], c_refl_rec))
            line["parity_checked"] = parity
            line["parity_note"] = ("frame 0: coefficients and reconstruction of the GPU path "
                                   f"bit-identical to the CPU {kind} (4 M coefficients + 4 M values)")
            line["coefficients"] = coefficient_histogram([("rgb", c_rgb), ("reflectance", c_refl)])
            if not parity:
                line["parity_note"] = "MISMATCH between the GPU path and the CPU " + kind
                emit_json(line)
                raise SystemExit("bench.py: GPU result differs from the CPU reference")
        emit_json(line)
    pool.shutdown()
    if distributed:
        dist.destroy_process_group()


def run_extras(args, pb, rank, world, params, qpset, frame, run_jobs):
    """Extra keys of the N=1 line (never the headline): the lifting path and the
    rows either side of the transform."""
    out = {}
    if rank != 0 or args.no_lifting:
        return out
    xyz, rgb, refl = frame
    # ---- the lifting path (SURVEY.md 8d config 4 shape): LoD build + weights +
    # lifting + quantisation + reconstruction of a dense 1M-point surface slice,
    # host-pointer ABI
    try:
        from pcc_attr_b200.synth import cloud_shell

        lxyz, lrgb = cloud_shell(N_POINTS, bits=11, seed=40)
        lp = pb.LodParams()
        lp.num_detail_levels, lp.lod_decimation_type, lp.dist2 = 12, 0, 0
        lp.num_pred_nearest_neighbours, lp.inter_lod_search_range = 3, 1100000
        lp.intra_lod_search_range, lp.intra_lod_prediction_skip_layers = 0, 13
        lp.prediction_with_distribution, lp.pred_weight_blending = 1, 0
        for i in range(3):
            lp.lod_neigh_bias[i] = 1
        for i in range(32):
            lp.lod_sampling_period[i] = 4
        lq = pb.QpSet()
        lq.num_layers, lq.max_qp, lq.fixed_point_qp_offset = 1, 51, 24
        lq.layers[0][0], lq.layers[0][1] = QP, CHROMA_OFFSET
        lf = 8
        pb.attr_lift_encode(lp, lq, lxyz, lrgb, lcp_enabled=1)
        t0 = time.perf_counter()
        pb.attr_lift_encode(lp, lq, lxyz, lrgb, lcp_enabled=1)
        single = time.perf_counter() - t0
        run_jobs([lambda: pb.attr_lift_encode(lp, lq, lxyz, lrgb, lcp_enabled=1)] * lf)
        t0 = time.perf_counter()
        run_jobs([lambda: pb.attr_lift_encode(lp, lq, lxyz, lrgb, lcp_enabled=1)] * lf)
        batch = time.perf_counter() - t0
        lifting = {
            "workload": "1M-point dense surface slice (11-bit), RGB, lifting transform, 12 LoDs, "
                        "distance subsampling, k=3, qp 34, LCP on: LoD build + weights + forward "
                        "lifting + quantisation + reconstruction, host-pointer ABI (H2D/D2H inside)",
            "single_call_ms": 1e3 * single,
            "mpoints_per_s_single": lxyz.shape[0] / single / 1e6,
            "mpoints_per_s_8_in_flight": lf * lxyz.shape[0] / batch / 1e6,
        }
        out["lifting_path"] = lifting
    except Exception as e:
        out["lifting_path"] = {"error": str(e)[:200]}

    # ---- recolouring (SURVEY.md 8f N3b): attribute transfer of the frame's colours
    # onto a half-resolution (duplicate-merged) geometry, host-pointer ABI
    try:
        half = np.ascontiguousarray(np.unique(np.rint(xyz * 0.5).astype(np.int32), axis=0))
        rp = pb.default_recolour_params()
        pb.recolour(rp, xyz, rgb, half, 0.5)
        t0 = time.perf_counter()
        got = pb.recolour(rp, xyz, rgb, half, 0.5)
        rec_s = time.perf_counter() - t0
        rec = {"source_points": int(xyz.shape[0]), "target_points": int(half.shape[0]),
               "ms": 1e3 * rec_s, "mpoints_per_s": xyz.shape[0] / rec_s / 1e6,
               "note": "RGB, defaults of tmc3/TMC3.cpp:1500-1551 (8 forward / 1 backward "
                       "neighbours), host-pointer ABI, pageable buffers, wall clock"}
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import pcc_testlib as tl
        if tl.recolourref_available():
            m = 200000  # bounded CPU sample: the first 200k source points and their targets
            sx, sa = xyz[:m], rgb[:m]
            st = np.ascontiguousarray(np.unique(np.rint(sx * 0.5).astype(np.int32), axis=0))
            t0 = time.perf_counter()
            ref = tl.ref_recolour(tl.make_recolour_params(), sx, sa, 0.5, (0, 0, 0), st)
            cpu_s = time.perf_counter() - t0
            mine = pb.recolour(rp, sx, sa, st, 0.5)
            rec["cpu_reference"] = {"source_points": m, "seconds_one_core": cpu_s,
                                    "mpoints_per_s": m / cpu_s / 1e6,
                                    "identical_points": float((mine == ref).all(axis=1).mean()),
                                    "mean_abs_diff": float(np.abs(mine - ref).mean())}
        out["recolouring"] = rec
        del got
    except Exception as e:
        out["recolouring"] = {"error": str(e)[:200]}

    # ---- the two rows either side of the transform (SURVEY.md 8f N2, N1)
    try:
        theta = np.rint(np.tan(np.linspace(-0.43, 0.04, 64)) * (1 << 18)).astype(np.int32)
        origin, weight = (0, 0, 0), (256, 640, 193128)
        pb.attr_spherical_positions(origin, theta, weight, xyz)
        t0 = time.perf_counter()
        pb.attr_spherical_positions(origin, theta, weight, xyz)
        sph = time.perf_counter() - t0
        pb.attr_raht_encode_symbols(params, qpset, xyz, rgb)
        t0 = time.perf_counter()
        _, runs, _, _, _ = pb.attr_raht_encode_symbols(params, qpset, xyz, rgb)
        sym = time.perf_counter() - t0
        out["adjacent_rows"] = {
            "spherical_positions_ms": 1e3 * sph,
            "spherical_positions_mpoints_per_s": xyz.shape[0] / sph / 1e6,
            "rgb_encode_with_symbols_ms": 1e3 * sym,
            "symbols": int(len(runs)),
            "note": "one 1M-point frame, host-pointer ABI, pageable buffers, wall clock",
        }
    except Exception as e:  # an extra: never take the headline down with it
        out["adjacent_rows"] = {"error": str(e)[:200]}
    return out


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lifting", action="store_true", help="skip the extra lifting-path measurement")
    ap.add_argument("--no-smooth", action="store_true", help="skip the extra smooth-frame measurement")
    ap.add_argument("--workload", default="raht1m", choices=["raht1m", "predlift3m", "lift10m", "raht30m"],
                    help="raht1m = BASELINE configs[1] (the headline); the others are configs[2]-[4] "
                         "(bench_workloads.py)")
    ap.add_argument("--points", type=int, default=0, help="override the point count of --workload")
    ap.add_argument("--frames", type=int, default=FRAMES_PER_STEP,
                    help="independent frames in flight per GPU per step (intra coding: frames "
                         "are independent work units)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of the last timed step's reconstructions and "
                         "coefficients, every frame, to DIR/*.npy (inputs are the same on every run)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "raht1m" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the raht1m workload of --impl ours")
    if args.workload != "raht1m":
        import bench_workloads

        if args.impl == "reference":
            bench_workloads.run_reference(args, sys.modules[__name__])
        else:
            bench_workloads.run(args, sys.modules[__name__])
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
