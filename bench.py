#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 VP8 decode hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload 1080p|features|4k|720p] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): "1080p30 IVF decode, 1 GPU".  No >= 1080p VP8 material exists, so the
streams are synthetic: six DISTINCT 30-frame GOPs produced by the reference's own encoder from seeded
generators at different quantisers / motion (tools/make_bench_streams.sh), repeated round-robin; GOPs are
independent (a key frame resets all codec state), so repeats are extra GOPs of a longer stream.
Other workloads: `features` (SPLITMV / B_PRED / segmentation / golden+altref / 1-8 partitions stream),
`4k` (config 4), `720p` (config 5: 8 distinct streams per GPU incl. the real 720p vector ff2941dd...).

One JSON line on stdout (rank 0):
  value      Mpix/s of the WHOLE decode through vp8gpu_decode_ivf: bitstream in host memory -> entropy
             front end (first partitions on the host, DCT partitions by k_tokens on the device) -> pixel
             kernels -> decoded frames LEFT ON THE DEVICE (SURVEY.md 8d's definition of the metric)
  e2e        the same call with every shown frame copied into pinned host memory inside the timed region
  roofline   per kernel: algorithmic bytes (DESIGN.md) / CUDA-event time vs the measured HBM peak, measured
             on HBM-resident parsed records (all streams advance one frame per batch); `resident_value`
             is that kernel-only throughput (no entropy decode, no copies) -- an explanation, not a claim
  single_stream  one 30-frame GOP decoded alone (latency-bound: fps and ms per frame incl. D2H)
  cpu_baseline   the unmodified reference decoder (oracle/_ref/ref_dump) on one host core
--impl reference: the reference's CPU decode on all usable host cores (one process per core, the clips of
the workload dealt round-robin), same metric / unit / config.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

BD = os.path.join(ROOT, "bench_data")
WORKLOADS = {
    # BASELINE.json configs[1]: six distinct GOPs (different seeds, motion kinds and quantisers)
    "1080p": ["synth1080p_medium_q90.ivf", "synth1080p_hard_q60_s7.ivf", "synth1080p_medium_q110_s21.ivf",
              "synth1080p_medium_q70_s33.ivf", "synth1080p_easy_q60_s5.ivf"],
    "features": ["features1080p_12f.ivf"],             # SPLITMV / B_PRED / multi-partition / golden+altref
    "4k": ["synth4k_medium_q90_30f.ivf"],              # configs[3]
    # configs[4]: 8 distinct 720p streams per GPU: the real 720p vector + 7 seeded synthetic ones
    "720p": [os.path.join(ROOT, "tests", "golden", "vectors", "ff2941dde20090835032c32c0644b6d401610c57"),
             "synth720p_medium_q90.ivf"] + ["synth720p_s%d.ivf" % k for k in range(1, 7)],
    "medium": ["synth1080p_medium_q90.ivf"], "easy": ["synth1080p_easy_q40.ivf"],
}
REF_DUMP = os.path.join(ROOT, "oracle", "_ref", "ref_dump")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def effective_cpus():
    """CPUs this process may actually use: affinity mask and cgroup quota (the GPU box gives the
    container a CPU quota well below the 128 logical CPUs it shows)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def clip_path(name):
    return name if os.path.isabs(name) else os.path.join(BD, name)


def load_instances(names, inst_len=30, per_clip=0):
    """The workload as independent streams ("instances"): every clip cut at key frames into runs of up to
    `inst_len` frames (one GOP of the synthetic clips; `inst_len` consecutive key frames of an all-key
    stream).  Returns (w, h, [list of frame bytes per instance])."""
    import oracle_lib as O  # read_ivf only
    w = h = None
    instances = []
    for n in names:
        cw, ch, frames = O.read_ivf(open(clip_path(n), "rb").read())
        assert w in (None, cw) and h in (None, ch), "clips of one workload share a frame size"
        w, h = cw, ch
        cur = None
        first = len(instances)
        for f in frames:
            key = not (f[0] & 1)
            if cur is None or (key and len(cur) >= inst_len):
                cur = []
                instances.append(cur)
            if len(cur) < inst_len or not key:
                cur.append(f)
        if per_clip:
            del instances[first + per_clip:]
    return w, h, [i for i in instances if i]


def make_ivf(w, h, frames):
    import struct
    out = [b"DKIF" + struct.pack("<HH4sHHIIII", 0, 32, b"VP80", w, h, 30, 1, len(frames), 0)]
    for k, f in enumerate(frames):
        out.append(struct.pack("<IQ", len(f), k))
        out.append(f)
    return b"".join(out)


def reference_mpix_per_s(paths, procs, reps=1):
    """`procs` concurrent reference decoders (one process per core), the clips dealt round-robin, each
    process decoding its whole clip `reps` times."""
    t0 = time.perf_counter()
    ps = [subprocess.Popen([REF_DUMP, "time", paths[k % len(paths)], str(reps)], stdout=subprocess.PIPE, text=True)
          for k in range(procs)]
    outs = [json.loads(p.communicate()[0]) for p in ps]
    wall = time.perf_counter() - t0
    mpix = sum(o["width"] * o["height"] * o["frames"] * reps for o in outs) / 1e6
    return mpix / wall, wall, outs


def run_reference_arm(a, rank, world):
    if rank != 0:
        return
    paths = [clip_path(n) for n in WORKLOADS[a.workload]]
    cores = a.ref_procs or effective_cpus()
    if not os.path.exists(REF_DUMP):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_dump not built"}))
        return
    for _ in range(a.warmup):
        reference_mpix_per_s(paths, cores)
    vals, walls = [], []
    for _ in range(a.steps):
        v, wall, _ = reference_mpix_per_s(paths, cores)
        vals.append(v)
        walls.append(wall)
    v = statistics.mean(vals)
    sample = "%d processes, the %d clips of the workload dealt round-robin, one whole clip per process per step" % (cores, len(paths))
    print(json.dumps({
        "impl": "reference", "metric": "decode_throughput", "value": v, "unit": "Mpix/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": statistics.mean(walls) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_name(a.workload) + "; reference CPU decoder, C++ fallback build (no yasm => no SSE2 asm)"},
        "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": cores, "kind": "reference", "sample": sample, "usable_cpus": effective_cpus()},
        "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def workload_name(wl):
    return {"1080p": "1920x1080 IVF decode, 6 distinct synthetic GOPs x 30 frames (reference-encoder output, seeds/quantisers/motion differ)",
            "features": "1920x1080 IVF decode, feature-complete stream (SPLITMV, B_PRED, segmentation, golden/altref, 1-8 partitions)",
            "4k": "3840x2160 IVF decode, synthetic GOP of 30 frames (BASELINE configs[3])",
            "720p": "1280x720 IVF decode, 8 distinct streams per GPU: real vector ff2941dd + 7 synthetic (BASELINE configs[4])",
            "medium": "1920x1080 IVF decode, synth1080p_medium_q90.ivf", "easy": "1920x1080 IVF decode, synth1080p_easy_q40.ivf"}[wl]


def ncu_traffic(kernel, path):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full`
    capture of this round (profiles/, condensed by tools/summarize_ncu.py); None when there is no capture"""
    if not os.path.exists(path):
        return None
    import csv
    rows = list(csv.reader(open(path)))
    hdr, units = rows[0], rows[1]
    r_i, w_i = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
    vals = [float(r[r_i]) * scale[units[r_i]] + float(r[w_i]) * scale[units[w_i]] for r in rows[2:]
            if kernel + "(" in r[0] or kernel + "_ll(" in r[0]]
    return sum(vals) / len(vals) if vals else None


def synth_1080p(t, w=1920, h=1080, seed=11):
    """seeded synthetic source: drifting smooth pattern, four translating softly textured tiles, light noise"""
    import numpy as np
    rng = np.random.default_rng(seed)
    tex = rng.integers(0, 256, (256, 256)).astype(np.float32)
    for _ in range(3):
        tex = (tex + np.roll(tex, 1, 0) + np.roll(tex, 1, 1) + np.roll(tex, (1, 1), (0, 1))) / 4
    tex = np.clip(128 + (tex - 128) * 3, 0, 255)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    y = 128 + 50 * np.sin(0.012 * (xx + 3 * t)) * np.cos(0.009 * (yy + 2 * t))
    for k, (vx, vy) in enumerate(((3, 1), (-2, 2), (1, -3), (-3, -2))):
        ox, oy = 200 + 400 * k + vx * t, 150 + 180 * k + vy * t
        y[oy:oy + 256, ox:ox + 256] = tex
    y += np.random.default_rng(seed + 1 + t).integers(-1, 2, (h, w))
    cy, cx = np.mgrid[0:(h + 1) // 2, 0:(w + 1) // 2].astype(np.float32)
    u = 128 + 30 * np.sin(0.01 * (cx + t))
    v = 128 + 30 * np.cos(0.012 * (cy - t))
    return tuple(np.clip(p, 0, 255).astype(np.uint8) for p in (y, u, v))


def bench_encode(a, local):
    """fps of Encoder::encode_with_target_size at 1080p through the C ABI (host planes in, compressed
    frame out, every step incl. H2D of the source and D2H of the records), next to the reference
    encoder (REALTIME_QUALITY, one core) on the same raw frames."""
    import numpy as np

    from alfalfa_b200 import Context, Encoder
    w, h, n = 1920, 1080, a.encode_frames
    src = [synth_1080p(t) for t in range(n)]
    ctx = Context(w, h, device=local, max_frames=32)
    enc = Encoder(ctx)
    enc.encode_with_target_size(*src[0], a.encode_target)  # warm-up (key frame, allocations)
    del enc
    enc = Encoder(ctx)
    sizes, qis, psnrs, times, ssims, lfs, blobs, sses, phases = [], [], [], [], [], [], [], [], []
    for t in range(n):
        t0 = time.perf_counter()
        blob, qi = enc.encode_with_target_size(*src[t], a.encode_target)
        times.append(time.perf_counter() - t0)
        sizes.append(len(blob))
        blobs.append(bytes(blob))
        qis.append(qi)
        phases.append(enc.timeline())
        st = enc.stats()
        ssims.append(st["ssim"])
        lfs.append(st["loop_filter_level"])
        rec = enc.reconstruction()
        ry = rec.planes()[0][:h, :w]
        rec.release()
        sses.append(float(np.sum((ry.astype(np.float64) - src[t][0].astype(np.float64)) ** 2)))
        mse = sses[-1] / (w * h)
        psnrs.append(99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse))
    launches = ctx.launch_count()
    del enc
    ctx.close()
    out = {"metric": "encode_with_target_size fps @1080p", "frames": n, "target_bytes": a.encode_target,
           "fps": (n - 1) / sum(times[1:]), "key_frame_ms": times[0] * 1e3, "inter_frame_ms": 1e3 * sum(times[1:]) / (n - 1),
           "bytes_per_frame": sum(sizes) / n, "qi": qis, "loop_filter_level": lfs, "psnr_y": sum(psnrs) / n,
           "ssim_y": sum(ssims) / n, "gpu_launches": int(launches),
           # host wall clock per phase of a call (vp8gpu_encoder_timeline), mean over the inter frames; every phase ends with
           # its device work finished; `writer` runs next to `loop_filter_search`, so the phases add up to more than `total`
           "inter_frame_phases_ms": {k: round(sum(p[k] for p in phases[1:]) / max(1, n - 1), 3) for k in (phases[0] if phases else {})},
           "key_frame_phases_ms": {k: round(v, 3) for k, v in (phases[0] if phases else {}).items()},
           "note": "the reference encoder's decisions on the device (k_enc_rd: rdcost, B_PRED trial, motion-vector census, diamond "
                   "search, chroma by distortion) and its writer policy: the frames are byte-identical to the reference encoder's "
                   "(tests/test_gpu_encoder.py; `reference.identical_frames` below compares this very run)",
           "searches": ("candidate by candidate (VP8GPU_ENC_SPECULATE=0)" if os.environ.get("VP8GPU_ENC_SPECULATE", "1")[:1] == "0" else
                        "the probes of the target-size bisection in one k_enc_rd launch (<= 33 sampled passes), the trials of the "
                        "loop-filter search in one k_loopfilter launch, the frame written on a host thread meanwhile "
                        "(same bytes as candidate by candidate: tests/test_gpu_encoder.py)")}
    # SURVEY 8(d), encode: the probe-free minimum of a frame is source P + reference P read, reconstruction P written
    # (P = 384 B per macroblock) + its coefficients; over the time of the full pass (k_enc_rd, one launch, incl. the
    # download of its records: `full_pass` of the timeline) that is the fraction of the HBM roofline the decision kernel
    # reaches -- it is a latency chain of (cols + rows) macroblock steps on 68 warps, not a bandwidth consumer
    if phases and n > 1:
        peak, peak_src = measured_peaks()
        mbs = ((w + 15) // 16) * ((h + 15) // 16)
        alg = 3 * 384 * mbs + 4.0 * (sum(sizes[1:]) / (n - 1))  # (tokens ~ bytes of the frame: an upper bound of 4 B per coded byte)
        fp_ms = out["inter_frame_phases_ms"].get("full_pass", 0.0)
        if fp_ms > 0:
            out["roofline"] = {"bound": "hbm", "kernel": "k_enc_rd (full pass of an inter frame)", "bytes_per_frame": alg,
                               "full_pass_ms": fp_ms, "achieved": alg / (fp_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                               "frac": alg / (fp_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": None}
    ref_enc = os.path.join(ROOT, "oracle", "_ref", "ref_encode")
    if os.path.exists(ref_enc):
        import tempfile
        m = min(n, 6)  # bounded sample: the reference runs at a few fps
        with tempfile.TemporaryDirectory() as d:
            raw = os.path.join(d, "src.yuv")
            with open(raw, "wb") as f:
                for t in range(m):
                    for p in src[t]:
                        f.write(p.tobytes())
            env = dict(os.environ, REF_RAW=raw, REF_TARGET=str(a.encode_target))
            r = subprocess.run([ref_enc, os.path.join(d, "o.ivf"), str(w), str(h), str(m), "1000", "0"], env=env,
                               capture_output=True, text=True)
            try:
                j = json.loads(r.stdout.strip().splitlines()[-1])
                # like for like over the SAME first m frames: bytes, PSNR of the pooled MSE (ref_encode.cc), frame identity
                from alfalfa_b200.decoder import read_ivf
                ref_frames = read_ivf(open(os.path.join(d, "o.ivf"), "rb").read())[2]
                pooled = sum(sses[:m]) / (w * h * m)
                out["reference"] = {"fps": j["fps"], "bytes_per_frame": j["bytes"] / m, "psnr_y": j["psnr_y"], "frames": m,
                                    "cores": 1, "kind": "reference", "sample": "unmodified reference encoder, REALTIME_QUALITY, "
                                    "encode_with_target_size, the same first %d raw frames" % m,
                                    "ours_same_frames": {"bytes_per_frame": sum(sizes[:m]) / m,
                                                         "psnr_y": 99.0 if pooled == 0 else 10 * np.log10(255.0 ** 2 / pooled)},
                                    "identical_frames": sum(1 for x, y in zip(ref_frames, blobs[:m]) if x == y)}
            except Exception as e:  # noqa: BLE001
                out["reference"] = {"unavailable": "%s %s" % (e, r.stderr[-200:])}
    return out


def run_exchange(rank, world, local, timeout=150, tool_args=()):
    """tools/split_gop_check.py on every rank's GPU, as child processes forming their own process group; rank 0 returns
    the tool's JSON (mismatches, hand-over time, raster exchange time per 1080p raster), the others None"""
    drop = ("TORCHELASTIC", "GROUP_", "ROLE_")  # torchrun's agent store must not be mistaken for the children's
    env = {k: v for k, v in os.environ.items() if not k.startswith(drop)}
    base = int(os.environ.get("MASTER_PORT", "29500"))
    env.update(RANK=str(rank), LOCAL_RANK=str(local), WORLD_SIZE=str(world), LOCAL_WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
               MASTER_PORT=str(base + 211 if base + 211 < 65000 else base - 211))
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "split_gop_check.py")] + list(tool_args), env=env, capture_output=True, text=True,
                           timeout=timeout)
        if rank != 0:
            return None
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if lines:
            out = json.loads(lines[-1])
            out["exit_code"] = r.returncode
            return out
        return {"error": (r.stderr or r.stdout)[-300:], "exit_code": r.returncode}
    except Exception as e:  # noqa: BLE001  (timeout, malformed output)
        return {"error": ("%s: %s" % (type(e).__name__, e))[:300]} if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="1080p", choices=list(WORKLOADS))
    ap.add_argument("--gop-instances", type=int, default=0, help="streams advanced together in the HBM-resident run (0 = 128; 4k: 16; 720p: 8)")
    ap.add_argument("--replicas", type=int, default=0, help="repeats of the instance set in the whole-decode runs (0 = auto)")
    ap.add_argument("--threads", type=int, default=0, help="host workers for the whole-decode runs (0 = auto)")
    ap.add_argument("--ref-procs", type=int, default=0, help="reference processes (0 = usable CPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-encode", action="store_true", help="skip the 1080p encode section")
    ap.add_argument("--no-reencode", action="store_true", help="skip the 1080p re-encoding (update_residues) section")
    ap.add_argument("--no-exchange", action="store_true", help="N > 1: skip the split-GOP hand-over over NCCL (exchange section)")
    ap.add_argument("--encode-frames", type=int, default=30)
    ap.add_argument("--encode-target", type=int, default=45000, help="bytes per frame for encode_with_target_size")
    ap.add_argument("--host-tokens", action="store_true",
                    help="whole-decode runs: DCT partitions decoded by the host workers instead of k_tokens on the device")
    ap.add_argument("--host-stats", action="store_true", help="diagnostic: print host time accounting to stderr")
    ap.add_argument("--ncu-summary", default=os.path.join(ROOT, "profiles", "r2_final_ncu_full_summary.csv"),
                    help="condensed `ncu --set full` capture; it was taken with 64 streams per launch (--ncu-streams)")
    ap.add_argument("--ncu-streams", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames the last e2e step decoded to DIR/*.npy (a seeded sample of "
                         "whole frames and per-plane sums of every frame), so that two builds can be compared")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 0)

    from alfalfa_b200 import multigpu as M
    if a.impl == "reference":  # CPU arm: rank 0 alone runs it, no process group needed
        rank, world, _ = M.rank_info()
        run_reference_arm(a, rank, world)
        return
    rank, world, local, dist = M.init()
    barrier, max_over_ranks, sum_over_ranks = M.barrier, M.reduce_max, M.reduce_sum

    import numpy as np

    from alfalfa_b200 import Context, capi

    w, h, instances = load_instances(WORKLOADS[a.workload], per_clip=1 if a.workload == "720p" else 0)
    mpix_frame = w * h / 1e6
    L = capi.lib()
    n_mbs = ((w + 15) // 16) * ((h + 15) // 16)
    # the wavefront kernels are latency bound: 128 streams per launch take barely longer than 64 (profiles/r2_notes.md)
    G = a.gop_instances or (8 if a.workload == "720p" else (16 if a.workload == "4k" else 128))
    n_inst = len(instances)
    max_len = max(len(i) for i in instances)

    # ---------------- set-up of the kernel-level run: parse every distinct instance once ----------------
    parsed = []  # per distinct instance: list of (desc, mbs, tok, split)
    h2d_host_tokens = [0] * n_inst
    h2d_dev_tokens = [0] * n_inst
    stat = {"inter": 0, "intra": 0, "tok": 0, "filt": 0, "z": 0, "inter_frames": 0, "frames": 0}
    inst_stat = []
    for k, frames in enumerate(instances):
        st, pf = C.c_void_p(), C.c_void_p()
        capi.check(L.vp8gpu_state_create(w, h, C.byref(st)))
        capi.check(L.vp8gpu_parsed_create(C.byref(pf)))
        cur = []
        ist = dict.fromkeys(stat, 0)
        for f in frames:
            capi.check(L.vp8gpu_parse_frame(st, f, len(f), pf), None, "parse")
            d = capi.FrameDesc.from_buffer_copy(bytes(L.vp8gpu_parsed_desc(pf).contents))
            mbs = np.frombuffer(C.string_at(L.vp8gpu_parsed_mbs(pf), n_mbs * 32), dtype=capi.MB_DTYPE).copy()
            tok = (np.frombuffer(C.string_at(L.vp8gpu_parsed_tokens(pf), d.n_tokens * 4), dtype="<u4").copy()
                   if d.n_tokens else np.zeros(1, "<u4"))
            sp = (np.frombuffer(C.string_at(L.vp8gpu_parsed_split(pf), d.n_split * 64), dtype="u1").copy()
                  if d.n_split else np.zeros(64, "u1"))
            cur.append((d, mbs, tok, sp))
            h2d_host_tokens[k] += n_mbs * 32 + d.n_tokens * 4 + d.n_split * 64 + 512
            h2d_dev_tokens[k] += n_mbs * 32 + d.n_split * 64 + 1536 + len(f)  # records + probabilities + raw partitions
            intra = mbs["ref_frame"] == 0
            ist["inter"] += int((~intra).sum())
            ist["intra"] += int(intra.sum())
            ist["tok"] += int(d.n_tokens)
            ist["filt"] += int((mbs["lf_level"] != 0).sum())
            ist["inter_frames"] += 0 if d.key_frame else 1
            ist["frames"] += 1
            if d.n_tokens:
                ist["z"] += len(np.unique((tok[:d.n_tokens] >> 20) & 31 | (np.repeat(np.arange(n_mbs), mbs["tok_cnt"]) << 5)))
            tok_intra = int(mbs["tok_cnt"][intra].sum())
            ist.setdefault("tok_intra", 0)
            ist["tok_intra"] += tok_intra
        L.vp8gpu_state_destroy(st)
        L.vp8gpu_parsed_destroy(pf)
        parsed.append(cur)
        inst_stat.append(ist)

    ctx = Context(w, h, device=local, max_frames=G * (max_len + 1) + 64)
    batches = (C.c_void_p * max_len)()
    keep = [{"refs": [-1, -1, -1], "frames": []} for _ in range(G)]
    launches_per_step = {"k_inter": 0, "k_intra": 0, "k_loopfilter": 0}
    for pos in range(max_len):
        members = [g for g in range(G) if pos < len(parsed[g % n_inst])]
        jobs = (capi.Job * len(members))()
        any_inter = False
        for j, g in enumerate(members):
            d, mbs, tok, sp = parsed[g % n_inst][pos]
            state = keep[g]
            out = ctx.alloc_frame()
            state["frames"].append(out)
            jobs[j].desc = C.pointer(d)
            jobs[j].mbs = mbs.ctypes.data
            jobs[j].tokens = tok.ctypes.data
            jobs[j].split = sp.ctypes.data
            jobs[j].refs[:] = state["refs"]
            jobs[j].out = out.id
            r = state["refs"]
            if d.key_frame:  # Frame::copy_to (frame.cc:272-307)
                r[0] = r[1] = r[2] = out.id
            else:
                any_inter = True
                if d.copy_to_alternate == 1:
                    r[2] = r[0]
                elif d.copy_to_alternate == 2:
                    r[2] = r[1]
                if d.copy_to_golden == 1:
                    r[1] = r[0]
                elif d.copy_to_golden == 2:
                    r[1] = r[2]
                if d.refresh_golden:
                    r[1] = out.id
                if d.refresh_alternate:
                    r[2] = out.id
                if d.refresh_last:
                    r[0] = out.id
        b = C.c_void_p()
        capi.check(L.vp8gpu_batch_upload(ctx.h, jobs, len(members), C.byref(b)), ctx.h, "batch_upload")
        batches[pos] = b
        launches_per_step["k_inter"] += 1 if any_inter else 0
        launches_per_step["k_intra"] += 1
        launches_per_step["k_loopfilter"] += 1
    ctx.sync()
    for k in stat:
        stat[k] = sum(inst_stat[g % n_inst][k] for g in range(G))
    stat["tok_intra"] = sum(inst_stat[g % n_inst]["tok_intra"] for g in range(G))
    frames_resident = stat["frames"]

    def resident_step():
        ms = C.c_float(0)
        capi.check(L.vp8gpu_batches_run(ctx.h, 0, batches, max_len, C.byref(ms)), ctx.h, "batches_run")
        return ms.value

    # ---------------- kernel-level run on HBM-resident records (roofline only) ----------------
    for _ in range(max(a.warmup, 3)):
        resident_step()
    ctx.sync()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier(dist)
    ctx.sync()
    step_ms = [resident_step() for _ in range(a.steps)]
    ctx.sync()
    barrier(dist)
    launches_resident = ctx.launch_count() - launches0
    resident_ms = max_over_ranks(dist, local, sum(step_ms))
    resident_value = sum_over_ranks(dist, local, frames_resident * mpix_frame * a.steps) / (resident_ms / 1e3)
    y, _, _ = keep[0]["frames"][-1].planes()
    assert y.std() > 1.0, "decoded frame looks empty"

    kt = np.zeros((max_len, 3))
    reps = 3
    for _ in range(reps):
        for pos in range(max_len):
            ms3 = (C.c_float * 3)()
            capi.check(L.vp8gpu_batch_run_timed(ctx.h, 0, batches[pos], ms3), ctx.h, "batch_run_timed")
            kt[pos] += np.array(list(ms3)) / reps
    k_total = kt.sum(axis=0)  # ms per step per kernel
    names = ["k_inter", "k_intra", "k_loopfilter"]
    # algorithmic bytes per step (DESIGN.md "kernels and their rooflines"); P = 384 bytes per macroblock
    step_bytes = {
        "k_inter": stat["inter"] * (384 * 2 + 32) + 4 * (stat["tok"] - stat["tok_intra"]),
        "k_intra": stat["intra"] * (384 + 32) + 4 * stat["tok_intra"],
        "k_loopfilter": stat["filt"] * (384 * 2 + 32),
    }
    peak, peak_src = measured_peaks()
    per_kernel = {}
    for k, nm in enumerate(names):
        nl = max(launches_per_step[nm], 1)
        gbs = step_bytes[nm] / (k_total[k] / 1e3) / 1e9 if k_total[k] > 0 else 0.0
        per_kernel[nm] = {"achieved": gbs, "frac": gbs / peak, "bytes_per_launch": step_bytes[nm] / nl,
                          "avg_launch_ms": float(k_total[k]) / nl, "launches_per_step": launches_per_step[nm],
                          # DRAM bytes of the ncu capture, scaled from its streams per launch to this run's
                          "traffic": (lambda t: None if t is None else t * G / a.ncu_streams)(ncu_traffic(nm, a.ncu_summary))}
    dname = names[int(np.argmax(k_total))]
    dk = per_kernel[dname]
    # whole-frame budget of SURVEY.md 8(d): P + I*P + 32 Z + 48 M per frame, charged to the sum of the kernels
    P = 384 * n_mbs
    pipeline_bytes = stat["frames"] * P + stat["inter_frames"] * P + 32 * stat["z"] + 48 * n_mbs * stat["frames"]
    pipeline_gbs = pipeline_bytes / (statistics.mean(step_ms) / 1e3) / 1e9
    roofline = {"bound": "hbm", "kernel": dname, "achieved": dk["achieved"], "peak": peak, "unit": "GB/s",
                "frac": dk["frac"], "traffic": dk["traffic"], "peak_source": peak_src,
                "bytes_per_launch": dk["bytes_per_launch"], "avg_launch_ms": dk["avg_launch_ms"],
                "kernel_ms_per_step": dict(zip(names, [float(x) for x in k_total])), "kernels": per_kernel,
                "pipeline_achieved": pipeline_gbs, "pipeline_frac": pipeline_gbs / peak,
                "resident_value": resident_value, "resident_ms_per_step": resident_ms / a.steps,
                "resident_frames_per_step": frames_resident,
                "resident_note": "%d streams (%d distinct) advanced one frame per batch, parsed records resident in HBM: "
                                 "pixel kernels only, no entropy decode, no copies" % (G, min(G, n_inst))}

    for b in batches:
        L.vp8gpu_batch_free(ctx.h, b)
    for s_ in keep:
        for fr in s_["frames"]:
            fr.release()
    ctx.close()

    # ---------------- whole decode through the public API: `value` (output stays on the device) and `e2e` ----------------
    # Host workers, shared by the ranks.  With the DCT partitions decoded on the device a worker only
    # walks first partitions, and the number of GOPs in flight (= workers) is what fills the device:
    # four per usable CPU; when the workers parse everything, two (they also wait on DMA / the dispatcher).
    per_cpu = 2 if a.host_tokens else 4
    threads = a.threads or max(2, min(96, per_cpu * effective_cpus() // max(world, 1)))
    frames_per_set = sum(len(i) for i in instances)
    # enough independent streams that every worker gets about four of them
    R = a.replicas or max(1, -(-4 * threads // n_inst))
    if a.workload == "4k":
        R = a.replicas or max(1, -(-threads // n_inst))
    ctx2 = Context(w, h, device=local, max_frames=threads * (10 if a.host_tokens else int(os.environ.get("VP8GPU_TOK_SLOTS", 96)) + 6) + 64)
    ctx2.set_device_tokens(not a.host_tokens)
    ctx2_display_bytes = ctx2.display_bytes
    dst = C.c_void_p()
    while True:  # the pinned output buffer is w*h*1.5 bytes per frame: halve the run if the box cannot pin that much
        out_bytes = ctx2.display_bytes * frames_per_set * R
        if L.vp8gpu_host_alloc(C.byref(dst), out_bytes) == 0:
            break
        if R <= 1:
            capi.check(capi.ERR_NOMEM, ctx2.h, "host_alloc")
        R = max(1, R // 2)
    all_frames = []
    for _ in range(R):
        for inst in instances:
            all_frames.extend(inst)
    big = make_ivf(w, h, all_frames)
    n_job_frames = len(all_frames)
    nd, ns = C.c_uint32(0), C.c_uint32(0)

    def decode_step(with_output):
        t0 = time.perf_counter()
        capi.check(L.vp8gpu_decode_ivf(ctx2.h, big, len(big), threads, dst if with_output else None,
                                       out_bytes if with_output else 0, C.byref(nd), C.byref(ns)), ctx2.h, "decode_ivf")
        capi.check(L.vp8gpu_ctx_sync(ctx2.h), ctx2.h, "sync")
        return time.perf_counter() - t0

    results = {}
    for name, with_output in (("value", False), ("e2e", True)):
        for _ in range(max(a.warmup, 1)):
            decode_step(with_output)
        l0 = ctx2.launch_count()
        barrier(dist)
        secs = [decode_step(with_output) for _ in range(a.steps)]
        barrier(dist)
        tot = max_over_ranks(dist, local, sum(secs))
        results[name] = {"mpix_s": sum_over_ranks(dist, local, n_job_frames * mpix_frame * a.steps) / tot,
                         "ms_per_step": tot / a.steps * 1e3, "launches": int(ctx2.launch_count() - l0)}
        if a.host_stats:
            stt = (C.c_double * 8)()
            L.vp8gpu_decode_ivf_stats(ctx2.h, stt)
            print("%s host stats (last step, s): parse %.3f wait_dispatch %.3f wait_dma %.3f | dispatcher: submit %.3f downloads %.3f "
                  "idle %.3f | batches %d frames %d | step wall %.3f" % (name, *list(stt)[:6], int(stt[6]), int(stt[7]), secs[-1]),
                  file=sys.stderr)
    clocks = sampler.stop()
    # sanity: the output buffer holds pictures (the real 720p vector opens with a flat frame: look at a few)
    probe = np.frombuffer(C.string_at(dst, min(int(out_bytes), 8 * ctx2_display_bytes)), dtype=np.uint8)
    assert probe.std() > 1.0
    if a.dump_outputs and rank == 0:
        dump_decoded_frames(a.dump_outputs, dst, ctx2_display_bytes, w, h, nd.value, ns.value)

    # ---------------- one stream alone (latency-bound): a single instance, one worker, frames copied out ----------------
    one = make_ivf(w, h, instances[0])
    single = None
    if rank == 0:
        def one_step():
            t0 = time.perf_counter()
            capi.check(L.vp8gpu_decode_ivf(ctx2.h, one, len(one), 1, dst, out_bytes, C.byref(nd), C.byref(ns)), ctx2.h, "decode_ivf")
            capi.check(L.vp8gpu_ctx_sync(ctx2.h), ctx2.h, "sync")
            return time.perf_counter() - t0
        one_step()
        ts = [one_step() for _ in range(3)]
        single = {"frames": len(instances[0]), "fps": len(instances[0]) / min(ts), "ms_per_frame": 1e3 * min(ts) / len(instances[0]),
                  "mpix_s": len(instances[0]) * mpix_frame / min(ts), "api": "vp8gpu_decode_ivf, 1 worker, host IVF -> pinned host YUV"}
    L.vp8gpu_host_free(dst)
    ctx2.close()

    # ---------------- encode: 1080p encode_with_target_size (BASELINE.json config 3) ----------------
    encode = None
    if rank == 0 and not a.no_encode:
        encode = bench_encode(a, local)

    # ---------------- re-encoding: Encoder::reencode / update_residues at 1080p (SURVEY 8 f3) ----------------
    # In a child process under a timeout: this path was finished after the round's GPU minutes were spent (checked
    # bit-exactly under the SIMT emulator only, DESIGN.md section 5), so whatever it does on hardware it must not be
    # able to take this line's other numbers with it.
    reencode = None
    if rank == 0 and not a.no_reencode:
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "reencode_bench.py"), "--device", str(local)],
                               capture_output=True, text=True, timeout=240)
            reencode = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as e:  # noqa: BLE001  (timeout, malformed output)
            reencode = {"error": ("%s: %s" % (type(e).__name__, e))[:300]}

    # ---------------- the exchange step (N > 1): a GOP that continues on other GPUs ----------------
    # BASELINE.json config 4: rank 0 decodes the first half of a single-GOP 1080p stream with live golden / altref
    # references and hands its Decoder over -- DecoderState record + the distinct reference rasters, ncclBroadcast
    # straight between rasters on the lane stream (vp8gpu_comm_*, csrc/comm.cc) -- every other rank continues the decode
    # and checks it bit for bit against decoding the whole stream alone.  Every rank runs tools/split_gop_check.py as a
    # child (own process group on another port, own CUDA context on the rank's GPU) under a timeout: a communicator that
    # does not come up costs this section, not the line.
    exchange = None
    if dist is not None and not a.no_exchange:
        dist.barrier()  # rank 0 comes from its encode sections: the children start together
        exchange = run_exchange(rank, world, local)
        dist.barrier()

    # ---------------- CPU baseline (rank 0, one core, bounded sample) ----------------
    cpu = None
    if rank == 0 and not a.no_cpu_baseline:
        paths = [clip_path(n) for n in WORKLOADS[a.workload]]
        if os.path.exists(REF_DUMP):
            v, wall, outs = reference_mpix_per_s(paths[:1], 1, reps=2)
            o = outs[0]
            cpu = {"value": o["mpix_per_s"], "unit": "Mpix/s", "cores": 1, "kind": "reference",
                   "sample": "first clip of the workload (%d frames), best of 2, unmodified reference decoder (C++ fallback, no yasm): "
                             "parse %.2fs recon %.2fs loopfilter %.2fs" % (o["frames"], o["parse_s"], o["recon_s"], o["loopfilter_s"])}
        else:
            import oracle_lib as O
            data = open(paths[0], "rb").read()
            ph = (C.c_double * 3)()
            n = C.c_uint32()
            O.lib().vp8o_time_ivf(data, len(data), 2, 100000, ph, C.byref(n))
            cpu = {"value": n.value * mpix_frame / sum(ph), "unit": "Mpix/s", "cores": 1, "kind": "port",
                   "sample": "first clip of the workload, best of 2, oracle/vp8_oracle.c"}

    if rank == 0:
        h2d = (h2d_host_tokens if a.host_tokens else h2d_dev_tokens)
        h2d_step = int(sum(h2d) * R)
        print(json.dumps({
            "metric": "decode_throughput", "value": results["value"]["mpix_s"], "unit": "Mpix/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": results["value"]["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(a.workload) + "; %d independent streams per step per GPU (%d distinct x %d)" % (n_inst * R, n_inst, R),
                       "value_definition": "whole decode by vp8gpu_decode_ivf: bitstream in host memory -> entropy decode (host first "
                                           "partitions + k_tokens) -> pixel kernels, decoded frames left on the device (SURVEY 8d)",
                       "frames_per_step": n_job_frames, "host_threads": threads,
                       "l2": "working set %.0f MB of rasters per step > 126 MB L2, no flush needed" % (n_job_frames * ctx_bytes(w, h) / 1e6),
                       "bit_exact": "tests/test_gpu_parity.py (53/53 golden SHA-1 + per-frame oracle + reference SHA-1 of every bench clip)"},
            "e2e": {"value": results["e2e"]["mpix_s"], "unit": "Mpix/s", "h2d_bytes_per_step": h2d_step,
                    "dct_partitions": "host workers" if a.host_tokens else "k_tokens on the device",
                    "d2h_bytes_per_step": int(out_bytes), "ms_per_step": results["e2e"]["ms_per_step"],
                    "api": "vp8gpu_decode_ivf (host IVF bytes -> pinned host YUV)"},
            "gpu_launches": results["value"]["launches"], "gpu_launches_e2e": results["e2e"]["launches"],
            "gpu_launches_resident": int(launches_resident),
            "roofline": roofline, "single_stream": single, "cpu_baseline": cpu, "encode": encode, "reencode": reencode,
            "exchange": exchange, "clocks": clocks}))
    if dist is not None:
        dist.destroy_process_group()


def dump_decoded_frames(out_dir, dst, frame_bytes, w, h, n_decoded, n_shown, max_bytes=48 << 20):
    """What the last timed e2e step handed its caller: the display rectangles (Y, U, V) of the shown frames in stream
    order.  Written as float64 per-plane sums of every frame (frame_plane_sums.npy, [n_shown, 3]), a seeded sample of
    whole frames (sampled_frames.npy, float32 [k, frame_bytes], at most `max_bytes`), their stream positions
    (sampled_frame_index.npy) and [n_decoded, n_shown] (frame_counts.npy)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frames = np.frombuffer((C.c_uint8 * (n_shown * frame_bytes)).from_address(dst.value), np.uint8).reshape(n_shown, frame_bytes)
    ys, cs = w * h, ((w + 1) // 2) * ((h + 1) // 2)
    planes = (frames[:, :ys], frames[:, ys:ys + cs], frames[:, ys + cs:])
    sums = np.stack([p.sum(axis=1, dtype=np.float64) for p in planes], axis=1)
    k = max(1, min(n_shown, max_bytes // (4 * frame_bytes)))
    index = np.sort(np.random.default_rng(0).choice(n_shown, k, replace=False))
    np.save(os.path.join(out_dir, "frame_plane_sums.npy"), sums)
    np.save(os.path.join(out_dir, "sampled_frames.npy"), frames[index].astype(np.float32))
    np.save(os.path.join(out_dir, "sampled_frame_index.npy"), index.astype(np.float64))
    np.save(os.path.join(out_dir, "frame_counts.npy"), np.array([n_decoded, n_shown], np.float64))


def ctx_bytes(w, h):
    return ((w + 15) // 16 * 16) * ((h + 15) // 16 * 16) * 1.5


if __name__ == "__main__":
    main()
