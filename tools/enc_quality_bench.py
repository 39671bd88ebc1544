#!/usr/bin/env python3
"""GPU-box tool: the encoder at REALTIME_QUALITY (Salsify's setting, the default) next to BEST_QUALITY (ExCamera's
xc-enc default) at 1080p on bench.py's encode clip (bench.synth_1080p).  Records, per quality:
  * frames per second of encode_with_quantizer and encode_with_target_size (inter frames; every call ends with the
    frame on the host, so host time around it covers the device work),
  * vp8gpu_encoder_timeline phases, mean over the inter frames,
  * SHA-1 of every emitted frame (repeats must agree),
and at BEST the rate of Encoder::reencode's two device paths (reencode_as_interframe, update_residues) on a chunk the
encoder itself wrote, the card's name and power limit, and -- where it is built -- the unmodified
reference encoder at BEST (oracle/_ref/ref_encode_best) on one core for two frames (and whether its frames equal ours).
usage: tools/enc_quality_bench.py [--frames N] [--qi Q] [--target BYTES] [--repeats R] [--out FILE.json]"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from alfalfa_b200 import Context, Decoder, Encoder  # noqa: E402

W, H = 1920, 1080


def card():
    """name and power limit of GPU 0, read next to the measurement"""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"name": "unavailable", "power_limit": "unavailable (%s)" % e}


def run_encoder(ctx, src, quality, mode, qi, target):
    """one Encoder over all frames: per-frame seconds, SHA-1s, quantisers, inter-frame timeline"""
    enc = Encoder(ctx, quality=quality)
    times, digests, qis, phases = [], [], [], []
    for planes in src:
        t0 = time.perf_counter()
        if mode == "quantizer":
            blob, q = enc.encode_with_quantizer(*planes, qi), qi
        else:
            blob, q = enc.encode_with_target_size(*planes, target)
        times.append(time.perf_counter() - t0)
        digests.append(hashlib.sha1(blob).hexdigest())
        qis.append(q)
        phases.append(enc.timeline())
    del enc
    inter = phases[1:]
    return {"fps_inter": (len(times) - 1) / sum(times[1:]), "key_frame_ms": 1e3 * times[0],
            "inter_frame_ms": [round(1e3 * t, 3) for t in times[1:]], "qi": qis, "frames_sha1": digests,
            "inter_frame_phases_ms": {k: round(sum(p[k] for p in inter) / len(inter), 3) for k in inter[0]}}


def reencode_rates(ctx, src, qi, repeats):
    """Encoder::reencode's device paths at BEST on a whole chunk (options 1 + 4): the previous chunk = frames 0..n/2
    (REALTIME, as a sender would have coded it), this chunk = frames n/2.. coded on their own; a BEST Encoder built
    from the receiver's state re-encodes it towards the source frames"""
    n = len(src)
    half = n // 2
    prev = Encoder(ctx)
    rx = Decoder(ctx)
    for planes in src[:half + 1]:
        rx.get_frame_output(prev.encode_with_quantizer(*planes, qi))[1].release()
    state = rx.serialize()
    del prev, rx
    chunk_enc = Encoder(ctx)
    chunk = [chunk_enc.encode_with_quantizer(*planes, qi) for planes in src[half:]]
    del chunk_enc
    pd = Decoder(ctx)
    preds = []
    for c in chunk:
        pf = pd.parse_frame(c, keep_labels=True)
        pd.decode_frame(pf)
        preds.append(pf)
    targets = src[half:]
    as_inter, residues, digests = [], [], None
    for _ in range(repeats):
        enc = Encoder.from_decoder(ctx, Decoder.deserialize(ctx, state), quality="best")
        out = []
        t0 = time.perf_counter()
        out.append(enc.reencode_as_interframe(*targets[0], preds[0], qi))
        as_inter.append(time.perf_counter() - t0)
        for i in range(1, len(preds)):
            t0 = time.perf_counter()
            out.append(enc.update_residues(*targets[i], preds[i], -1, i == len(preds) - 1))
            residues.append(time.perf_counter() - t0)
        d = [hashlib.sha1(b).hexdigest() for b in out]
        assert digests is None or d == digests, "re-encoding is not deterministic"
        digests = d
        del enc
    del pd, preds
    return {"chunk_frames": len(chunk), "reencode_as_interframe_fps": len(as_inter) / sum(as_inter),
            "update_residues_fps": len(residues) / sum(residues), "frames_sha1": digests}


def reference_best(src, qi, ours):
    """the unmodified reference encoder, BEST_QUALITY, encode_with_quantizer, one process (single-threaded)"""
    tool = os.path.join(ROOT, "oracle", "_ref", "ref_encode_best")
    if not os.path.exists(tool):
        return {"unavailable": "oracle/_ref/ref_encode_best is not built"}
    with tempfile.TemporaryDirectory() as d:
        raw, out = os.path.join(d, "src.yuv"), os.path.join(d, "o.ivf")
        with open(raw, "wb") as f:
            for planes in src:
                for p in planes:
                    f.write(p.tobytes())
        pin = ["taskset", "-c", "0"] if shutil.which("taskset") else []
        r = subprocess.run(pin + [tool, out, str(W), str(H), str(len(src)), "1000", str(qi)],
                           env=dict(os.environ, REF_RAW=raw), capture_output=True, text=True)
        if r.returncode != 0:
            return {"unavailable": r.stderr[-300:]}
        j = json.loads(r.stdout.strip().splitlines()[-1])
        from alfalfa_b200.decoder import read_ivf
        frames = read_ivf(open(out, "rb").read())[2]
    return {"fps": j["fps"], "frames": len(src), "cores": 1, "quality": "best", "mode": "encode_with_quantizer q%d" % qi,
            "identical_frames": sum(1 for f, s in zip(frames, ours) if hashlib.sha1(f).hexdigest() == s)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--qi", type=int, default=60)
    ap.add_argument("--target", type=int, default=45000)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    src = [bench.synth_1080p(t) for t in range(a.frames)]
    ctx = Context(W, H, device=0, max_frames=48)
    warm = Encoder(ctx, quality="best")  # module load, allocations, the buffer pool of the context
    warm.encode_with_quantizer(*src[0], a.qi)
    warm.encode_with_target_size(*src[1], a.target)
    del warm
    res = {"card": card(), "size": "%dx%d" % (W, H), "clip": "bench.synth_1080p", "frames": a.frames, "qi": a.qi,
           "target_bytes": a.target, "repeats": a.repeats, "runs": {}}
    for mode in ("quantizer", "target_size"):
        for quality in ("realtime", "best"):
            res["runs"]["%s/%s" % (mode, quality)] = []
        for rep in range(a.repeats):  # the two qualities alternate, so that drift on a shared host hits both
            order = ("realtime", "best") if rep % 2 == 0 else ("best", "realtime")
            for quality in order:
                res["runs"]["%s/%s" % (mode, quality)].append(run_encoder(ctx, src, quality, mode, a.qi, a.target))
    summary = {}
    for k, runs in res["runs"].items():
        assert all(r["frames_sha1"] == runs[0]["frames_sha1"] for r in runs), "%s: repeats emitted different frames" % k
        fps = sorted(r["fps_inter"] for r in runs)
        summary[k] = {"fps_inter": [round(x, 3) for x in fps], "frames_sha1": runs[0]["frames_sha1"], "qi": runs[0]["qi"],
                      "inter_frame_phases_ms": runs[0]["inter_frame_phases_ms"]}
    res["summary"] = summary
    res["reencode_best"] = reencode_rates(ctx, src, a.qi, a.repeats)
    res["reference_best"] = reference_best(src[:2], a.qi, summary["quantizer/best"]["frames_sha1"][:2])
    res["card_after"] = card()
    ctx.close()
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")
    print(json.dumps({k: (v["fps_inter"], v["qi"][-1]) for k, v in summary.items()}))
    print(json.dumps({"reencode_best": {k: v for k, v in res["reencode_best"].items() if k != "frames_sha1"},
                      "reference_best": res["reference_best"], "card": res["card"]}))


if __name__ == "__main__":
    main()
