"""Degraded read with a loss pattern per chunk: the masked call against what a caller does without it.

Arms, per workload (CUDA events around each arm, warm-up, median of --reps repetitions):
  (a) Engine.recover_chunks_masked_dev on the whole batch;
  (b) the same chunks grouped by pattern, one lzgpu_recover_chunks_dev call per group on one stream, in sequence (the batch is laid out
      pattern by pattern, so every group is one run of chunks and needs no copy);
  (c) workload 4 only: one lzgpu_recover_chunks_dev call (the batch has one pattern).
Every timed output of (a) is compared byte for byte with (b).  Workloads:
  1  ec(8,2), 64 MiB chunks, 90 chunks: every two-loss pattern twice
  2  ec(8,2), 64 MiB chunks, 64 chunks over the 10 single-loss patterns
  3  ec(5,3), 64 MiB chunks, 93 chunks: every pattern of up to three lost parts
  4  ec(8,2), 64 MiB chunks, 90 chunks, parts 1 and 4 lost in every chunk
  5  ec(8,2), 1 MiB chunks, 1024 per call over the 55 one- and two-loss patterns
The lost data parts are requested (a degraded read) and the stored CRCs are verified; no image.  Inputs are 3-7 GB per workload,
well past the 126 MB L2.  Writes one JSON document to --out."""
import argparse
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lizardfs_b200 as L  # noqa: E402

BLOCK = 65536


def bits(idx):
    return sum(1 << int(i) for i in idx)


def workloads():
    p82 = [c for r in (1, 2) for c in itertools.combinations(range(10), r)]
    pairs = list(itertools.combinations(range(10), 2))
    return [
        ("1: ec(8,2) 64 MiB, every two-loss pattern twice", "ec(8,2)", 1024, pairs * 2),
        ("2: ec(8,2) 64 MiB, 64 chunks over the single-loss patterns", "ec(8,2)", 1024, [(i % 10,) for i in range(64)]),
        ("3: ec(5,3) 64 MiB, every pattern of up to three lost", "ec(5,3)", 1024,
         [c for r in (0, 1, 2, 3) for c in itertools.combinations(range(8), r)]),
        ("4: ec(8,2) 64 MiB, uniform (parts 1 and 4 lost)", "ec(8,2)", 1024, [(1, 4)] * 90),
        ("5: ec(8,2) 1 MiB, 1024 chunks over the one- and two-loss patterns", "ec(8,2)", 16, [p82[i % len(p82)] for i in range(1024)]),
    ]


def gpu_facts():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, plim, sm, smmax = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": plim, "sm_clock": sm, "sm_clock_max": smmax}
    except Exception as e:   # reported, not fatal: the timings stand on the CUDA events
        return {"gpu": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", required=True, help="path of the JSON document (outside the source tree when that is read-only)")
    ap.add_argument("--only", type=int, nargs="*", help="workload numbers")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("recover_masked_bench: no CUDA device (this measurement has no CPU fallback)")
    dev = torch.device("cuda", 0)
    eng = L.Engine()
    # one explicit stream for the inputs built with torch, the arms and the events (the default stream's handle is 0, which the library
    # reads as "the context's own stream": that one is not ordered with torch's work)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    stream = side.cuda_stream
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    else:
        peak, peak_src = 7700.0, "HGX B200 data sheet, 7.7 TB/s per GPU (not measured)"
    doc = {"facts_before": gpu_facts(), "peak_gbs": peak, "peak_source": peak_src, "reps": args.reps, "workloads": []}
    for wi, (name, text, nb, losses) in enumerate(workloads(), 1):
        if args.only and wi not in args.only:
            continue
        goal = L.SliceType(text)
        k, m = goal.k, goal.m
        N, n = k + m, len(losses)
        pb = (nb + k - 1) // k
        plen = pb * BLOCK
        losses = sorted(losses)              # pattern by pattern: every group of arm (b) is one run of chunks
        masks = [(bits(set(range(N)) - set(lost)), bits([i for i in lost if i < k])) for lost in losses]
        # inputs: seeded chunks, parts and CRCs from the library's own encoder
        data = torch.empty(n * nb * BLOCK, dtype=torch.uint8, device=dev)
        eng.fill_chunks_dev(data.data_ptr(), n, nb * BLOCK, nb * BLOCK, 1000 + wi)
        parts = [torch.empty(n * plen, dtype=torch.uint8, device=dev) for _ in range(N)]
        eng.split_chunks_dev(goal, n, nb, data.data_ptr(), nb * BLOCK, [parts[j].data_ptr() for j in range(k)], plen)
        par = torch.empty(n * m * plen, dtype=torch.uint8, device=dev)
        n_crc = nb + m * pb
        crc = torch.empty(n * n_crc, dtype=torch.int32, device=dev)
        eng.encode_chunks_dev(goal, n, nb * BLOCK, data.data_ptr(), nb * BLOCK, par.data_ptr(), m * plen, crc.data_ptr(), n_crc)
        eng.sync()
        del data
        par = par.view(n, m, plen)
        crc = crc.view(n, n_crc)
        crcs = []
        dcrc = torch.full((n, pb * k), -0x28687115, dtype=torch.int32, device=dev)
        dcrc[:, :nb] = crc[:, :nb]
        dcrc = dcrc.view(n, pb, k)
        for i in range(N):
            if i >= k:
                parts[i].view(n, plen)[:] = par[:, i - k]
                crcs.append(crc[:, nb + (i - k) * pb: nb + (i - k + 1) * pb].contiguous())
            else:
                crcs.append(dcrc[:, :, i].contiguous())
        del par, crc, dcrc
        outs_a = [torch.zeros(n * plen, dtype=torch.uint8, device=dev) for _ in range(N)]
        outs_b = [torch.zeros(n * plen, dtype=torch.uint8, device=dev) for _ in range(N)]
        d_parts = [p.data_ptr() for p in parts]
        d_crcs = [c.data_ptr() for c in crcs]
        mk_arr = L.Engine.chunk_masks(masks)   # the lzgpu_chunk_mask array, built once outside the timed window
        groups = {}
        for c, mk in enumerate(masks):
            groups.setdefault(mk, []).append(c)

        def arm_a():
            eng.recover_chunks_masked_dev(goal, n, nb, mk_arr, d_parts, plen, d_crcs, [o.data_ptr() for o in outs_a], stream=stream)

        def arm_b():
            for (a, w), cs in groups.items():
                want = [1 if w >> i & 1 else 0 for i in range(N)]
                runs = []
                for c in cs:
                    if runs and runs[-1][1] == c:
                        runs[-1][1] = c + 1
                    else:
                        runs.append([c, c + 1])
                for c0, c1 in runs:
                    eng.recover_chunks_dev(goal, c1 - c0, nb, [d_parts[i] + c0 * plen if a >> i & 1 else 0 for i in range(N)], plen,
                                           [d_crcs[i] + c0 * pb * 4 for i in range(N)], want, [o.data_ptr() + c0 * plen for o in outs_b],
                                           stream=stream)

        def arm_c():
            a, w = masks[0]
            eng.recover_chunks_dev(goal, n, nb, [d_parts[i] if a >> i & 1 else 0 for i in range(N)], plen, d_crcs,
                                   [1 if w >> i & 1 else 0 for i in range(N)], [o.data_ptr() for o in outs_b], stream=stream)

        arms = {"a_masked": arm_a, "b_grouped": arm_b}
        if len(groups) == 1:
            arms["c_single_call"] = arm_c
        # outputs: (a) against (b) on every byte the chunks rebuild
        arm_a()
        arm_b()
        torch.cuda.synchronize()
        for i in range(N):
            ov_a, ov_b = outs_a[i].view(n, plen), outs_b[i].view(n, plen)
            for c, (a, w) in enumerate(masks):
                if not a >> i & 1 and w >> i & 1:
                    assert torch.equal(ov_a[c], ov_b[c]), (name, "chunk", c, "part", i)
        times = {}
        order = list(arms)
        samples = {a: [] for a in order}
        for a in order:
            for _ in range(args.warmup):
                arms[a]()
        torch.cuda.synchronize()
        for r in range(args.reps):
            for a in (order if r % 2 == 0 else order[::-1]):       # alternate the arms
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                arms[a]()
                e1.record()
                torch.cuda.synchronize()
                samples[a].append(e0.elapsed_time(e1))
        pl = L.Engine.plan_recover_masked(goal, nb, masks, True, False, plen)
        alg = sum(k * pb * BLOCK + 4 * k * pb + bin(int(w) & ~int(a) & ((1 << N) - 1)).count("1") * pb * BLOCK for a, w in masks)
        for a in order:
            med = float(np.median(samples[a]))
            times[a] = {"median_ms": med, "min_ms": float(np.min(samples[a])), "max_ms": float(np.max(samples[a])),
                        "alg_gbs": alg / med / 1e6, "of_peak": alg / med / 1e6 / peak}
        doc["workloads"].append({"name": name, "goal": text, "nb": nb, "chunks": n, "patterns": len(groups),
                                 "plan": {f: pl[f] for f in ("delegated", "rebuild_launches", "e_chunks", "fallback_groups")},
                                 "alg_bytes": alg, "arms": times,
                                 "a_over_b": times["b_grouped"]["median_ms"] / times["a_masked"]["median_ms"]})
        print(json.dumps(doc["workloads"][-1]), flush=True)
        del parts, crcs, outs_a, outs_b
        torch.cuda.empty_cache()
    doc["facts_after"] = gpu_facts()
    doc["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
