#!/usr/bin/env python
"""bench.py — headline benchmark of the erasure-coding + CRC engine (contract: task brief ④).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; no data-path collective — chunks are independent,
   tiles are dealt round-robin, NCCL is used only for the barrier / max-over-ranks of the timing.)

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): ec(8,2) parity encode +
CRC32 of every 64 KiB data and parity block over 64 MiB chunks.  The 4096-chunk batch (256 GiB) does not
fit one B200, so a *step* is one pass of the hot path over one HBM-resident tile of --tile-chunks chunks
per GPU (default 512 = 32 GiB in, 8 GiB parity out); 8 steps on 1 GPU == the 4096-chunk batch.

One JSON line on stdout (rank 0).  `value` = chunk-data GiB/s with inputs resident in HBM; `e2e` = the
same metric through the host-buffer C-ABI call (pinned host memory, H2D + kernel + D2H inside the timed
region); `roofline` = algorithmic bytes / measured duration against the measured HBM peak;
`cpu_baseline` = the reference CPU implementation timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 65536
CHUNK = 64 << 20
GIB = float(1 << 30)
METRIC = "GiB/s encoded+CRC (ec(8,2), 64 MiB chunks)"


class stdout_to_stderr:
    """NCCL prints its version banner on fd 1 when the first communicator is created; the contract is ONE JSON line
    on stdout, so fd 1 is pointed at fd 2 while torch.distributed initialises."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--goal", default="ec(8,2)")
    ap.add_argument("--tile-chunks", type=int, default=512)
    ap.add_argument("--e2e-chunks", type=int, default=64, help="chunks per host-buffer call in the e2e leg (configs are quoted on >= 64)")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configurations (extra[])")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--pool-gpus", type=int, default=0, help="ONE process, N GPUs through lzgpu_pool: prints the e2e rate of the host-buffer call (not the contract line)")
    ap.add_argument("--cpu-chunks", type=int, default=0, help="chunks in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (rank 0): every block "
                                                          "CRC and a fixed, seeded sample of the parity bytes, to compare two builds output for output")
    return ap.parse_args()


DUMP_PARITY_SAMPLES = 1 << 23


def dump_outputs(torch, out_dir, d_par, d_crc):
    """The headline step's results as float arrays: crc.npy holds every block CRC of the tile (float64, exact for uint32) in the
    layout encode_chunks_dev writes, parity_sample.npy the parity bytes (float32) at DUMP_PARITY_SAMPLES positions drawn with a
    fixed seed (the whole parity output of a tile is gigabytes).  The inputs come from a fixed seed as well, so two runs with
    the same arguments dump the same arrays."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(2024).integers(0, d_par.numel(), size=DUMP_PARITY_SAMPLES, dtype=np.int64))
    sample = d_par[torch.from_numpy(idx).to(d_par.device)].cpu().numpy()
    np.save(os.path.join(out_dir, "parity_sample.npy"), sample.astype(np.float32))
    np.save(os.path.join(out_dir, "crc.npy"), d_crc.cpu().numpy().view(np.uint32).astype(np.float64))


def algorithmic_bytes_per_chunk(k, m, chunk_len=CHUNK):
    """SURVEY.md §8(d): read S + write m*pb*B + write 4*(nb + m*pb)."""
    nb = (chunk_len + BLOCK - 1) // BLOCK
    pb = (nb + k - 1) // k
    return chunk_len + m * pb * BLOCK + 4 * (nb + m * pb)


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi, during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device_index):
        self.dev = device_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in the timed region"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w": float(np.median(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm
# ------------------------------------------------------------------------------------------------
class Goal:
    """goal text -> kind / k / m without touching the product package (the reference arm must not load liblzgpu.so):
    xorN = kind 0 (N data + 1 parity), ec(k,m) = kind 1 (goal_config_loader.cc:228-245)"""

    def __init__(self, text):
        import re
        t = text.strip().lstrip("$")
        mx = re.fullmatch(r"xor([2-9])", t)
        me = re.fullmatch(r"ec\((\d+),(\d+)\)", t)
        if mx:
            self.kind, self.k, self.m = 0, int(mx.group(1)), 1
        elif me and 2 <= int(me.group(1)) <= 32 and 1 <= int(me.group(2)) <= 32:
            self.kind, self.k, self.m = 1, int(me.group(1)), int(me.group(2))
        else:
            raise ValueError(f"bad goal {text!r}")
        self.text = t

    def __str__(self):
        return self.text


def cpu_reference_run(goal_text, n_chunks, threads, reps=1):
    """Times the reference CPU implementation (oracle/_ref when present, else the oracle port) on
    `n_chunks` synthetic 64 MiB chunks using `threads` host threads (chunk-level parallelism; ctypes
    releases the GIL).  Uses the reference CALL PATTERN (per stripe, per parity part rs.recover +
    mycrc32 per block: chunk_writer.cc:365-401, write_executor.cc:97).  Returns (GiB/s, kind, seconds)."""
    from concurrent.futures import ThreadPoolExecutor

    import ctypes as C

    from tests import _oracle as O

    g = Goal(goal_text)
    oracle = O.load_oracle()
    ref = O.load_ref()
    lib, kind = (ref, "reference") if ref is not None else (oracle, "port")
    nb = CHUNK // BLOCK
    pb = (nb + g.k - 1) // g.k
    n_buf = min(n_chunks, max(threads, 1))
    chunks = [O.fill_chunk(oracle, CHUNK, 12345, c) for c in range(n_buf)]
    par = [np.zeros(g.m * pb * BLOCK, dtype=np.uint8) for _ in range(n_buf)]
    crc = [np.zeros(nb + g.m * pb, dtype=np.uint32) for _ in range(n_buf)]
    fn = lib.fn("encode_chunk")

    def one(i):
        b = i % n_buf
        rc = fn(g.kind, g.k, g.m, chunks[b].ctypes.data_as(C.c_void_p), C.c_size_t(CHUNK), par[b].ctypes.data_as(C.c_void_p),
                crc[b].ctypes.data_as(C.c_void_p))
        assert rc == 0
    one(0)  # warm-up (tables, page faults)
    best = None
    with ThreadPoolExecutor(max_workers=threads) as ex:
        for _ in range(reps):
            t0 = time.perf_counter()
            list(ex.map(one, range(n_chunks)))
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return n_chunks * CHUNK / GIB / best, kind, best


def cpu_reference_best_case(goal_text, n_chunks, threads):
    """SURVEY.md §8d(ii) "best-case reference kernel": ONE rs.encode over whole part-major parts
    (reed_solomon.h:134-155) + mycrc32 per block, parts prepared outside the timed region.  Only with oracle/_ref."""
    from concurrent.futures import ThreadPoolExecutor

    import ctypes as C

    from tests import _oracle as O

    ref = O.load_ref()
    if ref is None:
        return None
    g = Goal(goal_text)
    oracle = O.load_oracle()
    nb = CHUNK // BLOCK
    pb = (nb + g.k - 1) // g.k
    n_buf = min(n_chunks, max(threads, 1))
    bufs = []
    for c in range(n_buf):
        parts, _ = O.split_parts(O.fill_chunk(oracle, CHUNK, 12345, c), g.k)
        parts = [np.ascontiguousarray(p) for p in parts]
        bufs.append((parts, O.ptr_array(parts), np.zeros(g.m * pb * BLOCK, dtype=np.uint8), np.zeros((g.k + g.m) * pb, dtype=np.uint32)))
    fn = ref.fn("encode_parts")

    def one(i):
        parts, ptrs, par, crc = bufs[i % n_buf]
        assert fn(g.kind, g.k, g.m, ptrs, C.c_uint32(pb), par.ctypes.data_as(C.c_void_p), crc.ctypes.data_as(C.c_void_p)) == 0
    one(0)
    with ThreadPoolExecutor(max_workers=threads) as ex:
        t0 = time.perf_counter()
        list(ex.map(one, range(n_chunks)))
        dt = time.perf_counter() - t0
    return n_chunks * CHUNK / GIB / dt


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_threads()
    n_chunks = args.cpu_chunks or max(cores, 8)
    # one "step" = a bounded sample of n_chunks chunks; warm-up steps are real runs as well
    for _ in range(min(args.warmup, 1)):
        cpu_reference_run(args.goal, min(n_chunks, cores), cores)
    vals, secs, kind = [], 0.0, "port"
    for _ in range(args.steps):
        v, kind, dt = cpu_reference_run(args.goal, n_chunks, cores)
        vals.append(v); secs += dt
    value = float(np.mean(vals))
    g = Goal(args.goal)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * secs / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{g} encode + per-64KiB-block CRC32, 64 MiB chunks, reference CPU call pattern "
                               f"(ChunkWriter::computeParityBlock per stripe/parity + mycrc32 per block)",
                   "chunks_per_step": n_chunks, "host_threads": cores},
        "cpu_baseline": {"value": value, "unit": "GiB/s", "cores": cores, "kind": kind,
                         "sample": f"{n_chunks} x 64 MiB chunks per step, {args.steps} steps"},
        "e2e": {"value": value, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def _ref_lib():
    """the checker for the in-run parity spot checks: the compiled reference when present, else the oracle restatement"""
    from tests import _oracle as O
    ref = O.load_ref()
    return (ref, "oracle/_ref (the reference compiled from its sources)") if ref is not None else (O.load_oracle(), "oracle port")


class Extras:
    """The other BASELINE.json configurations, measured in the same run as the headline and checked against the reference at the
    size that is timed:  configs[1] ec(3,2) encode,  configs[3] ec(8,2) degraded read with data parts 1 and 4 lost (stored CRCs
    verified, rebuilt parts + chunk image written),  configs[4] xor2 / xor3 / ec(5,3) / ec(8,4) x {1, 4, 16, 64, 37.31 MiB} chunks.
    Every entry: algorithmic bytes (DESIGN.md §4), ms per launch, GiB/s of chunk data summed over the ranks, fraction of the
    measured HBM peak, and the number of chunks of the timed buffers compared bit for bit with the reference afterwards."""

    def __init__(self, torch, L, eng, dev, stream, d_data, tile_bytes, peak, world, dist, rank, steps, warmup):
        self.torch, self.L, self.eng, self.dev, self.stream = torch, L, eng, dev, stream
        self.sp = stream.cuda_stream
        self.d_data, self.tile_bytes, self.peak = d_data, tile_bytes, peak
        self.world, self.dist, self.rank = world, dist, rank
        self.steps, self.warmup = steps, max(warmup, 3)
        self.checker, self.checker_name = _ref_lib()
        self.out = []
        self.launches = 0

    def _time(self, fn):
        torch = self.torch
        for _ in range(self.warmup):
            fn()
        torch.cuda.synchronize(self.dev)
        if self.dist:
            self.dist.barrier()
        l0 = self.eng.stats()["kernel_launches"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(self.steps):
            fn()
        e1.record(self.stream)
        torch.cuda.synchronize(self.dev)
        self.launches += self.eng.stats()["kernel_launches"] - l0
        ms = e0.elapsed_time(e1) / self.steps
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def _entry(self, name, config, n, clen, alg_bytes, ms, checked, what):
        gibs = self.world * n * clen / GIB / (ms / 1e3)
        gbs = n * alg_bytes / (ms / 1e3) / 1e9   # per GPU: the roofline is a per-device quantity
        self.out.append({"name": name, "config": config, "chunks_per_launch_per_gpu": n, "chunk_bytes": clen, "ms": ms,
                         "value": gibs, "unit": "GiB/s of chunk data, all ranks", "algorithmic_bytes_per_launch": n * alg_bytes,
                         "achieved_gbs_per_gpu": gbs, "frac_of_measured_hbm": gbs / self.peak,
                         "parity": f"{checked} chunk(s) of the timed buffers bit-exact vs {self.checker_name}: {what}"})

    def encode(self, goal_text, clen, config, max_chunks=512, n_check=4):
        torch, L, eng = self.torch, self.L, self.eng
        g = L.SliceType(goal_text)
        k, m = g.k, g.m
        nb = (clen + BLOCK - 1) // BLOCK
        pb = (nb + k - 1) // k
        stride = nb * BLOCK
        n = min(self.tile_bytes // stride, max_chunks)
        par_stride, crc_stride = m * pb * BLOCK, nb + m * pb
        d_par = torch.empty(n * par_stride, dtype=torch.uint8, device=self.dev)
        d_crc = torch.empty(n * crc_stride, dtype=torch.int32, device=self.dev)
        ms = self._time(lambda: eng.encode_chunks_dev(g, n, clen, self.d_data.data_ptr(), stride, d_par.data_ptr(), par_stride,
                                                      d_crc.data_ptr(), crc_stride, stream=self.sp))
        # parity + CRC of chunks spread over the timed batch against the reference, outside the timed region
        rng = np.random.default_rng(1234 + self.rank)
        picks = sorted(set([0, n - 1] + [int(x) for x in rng.integers(0, n, size=max(0, n_check - 2))]))[:n_check]
        for c in picks:
            chunk = self.d_data[c * stride: c * stride + clen].cpu().numpy()
            p_ref, c_ref = self.checker.encode_chunk(g.kind, k, m, chunk)
            p_got = d_par[c * par_stride: (c + 1) * par_stride].cpu().numpy().reshape(m, pb * BLOCK)
            c_got = d_crc[c * crc_stride: (c + 1) * crc_stride].cpu().numpy().view(np.uint32)
            assert (p_got == p_ref).all(), f"bench parity check failed: {goal_text} {clen} chunk {c}: parity differs from the reference"
            assert (c_got == c_ref).all(), f"bench parity check failed: {goal_text} {clen} chunk {c}: CRCs differ from the reference"
        self._entry(f"encode {goal_text} {clen / (1 << 20):.2f} MiB", config, n, clen, algorithmic_bytes_per_chunk(k, m, clen), ms,
                    len(picks), "parity parts and every block CRC")
        del d_par, d_crc

    def recover(self, goal_text, lost, config, n=128, n_check=2):
        """degraded read of `n` 64 MiB chunks: part-major inputs are built from the resident data (split + encode, untimed)"""
        torch, L, eng = self.torch, self.L, self.eng
        g = L.SliceType(goal_text)
        k, m = g.k, g.m
        clen, nb = CHUNK, CHUNK // BLOCK
        pb = (nb + k - 1) // k
        ps = pb * BLOCK
        d_par = torch.empty(n * m * ps, dtype=torch.uint8, device=self.dev)
        d_crc = torch.empty(n * (nb + m * pb), dtype=torch.int32, device=self.dev)
        eng.encode_chunks_dev(g, n, clen, self.d_data.data_ptr(), clen, d_par.data_ptr(), m * ps, d_crc.data_ptr(), nb + m * pb, stream=self.sp)
        parts = [torch.zeros(n * ps, dtype=torch.uint8, device=self.dev) for _ in range(k)]
        eng.split_chunks_dev(g, n, nb, self.d_data.data_ptr(), clen, [p.data_ptr() for p in parts], ps, stream=self.sp)
        torch.cuda.synchronize(self.dev)
        crc_all = d_crc.view(n, nb + m * pb)
        pcrc = []
        for j in range(k):
            cj = torch.full((n, pb), -0x28687115, dtype=torch.int32, device=self.dev)  # 0xD7978EEB: zero padding blocks
            sub = crc_all[:, j:nb:k]
            cj[:, : sub.shape[1]] = sub
            pcrc.append(cj.contiguous())
        for r in range(m):
            parts.append(d_par.view(n, m, ps)[:, r].contiguous().view(-1))
            pcrc.append(crc_all[:, nb + r * pb: nb + (r + 1) * pb].contiguous())
        outs = [torch.empty(n * ps, dtype=torch.uint8, device=self.dev) if i in lost else None for i in range(k + m)]
        img = torch.empty(n * clen, dtype=torch.uint8, device=self.dev)
        dp = [0 if i in lost else parts[i].data_ptr() for i in range(k + m)]
        dc = [0 if i in lost else pcrc[i].data_ptr() for i in range(k + m)]
        do = [outs[i].data_ptr() if i in lost else 0 for i in range(k + m)]
        want = [1 if i in lost else 0 for i in range(k + m)]
        # back-to-back launches: the verdict of every verifying call is collected by eng.sync() (deferred verification), which
        # raises on a CRC mismatch
        eng.set_deferred_verify(True)
        ms = self._time(lambda: eng.recover_chunks_dev(g, n, nb, dp, ps, dc, want, do, img.data_ptr(), clen, stream=self.sp))
        eng.sync()
        eng.set_deferred_verify(False)
        # exact on the device for the whole batch (rebuilt parts == the parts that were withheld, image == the chunks) ...
        for i in lost:
            assert torch.equal(outs[i], parts[i]), f"bench parity check failed: recover {goal_text} part {i}"
        assert torch.equal(img, self.d_data[: n * clen]), "bench parity check failed: chunk image"
        # ... and against the reference's own recover for a few chunks
        for c in sorted({0, n - 1})[:n_check]:
            hp = [None if i in lost else parts[i][c * ps: (c + 1) * ps].cpu().numpy() for i in range(k + m)]
            rc, ro, _ = self.checker.recover_chunk(g.kind, k, m, hp, None, want, pb)
            assert rc == 0
            for i in lost:
                assert (ro[i] == outs[i][c * ps: (c + 1) * ps].cpu().numpy()).all(), f"bench parity check failed: recover {goal_text} chunk {c} part {i} vs reference"
        e = len(lost)
        alg = k * ps + 4 * k * pb + e * ps + nb * BLOCK   # read k parts + their stored CRCs, write e parts + the image
        self._entry(f"recover {goal_text} parts {sorted(lost)} lost (verify + rebuild + image)", config, n, clen, alg, ms, n,
                    f"rebuilt parts and image identical on the device for all {n} chunks; {min(n_check, 2)} chunk(s) also vs the reference's recover")
        del parts, pcrc, outs, img, d_par, d_crc


    def convert(self, src_text, lost, dst_text, config, n=64, n_check=2):
        """slice-type conversion for replication (SURVEY.md 8(f1), SliceRecoveryPlanner): `n` 64 MiB chunks of slice type `src` with the
        `lost` parts missing -> every part of slice type `dst` + its block CRCs, source CRCs verified"""
        torch, L, eng = self.torch, self.L, self.eng
        gs, gd = L.SliceType(src_text), L.SliceType(dst_text)
        clen, nb = CHUNK, CHUNK // BLOCK

        def slice_of(g):
            k, m = g.k, g.m
            pb = (nb + k - 1) // k
            ps = pb * BLOCK
            d_par = torch.empty(n * m * ps, dtype=torch.uint8, device=self.dev)
            d_crc = torch.empty(n * (nb + m * pb), dtype=torch.int32, device=self.dev)
            eng.encode_chunks_dev(g, n, clen, self.d_data.data_ptr(), clen, d_par.data_ptr(), m * ps, d_crc.data_ptr(), nb + m * pb, stream=self.sp)
            parts = [torch.zeros(n * ps, dtype=torch.uint8, device=self.dev) for _ in range(k)]
            eng.split_chunks_dev(g, n, nb, self.d_data.data_ptr(), clen, [p.data_ptr() for p in parts], ps, stream=self.sp)
            torch.cuda.synchronize(self.dev)
            crc_all = d_crc.view(n, nb + m * pb)
            pcrc = []
            for j in range(k):
                cj = torch.full((n, pb), -0x28687115, dtype=torch.int32, device=self.dev)  # 0xD7978EEB: zero padding blocks
                sub = crc_all[:, j:nb:k]
                cj[:, : sub.shape[1]] = sub
                pcrc.append(cj.contiguous())
            for r in range(m):
                parts.append(d_par.view(n, m, ps)[:, r].contiguous().view(-1))
                pcrc.append(crc_all[:, nb + r * pb: nb + (r + 1) * pb].contiguous())
            return parts, pcrc, pb, ps

        sparts, scrc, pbs, pss = slice_of(gs)
        ns, nd = gs.k + gs.m, gd.k + gd.m
        pbd = (nb + gd.k - 1) // gd.k
        psd = pbd * BLOCK
        outs = [torch.empty(n * psd, dtype=torch.uint8, device=self.dev) for _ in range(nd)]
        ocrc = [torch.empty((n, pbd), dtype=torch.int32, device=self.dev) for _ in range(nd)]
        dp = [0 if i in lost else sparts[i].data_ptr() for i in range(ns)]
        dc = [0 if i in lost else scrc[i].data_ptr() for i in range(ns)]
        eng.set_deferred_verify(True)
        ms = self._time(lambda: eng.convert_chunks_dev(gs, gd, n, nb, dp, pss, [1] * nd, [o.data_ptr() for o in outs], psd, d_part_crc=dc,
                                                       d_out_crc=[o.data_ptr() for o in ocrc], stream=self.sp))
        eng.sync()
        eng.set_deferred_verify(False)
        plan = L.Engine.plan_convert(gs, gd, [0 if i in lost else 1 for i in range(ns)], [1] * nd)
        del sparts, scrc
        # exact on the device for the whole batch: every destination part and CRC equals a direct encode / split of the same chunks ...
        dparts, dcrc, _, _ = slice_of(gd)
        for i in range(nd):
            assert torch.equal(outs[i], dparts[i]), f"bench parity check failed: convert {src_text} -> {dst_text} part {i}"
            nreal = gd.part_blocks(i, nb)
            assert torch.equal(ocrc[i][:, :nreal], dcrc[i][:, :nreal]), f"bench parity check failed: convert {src_text} -> {dst_text} CRCs of part {i}"
        # ... and the parity parts against the reference's own encoder for a few chunks
        for c in sorted({0, n - 1})[:n_check]:
            chunk = self.d_data[c * clen: (c + 1) * clen].cpu().numpy()
            p_ref, c_ref = self.checker.encode_chunk(gd.kind, gd.k, gd.m, chunk)
            for r in range(gd.m):
                assert (outs[gd.k + r][c * psd: (c + 1) * psd].cpu().numpy() == p_ref[r]).all(), f"bench parity check failed: convert parity {r} chunk {c} vs reference"
                assert (ocrc[gd.k + r][c].cpu().numpy().view(np.uint32) == c_ref[nb + r * pbd: nb + (r + 1) * pbd]).all()
        # algorithmic bytes (DESIGN.md 4.5): the k source parts that are read + their stored CRCs, every destination part + its CRCs, once
        alg = gs.k * pbs * (BLOCK + 4) + nd * pbd * (BLOCK + 4)
        self._entry(f"convert {src_text} parts {sorted(lost)} lost -> {dst_text} (verify + all parts + CRCs)", config, n, clen, alg, ms, n,
                    f"all destination parts and CRCs identical on the device to a direct encode / split for all {n} chunks; parity parts of "
                    f"{min(n_check, 2)} chunk(s) also vs the reference's encoder; route: {'one pass' if plan['one_pass'] else 'two passes'}")
        del outs, ocrc, dparts, dcrc


def copy_roofline(torch, dev, in_bytes, out_bytes, dist, reps=3):
    """e2e ceiling of this host/GPU pair: pinned H2D of `in_bytes` and D2H of `out_bytes` issued together on two streams (what the
    3-slot pipeline overlaps), all ranks at once.  Returns seconds (max over ranks) for one such exchange."""
    h_in = torch.empty(in_bytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(in_bytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    best = None
    for i in range(reps + 1):
        torch.cuda.synchronize(dev)
        if dist:
            dist.barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if i:  # first pass warms the page tables
            best = float(t.item()) if best is None else min(best, float(t.item()))
    return best


def run_pool(args):
    """Single-process multi-GPU: lzgpu_pool_encode_chunks over N devices from pinned host buffers (the in-process form the mount and
    the chunkserver need; SURVEY.md §7.3b).  Same workload and timing rule as the e2e leg of the torchrun arm."""
    import ctypes as C

    import torch

    import lizardfs_b200 as L
    n_dev = args.pool_gpus
    pool = L.Pool(list(range(n_dev)))
    goal = L.SliceType(args.goal)
    k, m = goal.k, goal.m
    nb = CHUNK // BLOCK
    pb = (nb + k - 1) // k
    E = args.e2e_chunks * n_dev
    par_stride, crc_stride = m * pb * BLOCK, nb + m * pb
    # One contiguous caller buffer per array, as the C ABI wants; each device's share of it is first-touched from a thread bound
    # to the CPUs local to that GPU (so its pages live on that GPU's NUMA node, what a torchrun rank gets for free), then the
    # whole buffer is page-locked in place with lzgpu_host_register.
    import threading
    h_in = torch.empty(E * CHUNK, dtype=torch.uint8)
    h_par = torch.empty(E * par_stride, dtype=torch.uint8)
    h_crc = torch.empty(E * crc_stride, dtype=torch.int32)
    eng = L.Engine(0)
    one = torch.empty(args.e2e_chunks * CHUNK, dtype=torch.uint8, device="cuda:0")
    eng.fill_chunks_dev(one.data_ptr(), args.e2e_chunks, CHUNK, CHUNK, seed=12345)
    torch.cuda.synchronize()
    one_h = one.cpu()
    del one
    placement = []

    def touch(d):
        note = "unbound"
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(d))   # affinity of THIS thread (Linux: per thread)
            note = f"{len(os.sched_getaffinity(0))} local CPUs"
        except Exception as exc:
            note = f"unbound ({type(exc).__name__})"
        n = args.e2e_chunks
        h_in[d * n * CHUNK:(d + 1) * n * CHUNK].copy_(one_h)            # first touch = placement
        h_par[d * n * par_stride:(d + 1) * n * par_stride].zero_()
        h_crc[d * n * crc_stride:(d + 1) * n * crc_stride].zero_()
        placement.append((d, note))
    ths = [threading.Thread(target=touch, args=(d,)) for d in range(n_dev)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    for t_ in (h_in, h_par, h_crc):
        rc = eng.lib.lzgpu_host_register(eng.h, t_.data_ptr(), t_.numel() * t_.element_size())
        assert rc == 0, L._lib.last_error()
    eng.close()
    lib = pool.lib
    a_in, a_par, a_crc = h_in.data_ptr(), h_par.data_ptr(), h_crc.data_ptr()

    def step():
        rc = lib.lzgpu_pool_encode_chunks(pool.h, C.byref(goal.c), E, CHUNK, a_in, CHUNK, a_par, par_stride, a_crc, crc_stride)
        assert rc == 0, L._lib.last_error()
    for _ in range(2):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    crc = h_crc.numpy().view(np.uint32).reshape(E, crc_stride)
    assert (crc[0] == crc[args.e2e_chunks]).all() if n_dev > 1 else True   # same chunks on device 0 and 1 -> same CRCs
    st = pool.stats()
    print(json.dumps({"mode": "single-process pool", "n_gpus": n_dev, "e2e_value": E * args.steps * CHUNK / GIB / dt, "unit": "GiB/s of chunk data",
                      "chunks_per_call": E, "steps": args.steps, "h2d_bytes_per_step": E * CHUNK, "d2h_bytes_per_step": E * (par_stride + 4 * crc_stride),
                      "kernel_launches": st["kernel_launches"], "device_gbps_mean_per_batch": st["batch_gbps_mean"],
                      "host_placement": sorted(placement)}), flush=True)
    pool.close()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.pool_gpus:
        run_pool(args)
        return

    import torch

    import lizardfs_b200 as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # Host buffers of the e2e leg should live on the NUMA node next to this rank's GPU: bind the process to the GPU's
    # ideal CPUs before anything is allocated (restored before the CPU baseline, which must see every core).
    all_cpus = os.sched_getaffinity(0)
    numa_note = "not bound"
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else local
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
        numa_note = f"bound to {len(os.sched_getaffinity(0))} CPUs local to GPU {phys}"
    except Exception as exc:  # no NVML / not permitted: keep the default placement
        numa_note = f"not bound ({type(exc).__name__})"
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
    dev = torch.device("cuda", local)
    eng = L.Engine(local)
    goal = L.SliceType(args.goal)
    k, m = goal.k, goal.m
    nb = CHUNK // BLOCK
    pb = (nb + k - 1) // k
    T = args.tile_chunks
    par_stride = m * pb * BLOCK
    crc_stride = nb + m * pb

    d_data = torch.empty(T * CHUNK, dtype=torch.uint8, device=dev)
    d_par = torch.empty(T * par_stride, dtype=torch.uint8, device=dev)
    d_crc = torch.empty(T * crc_stride, dtype=torch.int32, device=dev)
    # a dedicated non-default stream: handle 0 (torch's legacy default stream) would make the library
    # pick its own stream and the CUDA events below would not bracket the kernels
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0
    eng.fill_chunks_dev(d_data.data_ptr(), T, CHUNK, CHUNK, seed=12345, first_chunk=rank * T, stream=sptr)

    def step():
        eng.encode_chunks_dev(goal, T, CHUNK, d_data.data_ptr(), CHUNK, d_par.data_ptr(), par_stride, d_crc.data_ptr(), crc_stride, stream=sptr)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = eng.stats()["kernel_launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    t_wall0 = time.time()
    ev[0].record(stream)
    for i in range(args.steps):
        step()
        ev[i + 1].record(stream)
    barrier()
    t_wall1 = time.time()
    launches = eng.stats()["kernel_launches"] - launches0
    ms_total = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total_max = float(t.item())
    value = world * T * args.steps * CHUNK / GIB / (ms_total_max / 1e3)
    lib_stats = eng.stats()   # the library's own per-batch device timing of the same launches (lzgpu_stats.batch_*)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, d_par, d_crc)

    # ---- the timed launches' results against the reference: parity parts and CRCs of chunks spread over the resident tile
    checker, checker_name = _ref_lib()
    probing = bool(os.environ.get("LZGPU_PROBE"))
    rng = np.random.default_rng(99 + rank)
    picks = sorted(set([0, T - 1] + [int(x) for x in rng.integers(0, T, size=2)]))
    headline_checked = 0
    if not probing and not args.no_parity_check:
        for c in picks:
            chunk = d_data[c * CHUNK: (c + 1) * CHUNK].cpu().numpy()
            p_ref, c_ref = checker.encode_chunk(goal.kind, k, m, chunk)
            assert (d_par[c * par_stride: (c + 1) * par_stride].cpu().numpy().reshape(m, pb * BLOCK) == p_ref).all(), f"headline parity differs from the reference (chunk {c})"
            assert (d_crc[c * crc_stride: (c + 1) * crc_stride].cpu().numpy().view(np.uint32) == c_ref).all(), f"headline CRCs differ from the reference (chunk {c})"
            headline_checked += 1
    crc_host = d_crc[:crc_stride].cpu().numpy().view(np.uint32)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"

    # ---- the other BASELINE configurations, same run, same buffers
    extra, extra_launches = [], 0
    if not args.no_extra and not probing:
        del d_par, d_crc
        ex = Extras(torch, L, eng, dev, stream, d_data, T * CHUNK, peak, world, dist, rank, steps=5, warmup=3)
        ex.encode("ec(3,2)", CHUNK, "BASELINE.json configs[1]: ec(3,2) encode + CRC, 64 MiB chunks", max_chunks=512)
        ex.recover("ec(8,2)", (1, 4), "BASELINE.json configs[3]: ec(8,2) degraded read, data parts 1 and 4 lost", n=128)
        ex.convert("ec(8,2)", (1, 4), "ec(3,2)", "SURVEY.md 8(f1): slice conversion for replication, ec(8,2) with data parts 1 and 4 lost -> ec(3,2)", n=64)
        for gt in ("xor2", "xor3", "ec(5,3)", "ec(8,4)"):
            for clen in (1 << 20, 4 << 20, 16 << 20, 64 << 20, (37 << 20) + 5 * BLOCK):
                ex.encode(gt, clen, "BASELINE.json configs[4]: mixed-goal sweep", max_chunks=8192, n_check=3 if clen >= (16 << 20) else 4)
        # beyond BASELINE.json: the degraded read with THREE lost data parts (bs_recover_kernel.cuh), same in-run checks; reported as an
        # entry of its own and never allowed to take the line down
        try:
            ex.recover("ec(5,3)", (0, 1, 4), "SURVEY.md 8(a10): ec(5,3) degraded read, data parts 0, 1 and 4 lost", n=64)
        except Exception as exc:  # noqa: BLE001
            ex.out.append({"name": "recover ec(5,3) parts [0, 1, 4] lost (verify + rebuild + image)", "error": f"{type(exc).__name__}: {exc}"[:300]})
        extra, extra_launches = ex.out, ex.launches

    # ---- end-to-end through the host-buffer C-ABI call (pinned memory, copies inside the timed region)
    e2e = None
    if not args.no_e2e:
        E = args.e2e_chunks
        import ctypes as C
        lib = eng.lib
        h_in = torch.empty(E * CHUNK, dtype=torch.uint8).pin_memory()
        h_par = torch.empty(E * par_stride, dtype=torch.uint8).pin_memory()
        h_crc = torch.empty(E * crc_stride, dtype=torch.int32).pin_memory()
        h_in.copy_(d_data[: E * CHUNK])
        np_in, np_par, np_crc = h_in.numpy(), h_par.numpy(), h_crc.numpy().view(np.uint32)

        def e2e_step():
            rc = lib.lzgpu_encode_chunks(eng.h, C.byref(goal.c), E, CHUNK, np_in.ctypes.data_as(C.c_void_p), CHUNK,
                                         np_par.ctypes.data_as(C.c_void_p), par_stride, np_crc.ctypes.data_as(C.c_void_p), crc_stride)
            assert rc == 0, L._lib.last_error()

        def timed(fn, steps):
            for _ in range(2):
                fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if dist:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        dt = timed(e2e_step, args.steps)
        assert (np_crc[:crc_stride] == crc_host).all(), "e2e result differs from the resident run"
        e2e_value = world * E * args.steps * CHUNK / GIB / dt
        # the ceiling of this path on this host: the same bytes as pure pinned copies, both directions at once, all ranks together
        t_copy = copy_roofline(torch, dev, E * CHUNK, E * (par_stride + 4 * crc_stride), dist)
        copy_peak = world * E * CHUNK / GIB / t_copy
        e2e = {"value": e2e_value, "unit": "GiB/s", "h2d_bytes_per_step": E * CHUNK,
               "d2h_bytes_per_step": E * (par_stride + 4 * crc_stride), "chunks_per_step": E,
               "timing": "host wall clock around the synchronous C-ABI call, max over ranks", "host_placement": numa_note,
               "roofline": {"bound": "pcie", "peak": copy_peak, "unit": "GiB/s of chunk data", "frac": e2e_value / copy_peak,
                            "how": f"pinned H2D of {E * CHUNK} B and D2H of {E * (par_stride + 4 * crc_stride)} B issued together on two streams, "
                                   f"all {world} rank(s) at once, best of 3; h2d {world * E * CHUNK / t_copy / 1e9:.1f} GB/s aggregate"}}
        # pageable caller buffers (what a chunkserver has unless it registers its pool): same call, plain numpy memory
        if True:
            Ep = min(E, 8)
            pg_in = np.empty(Ep * CHUNK, dtype=np.uint8)
            pg_in[:] = np_in[: Ep * CHUNK]
            pg_par = np.empty(Ep * par_stride, dtype=np.uint8)
            pg_crc = np.empty(Ep * crc_stride, dtype=np.uint32)

            def pg_step():
                rc = lib.lzgpu_encode_chunks(eng.h, C.byref(goal.c), Ep, CHUNK, pg_in.ctypes.data_as(C.c_void_p), CHUNK,
                                             pg_par.ctypes.data_as(C.c_void_p), par_stride, pg_crc.ctypes.data_as(C.c_void_p), crc_stride)
                assert rc == 0, L._lib.last_error()
            dtp = timed(pg_step, 2)
            e2e["pageable_value"] = world * Ep * 2 * CHUNK / GIB / dtp
            rc = lib.lzgpu_host_register(eng.h, pg_in.ctypes.data_as(C.c_void_p), pg_in.nbytes)
            rc |= lib.lzgpu_host_register(eng.h, pg_par.ctypes.data_as(C.c_void_p), pg_par.nbytes)
            if rc == 0:
                dtr = timed(pg_step, 2)
                e2e["registered_value"] = world * Ep * 2 * CHUNK / GIB / dtr
                lib.lzgpu_host_unregister(eng.h, pg_in.ctypes.data_as(C.c_void_p))
                lib.lzgpu_host_unregister(eng.h, pg_par.ctypes.data_as(C.c_void_p))
            e2e["pageable_note"] = f"{Ep} chunks per call from plain (pageable) numpy buffers, then the same buffers after lzgpu_host_register"
        del h_in, h_par, h_crc
        # degraded read end to end (configs[3] through the host-buffer call): k parts + stored CRCs in, 2 parts + image out
        Er = max(8, min(E, 32))
        ps = pb * BLOCK
        g82 = goal
        parts_h = [torch.empty(Er * ps, dtype=torch.uint8).pin_memory() for _ in range(k + m)]
        crc_h = [torch.empty(Er * pb, dtype=torch.int32).pin_memory() for _ in range(k + m)]
        d_par2 = torch.empty(Er * par_stride, dtype=torch.uint8, device=dev)
        d_crc2 = torch.empty(Er * crc_stride, dtype=torch.int32, device=dev)
        eng.encode_chunks_dev(g82, Er, CHUNK, d_data.data_ptr(), CHUNK, d_par2.data_ptr(), par_stride, d_crc2.data_ptr(), crc_stride, stream=sptr)
        dparts = [torch.zeros(Er * ps, dtype=torch.uint8, device=dev) for _ in range(k)]
        eng.split_chunks_dev(g82, Er, nb, d_data.data_ptr(), CHUNK, [p.data_ptr() for p in dparts], ps, stream=sptr)
        torch.cuda.synchronize(dev)
        ca = d_crc2.view(Er, crc_stride)
        for j in range(k):
            parts_h[j].copy_(dparts[j])
            crc_h[j].view(Er, pb).copy_(ca[:, j:nb:k])
        for r in range(m):
            parts_h[k + r].view(Er, ps).copy_(d_par2.view(Er, m, ps)[:, r])
            crc_h[k + r].view(Er, pb).copy_(ca[:, nb + r * pb: nb + (r + 1) * pb])
        lost = (1, 4) if k > 4 else (0, 1)
        out_h = {i: torch.empty(Er * ps, dtype=torch.uint8).pin_memory() for i in lost}
        img_h = torch.empty(Er * CHUNK, dtype=torch.uint8).pin_memory()
        PP = C.c_void_p * (k + m)
        a_parts = PP(*[None if i in lost else parts_h[i].data_ptr() for i in range(k + m)])
        a_crc = PP(*[None if i in lost else crc_h[i].data_ptr() for i in range(k + m)])
        a_out = PP(*[out_h[i].data_ptr() if i in lost else None for i in range(k + m)])
        want = np.array([1 if i in lost else 0 for i in range(k + m)], dtype=np.uint8)
        bad = (C.c_int64 * 3)(-1, -1, -1)

        def rec_step():
            rc = lib.lzgpu_recover_chunks(eng.h, C.byref(g82.c), Er, nb, a_parts, ps, a_crc, want.ctypes.data_as(C.c_void_p), a_out,
                                          img_h.data_ptr(), CHUNK, bad)
            assert rc == 0, L._lib.last_error()
        dtr = timed(rec_step, max(2, args.steps // 2))
        for i in lost:
            assert torch.equal(out_h[i], dparts[i].cpu()), "e2e recover: rebuilt part differs"
        assert torch.equal(img_h, d_data[: Er * CHUNK].cpu()), "e2e recover: chunk image differs"
        rec_in, rec_out = Er * k * (ps + 4 * pb), Er * (len(lost) * ps + CHUNK)
        t_copy_r = copy_roofline(torch, dev, rec_in, rec_out, dist)
        rec_value = world * Er * max(2, args.steps // 2) * CHUNK / GIB / dtr
        rec_peak = world * Er * CHUNK / GIB / t_copy_r
        e2e["recover"] = {"value": rec_value, "unit": "GiB/s of chunk data", "config": f"{g82} degraded read, parts {list(lost)} lost, stored CRCs verified, "
                          f"rebuilt parts + chunk image returned; {Er} chunks per call", "h2d_bytes_per_step": rec_in, "d2h_bytes_per_step": rec_out,
                          "roofline": {"bound": "pcie", "peak": rec_peak, "frac": rec_value / rec_peak,
                                       "how": "the same bytes as pinned copies, H2D and D2H together (D2H is the larger direction here)"}}
        del parts_h, crc_h, out_h, img_h, dparts, d_par2, d_crc2

    if rank != 0:
        if dist:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    launches_per_step = launches / max(1, args.steps)
    alg = algorithmic_bytes_per_chunk(k, m) * T
    kernel_ms = float(np.mean(step_ms))
    achieved = alg / (kernel_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_chunk") * T if tj.get("dram_bytes_per_chunk") else None
            traffic_src = "per-chunk DRAM bytes of the committed ncu --set full capture (profiles/roofline_traffic.json) x chunks per launch; NOT measured in this run"
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                "kernel": "fused encode+CRC step" if launches_per_step <= 1.01 else f"{launches_per_step:.0f} kernels per step (generic route); duration = whole step",
                "launch_ms": kernel_ms,
                "library_timer": {"batches": lib_stats["batches_timed"], "gbps_mean": lib_stats["batch_gbps_mean"],
                                  "note": "lzgpu_stats.batch_*: the library's own CUDA-event timing of the same launches (warm-up included)"}}

    cpu_baseline = None
    if not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)
        cores = host_threads()
        n = args.cpu_chunks or max(cores, 8)
        v, kind, secs = cpu_reference_run(args.goal, n, cores)
        best = cpu_reference_best_case(args.goal, n, cores)
        cpu_baseline = {"value": v, "unit": "GiB/s", "cores": cores, "kind": kind,
                        "sample": f"{n} x 64 MiB chunks ({secs:.1f} s), reference call pattern, {cores} threads",
                        "whole_part_kernel_value": best,
                        "whole_part_kernel_note": "one rs.encode over whole parts + mycrc32 per block (SURVEY 8d(ii)), parts pre-split outside the timed region"}

    line = {
        "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{goal} encode + per-64KiB-block CRC32, 64 MiB chunks (BASELINE.json configs[2])",
                   "chunks_per_step_per_gpu": T, "resident_bytes_per_gpu": T * (CHUNK + par_stride + 4 * crc_stride),
                   "l2_policy": "inputs (32 GiB/step) far larger than the 126 MB L2; no flush needed",
                   "parallelism": f"static round-robin of chunk tiles over {world} GPU(s), no collective",
                   "parity_check": f"{headline_checked} chunks of the timed tile (rank 0) bit-exact vs {checker_name}: parity parts and every block CRC"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "extra": extra, "extra_gpu_launches": int(extra_launches),
    }
    print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
