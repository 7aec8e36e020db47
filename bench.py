#!/usr/bin/env python
"""bench.py -- BFV ct x ct mul+relinearize throughput at N=2^15, 14x62-bit q (BASELINE.json).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--batch B] [--dump-outputs DIR]

A "step" is one pass of Multiplicator::multiply over one batch of `--batch` ciphertext pairs
per GPU (synthetic uniform residues, as fresh BFV ciphertext halves are).  Prints ONE JSON line
(rank 0).  `--impl reference` times the reference's CPU algorithm instead (the oracle port --
the Rust reference cannot be built in this image), on all host cores, same metric/config.
`--dump-outputs DIR` writes a fixed sample of rank 0's products of the last timed step to DIR
(see dump_outputs); the inputs depend only on the arguments, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEGREE = 1 << 15
N_MODULI = 14
PLAINTEXT = 786433          # generate_prime(20, 2N, 2^20), as benches/bfv.rs:28 does
NTT_CFG = dict(degree=1 << 14, n_moduli=8, batch=256)   # BASELINE config 2
METRIC = "bfv_ct_mul_relin_per_sec_n32768_14x62bit"
UNIT = "products/s"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ntt_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the two NTT tile kernels for one batched NTT of the roofline
    shape, from the committed ncu --set full capture (profiles/ntt_traffic.json), or None"""
    try:
        with open(os.path.join(ROOT, "profiles", "ntt_traffic.json")) as f:
            return float(json.load(f)["bytes_per_batched_ntt"])
    except Exception:
        return None


def ntt_multiplier_pipe():
    """busy fraction of the FMA-heavy pipe (where the integer multiplies run) of the same launches, same capture"""
    try:
        with open(os.path.join(ROOT, "profiles", "ntt_traffic.json")) as f:
            return json.load(f).get("fmaheavy_busy_pct")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


class DevArray:
    """__cuda_array_interface__ view of a batch's device storage (zero-copy fill from torch)."""

    def __init__(self, ptr, n_words):
        self.__cuda_array_interface__ = {"shape": (n_words,), "typestr": "<i8", "data": (ptr, False), "version": 3}


def fill_uniform(torch, ct, moduli, seed):
    """uniform residues in [0, q_i) written straight into the batch's HBM storage"""
    count, parts, limbs, n = ct.shape()
    view = torch.as_tensor(DevArray(ct.device_ptr(), count * parts * limbs * n), device="cuda").view(
        count, parts, limbs, n)
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    for i, q in enumerate(moduli[:limbs]):
        view[:, :, i, :].copy_(torch.randint(0, q, (count, parts, n), dtype=torch.int64, device="cuda", generator=g))
    torch.cuda.synchronize()


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; kind 'port'), all host cores,
    one ciphertext pair per worker per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    # one ciphertext pair per worker per step.  Capped at 32 workers: the scalar path is memory bound beyond that on
    # this pool's hosts (measured on a 128-core box: 32 workers 38.0 products/s, 128 workers 28.5 products/s);
    # FHE_BENCH_REF_WORKERS overrides the cap
    workers = max(1, min(cores, int(os.environ.get("FHE_BENCH_REF_WORKERS", "32"))))
    # load the checker's shared library in the parent, so that the forked workers (and any process-level accounting
    # of loaded native code) see oracle/libfhe_oracle.so from the start
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fhe_oracle as _O
    _O.lib()
    ctx = mp.get_context("fork")
    barrier = ctx.Barrier(workers + 1)
    q = ctx.Queue()

    def worker(idx):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import numpy as np
        import fhe_oracle as O
        rng = np.random.default_rng(1000 + idx)
        par = O.BfvParameters(DEGREE, PLAINTEXT, moduli_sizes=[62] * N_MODULI)
        ctxq = par.context_at_level(0)
        def rnd(shape_parts):
            a = np.zeros((shape_parts, N_MODULI, DEGREE), np.uint64)
            for i, qq in enumerate(ctxq.moduli):
                a[:, i, :] = rng.integers(0, qq, size=(shape_parts, DEGREE), dtype=np.uint64)
            return a
        ksk = O.KeySwitchingKey.from_arrays(par, rnd(N_MODULI), rnd(N_MODULI))
        m = O.Multiplicator.default(O.RelinearizationKey.from_ksk(ksk))
        a = O.Ciphertext.from_array(par, rnd(2), 0)
        b = O.Ciphertext.from_array(par, rnd(2), 0)
        for _ in range(args.warmup + args.steps):
            barrier.wait()
            m.multiply(a, b)
            barrier.wait()
        q.put(idx)

    procs = [ctx.Process(target=worker, args=(i,)) for i in range(workers)]
    for p in procs:
        p.start()
    times = []
    for s in range(args.warmup + args.steps):
        barrier.wait()
        t0 = time.perf_counter()
        barrier.wait()
        if s >= args.warmup:
            times.append(time.perf_counter() - t0)
    for p in procs:
        p.join()
    total = sum(times)
    value = workers * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "BASELINE configs[2]: n=2^15, 14x62-bit moduli, ct x ct mul + relinearize",
                   "batch_per_step": workers},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port",
                         "sample": "%d steps x %d products (one per worker process), C oracle of the reference "
                                   "algorithm (the Rust reference cannot be built here)" % (args.steps, workers)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _oracle_set_c():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fhe_oracle as O
    return O, O.BfvParameters(DEGREE, PLAINTEXT, moduli_sizes=[62] * N_MODULI)


def verify_against_oracle(np, A, Bt, out, rot, kc, gc, indices):
    """Outside the timed region: download operands and results of a few ciphertexts whose indices span the internal
    128-ciphertext chunks and compare them bit for bit with the CPU oracle (the checker, never the thing measured).
    `rot` (nullable) is the rotated batch of A under the Galois key gc."""
    O, opar = _oracle_set_c()
    om = O.Multiplicator.default(O.RelinearizationKey.from_ksk(O.KeySwitchingKey.from_arrays(opar, kc[0], kc[1])))
    ogk = O.GaloisKey.__new__(O.GaloisKey)
    ogk.exponent, ogk.ksk = 3, O.KeySwitchingKey.from_arrays(opar, gc[0], gc[1])
    one = np.empty((1, 2, N_MODULI, DEGREE), np.uint64)
    ok_mul, ok_rot = True, True
    for i in indices:
        a = A.to_host(one.copy(), first=i)[0]
        b = Bt.to_host(one.copy(), first=i)[0]
        got = out.to_host(one.copy(), first=i)[0]
        exp = om.multiply(O.Ciphertext.from_array(opar, a, 0), O.Ciphertext.from_array(opar, b, 0)).to_array()
        ok_mul &= bool((got == exp).all())
        if rot is not None:
            gr = rot.to_host(one.copy(), first=i)[0]
            ok_rot &= bool((gr == ogk.relinearize(O.Ciphertext.from_array(opar, a, 0)).to_array()).all())
    return ok_mul, ok_rot


def dump_outputs(np, out, directory, n_ct=16, n_coeff=2048):
    """Writes a fixed sample of the product batch `out` as float64 .npy files (about 15 MB):
      products.npy            [n_ct][2][N_MODULI][n_coeff][2]  each u64 residue as (high 32 bits, low 32 bits),
                                                               both exact in float64
      ciphertext_index.npy    [n_ct]     which ciphertexts of the batch (always the first, the last and both sides of
                                         the library's 256-ciphertext chunk boundary)
      coefficient_index.npy   [n_coeff]  which coefficients of every polynomial
    The sample is drawn from a fixed seed, so it is the same for every run with the same --batch."""
    count = out.shape()[0]
    rng = np.random.default_rng(12345)
    fixed = sorted(set(i for i in (0, 255, 256, count - 1) if i < count))
    rest = np.setdiff1d(np.arange(count), fixed)
    cts = np.sort(np.concatenate([fixed, rng.choice(rest, min(len(rest), n_ct - len(fixed)), replace=False)]))
    coeffs = np.sort(rng.choice(DEGREE, n_coeff, replace=False))
    one = np.empty((1, 2, N_MODULI, DEGREE), np.uint64)
    words = np.stack([out.to_host(one, first=int(i))[0][:, :, coeffs] for i in cts])
    split = np.stack([words >> np.uint64(32), words & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "products.npy"), split)
    np.save(os.path.join(directory, "ciphertext_index.npy"), cts.astype(np.float64))
    np.save(os.path.join(directory, "coefficient_index.npy"), coeffs.astype(np.float64))


def cpu_baseline_sample():
    """single-thread oracle port on a bounded sample (3 products at the full size)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import fhe_oracle as O
    rng = np.random.default_rng(5)
    par = O.BfvParameters(DEGREE, PLAINTEXT, moduli_sizes=[62] * N_MODULI)
    ctxq = par.context_at_level(0)

    def rnd(parts):
        a = np.zeros((parts, N_MODULI, DEGREE), np.uint64)
        for i, qq in enumerate(ctxq.moduli):
            a[:, i, :] = rng.integers(0, qq, size=(parts, DEGREE), dtype=np.uint64)
        return a
    ksk = O.KeySwitchingKey.from_arrays(par, rnd(N_MODULI), rnd(N_MODULI))
    m = O.Multiplicator.default(O.RelinearizationKey.from_ksk(ksk))
    a, b = O.Ciphertext.from_array(par, rnd(2), 0), O.Ciphertext.from_array(par, rnd(2), 0)
    m.multiply(a, b)  # warm tables / page-in
    n, t0 = 20, time.perf_counter()
    for _ in range(n):
        m.multiply(a, b)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d ct x ct mul+relin at n=2^15, 14x62-bit, single thread, C oracle of the reference "
                      "algorithm (Rust reference not buildable here)" % n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("FHE_BENCH_BATCH", "1024")))
    # end-to-end batch per step and GPU: a step drains its pipeline (the last chunk's multiply and download have nothing
    # to overlap with), so the larger the batch the closer the rate gets to the link: 256 -> 3100, 512 -> 3320,
    # 1024 -> 3440 products/s on one B200 (copy-only ceiling 3550).  512 keeps the pinned staging at 11 GB per rank.
    ap.add_argument("--e2e-batch", type=int, default=int(os.environ.get("FHE_BENCH_E2E_BATCH", "512")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the last timed step's products to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the products of the GPU path only")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import fhe_rs_b200 as F
    from fhe_rs_b200._capi import check
    L = F._capi.lib()

    # BfvParametersBuilder::set_moduli_sizes(&[62; 14]) -> the library generates the primes (parameters.rs:391)
    par = F.BfvParameters(DEGREE, PLAINTEXT, moduli_sizes=[62] * N_MODULI, device=local)
    moduli = par.moduli()
    B = args.batch
    # independent ciphertexts shard across ranks: every rank owns B pairs (weak scaling), keys replicated
    A = F.Ciphertext(par, B, 2)
    Bt = F.Ciphertext(par, B, 2)
    fill_uniform(torch, A, moduli, 1 + 2 * rank)
    fill_uniform(torch, Bt, moduli, 2 + 2 * rank)
    rng = np.random.default_rng(7)   # same key on every rank
    kc = np.zeros((2, N_MODULI, N_MODULI, DEGREE), np.uint64)
    for i, q in enumerate(moduli):
        kc[:, :, i, :] = rng.integers(0, q, size=(2, N_MODULI, DEGREE), dtype=np.uint64)
    rk = F.RelinearizationKey.from_arrays(par, kc[0], kc[1])
    gc = np.zeros((2, N_MODULI, N_MODULI, DEGREE), np.uint64)
    for i, q in enumerate(moduli):
        gc[:, :, i, :] = rng.integers(0, q, size=(2, N_MODULI, DEGREE), dtype=np.uint64)
    gk = F.GaloisKey.from_arrays(par, 3, gc[0], gc[1])     # column rotation by one (evaluation_key.rs:118)
    out = F.Ciphertext(par, B, 2)

    def step():
        check(L.fhe_b200_mul_relin(A._h, Bt._h, rk.ksk._h, 0, out._h, None))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = L.fhe_b200_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    launches = L.fhe_b200_launch_count() - l0
    from fhe_rs_b200.shard import bind_host_thread_to_gpu, gather_checksums, max_over_ranks
    ms = max_over_ranks(ev0.elapsed_time(ev1), device="cuda")     # device time of the slowest rank
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms * 1e-3)

    # ---- BASELINE configs[3]: GaloisKey rotate (exponent 3) of the same batch, CUDA events, same barriers
    rot = F.Ciphertext(par, B, 2)

    def rot_step():
        check(L.fhe_b200_galois(A._h, 3, gk.ksk._h, rot._h, None))
    for _ in range(2):
        rot_step()
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rot_steps = max(1, min(args.steps, 5))
    r0.record()
    for _ in range(rot_steps):
        rot_step()
    r1.record()
    barrier()
    rot_ms = max_over_ranks(r0.elapsed_time(r1), device="cuda") / rot_steps

    # ---- parity of the timed work, outside the timed region: products / rotations whose indices span the internal
    # chunks are compared with the CPU oracle on every rank; no `value` is printed unless all of them are bit-exact
    idx = sorted(set(i for i in ((0, 255, 256, B - 1) if rank == 0 else (0, B - 1)) if 0 <= i < B))   # 256 = the library's chunk
    ok_mul, ok_rot = verify_against_oracle(np, A, Bt, out, rot, kc, gc, idx)
    okt = torch.tensor([int(ok_mul), int(ok_rot)], device="cuda")
    if world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    ok_mul, ok_rot = bool(okt[0].item()), bool(okt[1].item())
    assert ok_mul, "timed mul+relin products differ from the oracle"
    assert ok_rot, "timed rotations differ from the oracle"
    # the one collective of the path: the (trivial) gather of results -- here one 63-bit checksum of every rank's
    # product batch, NCCL all-gather in global shard order
    n_out_words = B * 2 * N_MODULI * DEGREE
    cs = int(torch.as_tensor(DevArray(out.device_ptr(), n_out_words), device="cuda").sum().item()) & ((1 << 63) - 1)
    checksums = gather_checksums([cs], device="cuda")
    if args.dump_outputs and rank == 0:
        dump_outputs(np, out, args.dump_outputs)

    # ct + ct (the HBM-bound member of the family): rot += out, 3 rows of traffic per limb row
    for _ in range(2):
        check(L.fhe_b200_add(rot._h, out._h, None))
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(10):
        check(L.fhe_b200_add(rot._h, out._h, None))
    a1.record()
    barrier()
    add_ms = a0.elapsed_time(a1) / 10
    del rot

    # ---- end to end through the public host API (C ABI) with HOST buffers: every step uploads the step's
    # operands from pinned host memory, multiplies, and downloads the products; chunks of 32 pairs rotate over
    # several streams so that PCIe copies overlap the kernels of the other chunks
    numa = bind_host_thread_to_gpu(local)   # before the pinned staging buffers are allocated (first touch)
    Be = min(args.e2e_batch, B)
    ch = min(32, Be)
    Be -= Be % ch
    wpc = 2 * N_MODULI * DEGREE                    # words per ciphertext
    wc = os.environ.get("FHE_BENCH_WC", "0") == "1"   # upload staging in write-combining pages (fhe_b200_host_alloc)

    def staging(write_combined):
        import ctypes
        p = ctypes.c_void_p()
        check(L.fhe_b200_host_alloc(Be * wpc * 8, 1 if write_combined else 0, ctypes.byref(p)))
        return torch.frombuffer((ctypes.c_char * (Be * wpc * 8)).from_address(p.value), dtype=torch.int64)
    while True:
        try:
            ha, hb, ho = staging(wc), staging(wc), staging(False)
            break
        except Exception:              # the host refused to pin that much: halve the end-to-end batch (all ranks alike)
            if Be <= 2 * ch:
                raise
            ha = hb = ho = None
            Be //= 2
            Be -= Be % ch
    if world > 1:                      # every rank runs the same end-to-end batch
        bt = torch.tensor([Be], device="cuda")
        dist.all_reduce(bt, op=dist.ReduceOp.MIN)
        if int(bt.item()) != Be:
            Be = int(bt.item())
            ha, hb, ho = ha[: Be * wpc], hb[: Be * wpc], ho[: Be * wpc]
    ha.copy_(torch.as_tensor(DevArray(A.device_ptr(), Be * wpc), device="cuda"))
    hb.copy_(torch.as_tensor(DevArray(Bt.device_ptr(), Be * wpc), device="cuda"))
    torch.cuda.synchronize()
    n_slots = int(os.environ.get("FHE_BENCH_E2E_SLOTS", "3"))   # upload k+1 while k computes and k-1 downloads
    streams = [torch.cuda.Stream() for _ in range(n_slots)]
    # chunk plan: 32-pair chunks, the last 32 pairs tapered (16 + 8 + 8) so that the part of a step nothing overlaps --
    # the multiply and download of the final chunk -- is short.  Every (stream, chunk size) has its own device batches.
    plan, off_ct = [], 0
    tail = [ch // 2, ch // 4, ch // 4] if (ch % 4 == 0 and Be >= 2 * ch and os.environ.get("FHE_BENCH_E2E_TAPER", "1") == "1") else [ch]
    while off_ct + ch <= Be - ch:
        plan.append((off_ct, ch))
        off_ct += ch
    for n_t in (tail if Be - off_ct == ch else [Be - off_ct]):
        plan.append((off_ct, n_t))
        off_ct += n_t
    assert off_ct == Be
    slots = {}

    def slot(k, n_ct):
        key = (k % n_slots, n_ct)
        if key not in slots:
            slots[key] = (F.Ciphertext(par, n_ct, 2), F.Ciphertext(par, n_ct, 2), F.Ciphertext(par, n_ct, 2))
        return slots[key]

    def e2e_step():
        for k, (first, n_ct) in enumerate(plan):
            st = streams[k % n_slots].cuda_stream
            sa, sb, so = slot(k, n_ct)
            off = first * wpc * 8
            check(L.fhe_b200_batch_upload(sa._h, 0, n_ct, ha.data_ptr() + off, st))
            check(L.fhe_b200_batch_upload(sb._h, 0, n_ct, hb.data_ptr() + off, st))
            check(L.fhe_b200_mul_relin(sa._h, sb._h, rk.ksk._h, 0, so._h, st))
            check(L.fhe_b200_batch_download_async(so._h, 0, n_ct, ho.data_ptr() + off, st))
        for s_ in streams:
            check(L.fhe_b200_sync(s_.cuda_stream))

    e2e_step()
    barrier()
    # the end-to-end products must equal the device-resident ones (verified against the oracle above): first and
    # last product of the first chunk, first of the second chunk (another stream / slot), last of the batch
    for k in sorted(set((0, ch - 1, min(ch, Be - 1), Be - 1))):
        dev = torch.as_tensor(DevArray(out.device_ptr() + k * wpc * 8, wpc), device="cuda").cpu()
        assert bool((ho[k * wpc:(k + 1) * wpc] == dev).all()), "e2e product %d differs from the device-resident run" % k
    e2e_step()   # second warm-up pass: the stream-ordered pool has now seen the three-stream pattern
    barrier()
    e2e_steps = max(1, min(args.steps, 5))
    step_s = []
    for _ in range(e2e_steps):
        ts = time.perf_counter()
        e2e_step()               # ends with a synchronize of every stream it used
        step_s.append(time.perf_counter() - ts)
    barrier()
    # per-step wall times, max over ranks per step; the reported rate uses the median step (a single stalled step --
    # another tenant's PCIe burst, a pool growth -- is visible in step_ms instead of halving the figure)
    st_t = torch.tensor(step_s, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(st_t, op=dist.ReduceOp.MAX)
    step_s = sorted(float(x) for x in st_t.cpu())
    e2e_value = world * Be / step_s[len(step_s) // 2]
    words = Be * wpc
    # what the box gives plain pinned copies of the same buffers, every rank copying AT THE SAME TIME (diagnostic: the
    # end-to-end path is bound by the host side of the links -- one link alone at N = 1, the host's aggregate at N = 8)
    dbuf = torch.empty(Be * wpc, dtype=torch.int64, device="cuda")
    pcie = {}
    for name, dst_, src_ in (("h2d", dbuf, ha), ("d2h", ho, dbuf)):
        dst_.copy_(src_, non_blocking=True)
        barrier()
        t1 = time.perf_counter()
        for _ in range(3):
            dst_.copy_(src_, non_blocking=True)
        torch.cuda.synchronize()
        pcie[name] = 3 * Be * wpc * 8 / (time.perf_counter() - t1) / 1e9
    # both directions at once with the end-to-end step's own mix (two operand uploads per product download), every
    # rank at the same time: Be products' worth of traffic per pass -> the rate the links (and, at N = 8, the host's
    # memory system behind them) allow the end-to-end path, whatever the kernels do
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
    dbuf2 = torch.empty(Be * wpc, dtype=torch.int64, device="cuda")
    src_dev = torch.as_tensor(DevArray(out.device_ptr(), Be * wpc), device="cuda")
    barrier()
    t1 = time.perf_counter()
    for _ in range(3):
        with torch.cuda.stream(s_up):
            dbuf.copy_(ha, non_blocking=True)
            dbuf2.copy_(hb, non_blocking=True)
        with torch.cuda.stream(s_dn):
            ho.copy_(src_dev, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t1
    pcie["duplex_h2d"] = 3 * 2 * Be * wpc * 8 / dt / 1e9
    pcie["duplex_products_per_s"] = 3 * Be / dt
    del dbuf2
    del dbuf
    per_rank = [None] * world
    mine = {"rank": rank, "h2d": round(pcie["h2d"], 1), "d2h": round(pcie["d2h"], 1),
            "duplex_h2d": round(pcie["duplex_h2d"], 1), "copy_only_products_per_s": round(pcie["duplex_products_per_s"], 1),
            "host_numa": numa,
            "cpus": len(os.sched_getaffinity(0))}
    if world > 1:
        dist.all_gather_object(per_rank, mine)
    else:
        per_rank = [mine]

    # ---- roofline of the dominant kernel family (NTT), BASELINE config 2: [256][8][2^14] forward + inverse
    roof = None
    if rank == 0:
        par2 = F.BfvParameters(NTT_CFG["degree"], PLAINTEXT, moduli_sizes=[62] * NTT_CFG["n_moduli"], device=local)
        nm = par2.moduli()
        X = F.Ciphertext(par2, NTT_CFG["batch"], 1, repr=F.POWER_BASIS)
        fill_uniform(torch, X, nm, 99)
        for _ in range(3):
            X.into_ntt(); X.into_power_basis()
        torch.cuda.synchronize()
        reps = 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            X.into_ntt(); X.into_power_basis()
        e1.record()
        torch.cuda.synchronize()
        ntt_ms = e0.elapsed_time(e1) / (2 * reps)
        rows = NTT_CFG["batch"] * NTT_CFG["n_moduli"]
        alg_bytes = 16.0 * NTT_CFG["degree"] * rows          # SURVEY 8d: 16*N bytes per limb-NTT
        achieved = alg_bytes / (ntt_ms * 1e-3) / 1e9
        peak, how = peaks()
        roof = {"bound": "hbm", "kernel": "ntt_tma_cols_kernel<8,*> (cols pass) + ntt_tma_rows_pair_kernel<*> (rows pass), TMA-fed persistent: one batched %d-row NTT, N=2^14" % rows,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": how,
                "traffic": ntt_traffic(), "ms_per_launch": ntt_ms, "multiplier_pipe": ntt_multiplier_pipe(),
                "note": "algorithmic bytes = 16*N per limb-NTT (SURVEY 8d). The transform is bound by the integer "
                        "multiplier pipe, not by HBM: an N-point transform is N/2*log2(N) butterflies for 16*N bytes, so "
                        "the bare-butterfly peak (issue_roofline.peak) caps this fraction at 0.34 for N=2^14 (0.31 "
                        "for N=2^15); see DESIGN.md section 3.2",
                # second roofline for the same launches: 62-bit Harvey/Shoup butterflies per second against the
                # measured peak of this pool's B200 (bench_micro/bf_bench.cu: 3.42 butterflies/clk/SM at 1.9 GHz)
                "issue_roofline": {"unit": "T butterflies/s",
                                   "achieved": rows * (NTT_CFG["degree"] // 2) * 14 / (ntt_ms * 1e-3) / 1e12,
                                   "peak": 0.961, "peak_source": "measured butterfly-only kernel, profiles/microbench_r1.txt",
                                   "frac": rows * (NTT_CFG["degree"] // 2) * 14 / (ntt_ms * 1e-3) / 1e12 / 0.961}}

    if rank == 0:
        cpu = None if (args.no_cpu_baseline or world > 1) else cpu_baseline_sample()   # rank 0, N = 1 only
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "BASELINE configs[2]: n=2^15, 14x62-bit moduli, ct x ct mul + relinearize, "
                                   "batch %d ciphertext pairs per GPU" % B,
                       "batch_per_gpu": B, "parallelism": "independent ciphertexts sharded per rank, keys replicated",
                       "l2": "inputs (%.1f GB per step per GPU) exceed L2, no flush needed" % (2 * B * 7.34e-3)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * words * 8,
                    "d2h_bytes_per_step": words * 8, "batch": Be, "streams": n_slots,
                    "upload_staging": "write-combined pinned" if wc else "pinned",
                    "chunks": [n_ct for _, n_ct in plan][-6:], "n_chunks": len(plan),
                    "timing": "median of %d steps (wall clock around upload+multiply+download, max over ranks)" % e2e_steps,
                    "step_ms": [round(x * 1e3, 2) for x in step_s],
                    "pinned_copy_gbs": {"h2d": round(pcie["h2d"], 1), "d2h": round(pcie["d2h"], 1)}, "host_numa": numa,
                    # every rank's plain pinned-copy rate with all ranks copying concurrently: their sum is the
                    # host's aggregate ceiling for the end-to-end path (14.7 MB up + 7.3 MB down per product)
                    "concurrent_pinned_copy_gbs_per_rank": per_rank,
                    "aggregate_h2d_gbs": round(sum(r["duplex_h2d"] for r in per_rank), 1),
                    "link_bound_products_per_s": round(sum(r["copy_only_products_per_s"] for r in per_rank), 1)},
            "gpu_launches": int(launches),
            "verified": {"against": "CPU oracle (oracle/fhe_oracle), outside the timed region", "bit_exact": True,
                         "mul_relin_indices": idx, "rotate_indices": idx,
                         "e2e_vs_device_indices": sorted(set((0, ch - 1, min(ch, Be - 1), Be - 1))),
                         "ranks": world},
            "result_gather": {"collective": "all_gather of one 63-bit checksum per rank (NCCL)" if world > 1 else "none (1 rank)",
                              "checksums": checksums},
            "roofline": roof,
            "secondary": {
                "rotate": {"workload": "BASELINE configs[3]: n=2^15, 14x62-bit, GaloisKey rotate (exponent 3), batch %d per GPU" % B,
                           "value": world * B / (rot_ms * 1e-3), "unit": "rotations/s", "ms_per_step": rot_ms,
                           "steps": rot_steps,
                           "roofline": {"bound": "hbm", "unit": "GB/s", "algorithmic_mb_per_rotate": 143.0,
                                        "achieved": 143.0e-3 * B / (rot_ms * 1e-3), "peak": peaks()[0],
                                        "frac": 143.0e-3 * B / (rot_ms * 1e-3) / peaks()[0],
                                        "note": "SURVEY 8d stage model: 2 gathers, L iNTT, L^2 digit NTTs, inner product, add"}},
                "add": {"workload": "ct + ct, batch %d" % B, "value": B / (add_ms * 1e-3), "unit": "ct/s (one GPU)",
                        "roofline": {"bound": "hbm", "unit": "GB/s", "algorithmic_mb_per_add": 22.0,
                                     "achieved": 22.0e-3 * B / (add_ms * 1e-3), "peak": peaks()[0],
                                     "frac": 22.0e-3 * B / (add_ms * 1e-3) / peaks()[0]}},
            },
            "cpu_baseline": cpu,
            "vs_single_thread": None if cpu is None else {"device_resident": value / cpu["value"],
                                                          "e2e": e2e_value / cpu["value"], "cores": 1},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
