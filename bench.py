#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for the FHE ciphertext-arithmetic hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU arm (oracle port, all host threads)
    python bench.py --gpus 1 --steps K --dump-outputs DIR    # also write a sample of the last timed step's output to DIR

One "step" = one pass of ct x ct multiply + relinearise (dpfhe_ct_mul_relin) over one batch of synthetic ciphertexts,
N = 8192, L = 4: BASELINE.json config 2 (batch 4096) on one GPU, config 5 (65,536 ciphertexts over 8 GPUs = 8192 per GPU)
when launched on several.
  value      whole-job ct-mults/s, inputs resident in HBM, timed with CUDA events on the launch stream
  e2e        the same metric through the host-buffer C-ABI call (pinned host memory on the GPU's NUMA node, H2D + D2H inside)
  roofline   the fused key-switch kernel against the measured HBM copy bandwidth (MEASURED_PEAKS.json); int_pipe = what
             actually limits it (the integer multiplier), from the committed ncu capture
  ntt        NTTs/s of the standalone forward and inverse transforms (N = 8192 and N = 16384), with their rooflines
  cpu_baseline  the CPU oracle (kind "port": the reference has no CPU evaluator, DESIGN.md §1) on the SAME batch; its output is
             also the checker of the timed GPU result ("parity")
Multi-GPU: one process per GPU (torchrun), ciphertexts sharded by rank, no collective while computing (weak scaling).
The final result gather to rank 0 rides on the kernel's own output stores: every rank writes its finished rows straight
into rank 0's buffer (CUDA IPC mapping, NVLink), so the gather overlaps the compute ("gather"; the NCCL gather that
would otherwise follow the compute is timed beside it).
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

LOG_N, L, BATCH, BATCH_MULTI = 13, 4, 4096, 8192     # config 2 / the per-GPU shard of config 5
N = 1 << LOG_N
P_WORDS = L * N
CT_BYTES = 2 * P_WORDS * 8
ALGO_BYTES_CT_MUL = 6 * P_WORDS * 8      # read 2 cts, write 1 ct   (SURVEY.md §8d)
ALGO_BYTES_NTT = 2 * N * 8               # read + write one limb
SEED = 0xD3390002                        # 0xD3390000 + config id 2
DUMP_CTS = 32                            # ciphertexts of the last timed step written by --dump-outputs (2 x 16 MiB)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of the headline ct x ct multiply")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dpfhe", choices=["dpfhe", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="ciphertexts per GPU per step (default: 4096 on one GPU, 8192 per GPU on several)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the informational timings (special-prime key switching, N=16384 transforms)")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed, seeded sample of the ciphertexts the last timed step computed "
                    "to DIR/*.npy (rank 0's shard), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's output; use it without --impl reference")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_for(kernel, units):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `units` work units, scaled from the committed
    ncu --set full capture (profiles/traffic.json holds bytes per unit at the profiled batch); None if absent"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            rec = json.load(f).get(kernel)
        return float(rec["dram_bytes_per_unit"]) * units if rec else None
    except Exception:
        return None


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def pick_threads(o):
    """thread count for the CPU arm: the fastest of {all processors, half of them (one per core on SMT hosts), OpenMP's own
    default} on a short probe — more threads are not always faster (measured on this pool's host: 128 threads 2.8 k, 64
    threads 6.6 k ct-mult/s), and launchers such as torchrun cap OMP_NUM_THREADS at 1"""
    procs = o.host_threads()
    cands = sorted({procs, max(1, procs // 2), max(1, o.max_threads())}, reverse=True)
    s = o.keygen_secret(1)
    evk = o.keygen_relin(2, 65537, s)
    n = min(512, 8 * max(cands))     # several ciphertexts per thread: a probe of one each mostly times the thread start-up
    a = o.fill_uniform(SEED, 2 * n).reshape(n, 2, L, N)
    b = o.fill_uniform(SEED, 2 * n, first_poly=2 * n).reshape(n, 2, L, N)
    _, out = o.time_ct_mul_relin(a, b, evk, cands[0])
    best, best_t = cands[0], None
    for c in cands:
        t = min(o.time_ct_mul_relin(a, b, evk, c, out=out)[0] for _ in range(3))
        if best_t is None or t < best_t:
            best, best_t = c, t
    return best


def cpu_sample(oracle_ctx, seconds, threads):
    """times the oracle's ct_mul_relin on a bounded sample for about `seconds` of wall time;
    returns (ct-mults/s, ct-mults timed, seconds).  The sample is at most 1024 ciphertexts (1.5 GiB of host
    arrays) and is repeated until the time budget is used, so many-core hosts still get a 10-30 s measurement."""
    o = oracle_ctx
    s = o.keygen_secret(1)
    evk = o.keygen_relin(2, 65537, s)
    probe = max(threads, 1)
    a = o.fill_uniform(SEED, 2 * probe).reshape(probe, 2, L, N)
    b = o.fill_uniform(SEED, 2 * probe, first_poly=2 * probe).reshape(probe, 2, L, N)
    t, _ = o.time_ct_mul_relin(a, b, evk, threads)
    rate = probe / t
    n = int(max(probe, min(1024, rate * seconds)))
    n = max(threads, (n // max(threads, 1)) * max(threads, 1))
    a = o.fill_uniform(SEED, 2 * n).reshape(n, 2, L, N)
    b = o.fill_uniform(SEED, 2 * n, first_poly=2 * n).reshape(n, 2, L, N)
    _, out = o.time_ct_mul_relin(a, b, evk, threads)     # warm-up (page faults of the reused output buffer, thread pool)
    done, total = 0, 0.0
    while total < seconds and done < 64 * n:
        t, _ = o.time_ct_mul_relin(a, b, evk, threads, out=out)
        total += t
        done += n
    return done / total, done, total


def workload_name(world, batch):
    """config.workload of both arms: BASELINE.json config 2 on one GPU, config 5's layout (8192 per GPU) on several"""
    B = batch or (BATCH if world == 1 else BATCH_MULTI)
    if world == 1:
        return "ct x ct multiply + relinearise, N=8192, L=4, batch=%d (BASELINE.json config 2)" % B
    return ("ct x ct multiply + relinearise, N=8192, L=4, batch=%d sharded over %d GPUs, %d per GPU (BASELINE.json config 5: 65536 over 8)"
            % (world * B, world, B))


def dump_outputs(path, out):
    """DUMP_CTS ciphertexts of `out` (a device tensor [B][2][L][N] of residues), picked by a fixed seed, as float64 .npy files.
    A residue (up to 60 bits) does not fit a float64 mantissa, so each word is written as its high and low 30 bits, both exact:
    word = hi * 2^30 + lo."""
    import numpy as np
    import torch
    B = out.shape[0]
    idx = np.sort(np.random.default_rng(SEED).choice(B, min(DUMP_CTS, B), replace=False))
    words = out[torch.from_numpy(idx).to(out.device)].cpu().numpy().view(np.uint64)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "ct_mul_relin_hi30.npy"), (words >> np.uint64(30)).astype(np.float64))
    np.save(os.path.join(path, "ct_mul_relin_lo30.npy"), (words & np.uint64((1 << 30) - 1)).astype(np.float64))


def run_reference(args):
    """CPU arm: the oracle port on all host threads (the reference has no implementation to run)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle
    oracle.build()
    o = oracle.Oracle(LOG_N, L)
    threads = pick_threads(o)
    s = o.keygen_secret(1)
    evk = o.keygen_relin(2, 65537, s)
    # bounded sample per step: about 2 s of CPU work, at most 1024 ciphertexts
    rate, _, _ = cpu_sample(o, 1.0, threads)
    n = int(max(threads, min(1024, args.batch or BATCH, rate * 2.0)))
    a = o.fill_uniform(SEED, 2 * n).reshape(n, 2, L, N)
    b = o.fill_uniform(SEED, 2 * n, first_poly=2 * n).reshape(n, 2, L, N)
    _, out = o.time_ct_mul_relin(a, b, evk, threads)     # the output buffer is touched once and reused: no page faults in the timed steps
    for _ in range(args.warmup):
        o.time_ct_mul_relin(a, b, evk, threads, out=out)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.time_ct_mul_relin(a, b, evk, threads, out=out)
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    line = {
        "impl": "reference", "metric": "ct_mult_relin_per_s", "value": value, "unit": "ct-mult/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(int(os.environ.get("WORLD_SIZE", "1")), args.batch),
                   "sample": "%d ciphertexts per step on the host CPU (a bounded sample of that workload)" % n},
        "cpu_baseline": {"value": value, "unit": "ct-mult/s", "cores": threads, "kind": "port",
                         "sample": "%d ct-mults per step x %d steps, oracle/dpfhe_oracle.c with OpenMP" % (n, args.steps)},
        "e2e": {"value": value, "unit": "ct-mult/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def pipe_profile(kernel):
    """pipe utilisation of `kernel` from the committed ncu --set full capture (profiles/pipes.json, written by
    tools/summarize_ncu.py from the .ncu-rep of the bench batch); None if absent"""
    try:
        with open(os.path.join(ROOT, "profiles", "pipes.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


class DevMem:
    """raw device memory as a torch-visible array (__cuda_array_interface__), for buffers owned by the library / another process"""

    def __init__(self, ptr, n_words):
        self.__cuda_array_interface__ = {"shape": (n_words,), "typestr": "<i8", "data": (ptr, False), "version": 2}


def cpu_leg(o, threads, ha, hb, hk, gpu_out, seconds):
    """the CPU arm on the SAME batch the GPU just processed: oracle ct_mul_relin over all of it, repeated for about `seconds`;
    its output is compared bit for bit with the GPU's.  Returns (cpu_baseline, parity)."""
    import numpy as np
    n = ha.shape[0]
    t, out = o.time_ct_mul_relin(ha, hb, hk, threads)       # first pass: page faults of the output buffer, thread pool
    exact = bool(np.array_equal(out, gpu_out))
    done, total = 0, 0.0
    while total < seconds and done < 64 * n:
        t, _ = o.time_ct_mul_relin(ha, hb, hk, threads, out=out)
        total += t
        done += n
    cpu = {"value": done / total, "unit": "ct-mult/s", "cores": threads, "kind": "port",
           "sample": "%d ct-mults in %.1f s: the bench batch itself (%d ciphertexts, repeated), oracle/dpfhe_oracle.c with OpenMP "
                     "(the reference has no CPU evaluator)" % (done, total, n)}
    parity = {"checked_ciphertexts": n, "bit_exact": exact, "against": "oracle/dpfhe_oracle.c ct_mul_relin on the timed batch"}
    return cpu, parity


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    import deeppowers_b200 as dp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # keep stdout to the single JSON line: NCCL's banner ("NCCL version ...") otherwise lands there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B = args.batch or (BATCH if world == 1 else BATCH_MULTI)
    ctx = dp.Context(LOG_N, L, device=local_rank)
    # this rank's thread (and what it first-touches) stays on the socket its GPU hangs off
    numa = {"node": ctx.numa_node(), "cpus_bound": ctx.bind_thread_near() if world > 1 else 0}
    shape = (B, 2, L, N)
    a = torch.empty(shape, dtype=torch.int64, device="cuda")
    b = torch.empty(shape, dtype=torch.int64, device="cuda")
    out = torch.empty(shape, dtype=torch.int64, device="cuda")
    evk = torch.empty((L, 2, L, N), dtype=torch.int64, device="cuda")
    first = rank * 2 * B          # each rank owns a disjoint slice of the global synthetic stream
    ctx.fill_uniform(SEED, a, 2 * B, first_poly=first)
    ctx.fill_uniform(SEED + 1, b, 2 * B, first_poly=first)
    ctx.fill_uniform(SEED + 2, evk, 2 * L)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = ctx.launch_count()
    total_ms = timed(lambda: ctx.ct_mul_relin(a, b, evk, out, B), args.steps, args.warmup)
    # launches inside the timed region only: key_prepare_kernel + ks_fused_kernel per step
    launches = (ctx.launch_count() - n0) * args.steps // (args.steps + args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)     # before the timings below reuse `out` and transform `a` in place
    ms_per_step = total_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)
    peak, peak_src = peaks()
    kern = "ks_fused_kernel<13,256,3,MUL_RELIN> (dpfhe::fast, persistent cooperative, 3 CTAs/SM)"
    kern_gbs = B * ALGO_BYTES_CT_MUL / (ms_per_step * 1e-3) / 1e9      # per GPU: one launch per step
    roofline = {"bound": "hbm", "kernel": kern, "achieved": kern_gbs, "peak": peak, "unit": "GB/s", "frac": kern_gbs / peak,
                "traffic": traffic_for("ks_fused_kernel_mul_relin", B), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": B * ALGO_BYTES_CT_MUL,
                "limiter": "integer multiplier: 64-bit modular arithmetic has no tensor-core form, and IMAD.WIDE issues at a quarter of the "
                           "rate of the other integer instructions (fmaheavy pipe); DRAM stays far below its peak (DESIGN.md section 6)",
                "int_pipe": pipe_profile("ks_fused_kernel_mul_relin")}

    # standalone transforms on the same data (the NTTs/s half of the BASELINE metric): forward and inverse
    k_ntt = max(3, args.steps // 2)
    n_ntt = 2 * B * L

    def ntt_entry(ms, n, nbytes, kernel, tkey):
        gbs = n * nbytes / (ms * 1e-3) / 1e9
        return {"value": world * n / (ms * 1e-3), "unit": "NTT/s", "ms_per_step": ms,
                "roofline": {"bound": "hbm", "kernel": kernel, "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                             "traffic": traffic_for(tkey, n), "int_pipe": pipe_profile(tkey)}}

    fwd_ms = timed(lambda: ctx.ntt_fwd(a, 2 * B), k_ntt, 2) / k_ntt
    inv_ms = timed(lambda: ctx.ntt_inv(a, 2 * B), k_ntt, 2) / k_ntt
    ntt = ntt_entry(fwd_ms, n_ntt, ALGO_BYTES_NTT, "ntt_kernel<13,256,3,fwd> (dpfhe::fast, one CTA per limb, 3 CTAs/SM)", "ntt_kernel_fwd")
    ntt["metric"] = "ntt_fwd_per_s"
    ntt["inverse"] = ntt_entry(inv_ms, n_ntt, ALGO_BYTES_NTT, "ntt_inv_tma_kernel<13,256,3> (inverse passes of ntt_kernel, limb fetched by TMA)", "ntt_kernel_inv")
    ctx.fill_uniform(SEED, a, 2 * B, first_poly=first)     # restore `a` (the transforms ran in place)
    if not args.no_extras:
        # config 3's ring: N = 16384, L = 8 (1024 ciphertexts = 16384 limb transforms of 128 KiB)
        ctx14 = dp.Context(14, 8, device=local_rank)
        x14 = torch.empty((2048, 8, 1 << 14), dtype=torch.int64, device="cuda")
        ctx14.fill_uniform(SEED + 7, x14, 2048)
        f14 = timed(lambda: ctx14.ntt_fwd(x14, 2048), 3, 2) / 3
        i14 = timed(lambda: ctx14.ntt_inv(x14, 2048), 3, 2) / 3
        ntt["n16384"] = {"fwd": ntt_entry(f14, 2048 * 8, 2 * (1 << 14) * 8, "ntt_kernel<14,...,fwd>", "ntt_kernel_fwd_n16384"),
                         "inv": ntt_entry(i14, 2048 * 8, 2 * (1 << 14) * 8, "ntt_kernel<14,...,inv>", "ntt_kernel_inv_n16384")}
        ctx14.close()
        del x14

    # SURVEY.md section 8 row f-2 (informational, not the headline): the same ciphertexts through special-prime hybrid
    # key switching (context = the four ciphertext moduli + one special prime; 30 transforms per ct-mult instead of 16)
    extras = None
    if not args.no_extras:
        ctx5 = dp.Context(LOG_N, L + 1, device=local_rank)
        hkey = torch.empty((L, 2, L + 1, N), dtype=torch.int64, device="cuda")
        ctx5.fill_uniform(SEED + 3, hkey, 2 * L)
        k = max(3, args.steps // 3)
        hyb_ms = timed(lambda: ctx5.ct_mul_relin_hybrid(a, b, hkey, out, B, 65537), k, 2) / k
        extras = {"ct_mul_relin_hybrid": {"value": world * B / (hyb_ms * 1e-3), "unit": "ct-mult/s", "ms_per_step": hyb_ms,
                                          "kernel": "ks_hybrid_kernel<13,256,3,MUL_RELIN>", "GBps": B * ALGO_BYTES_CT_MUL / (hyb_ms * 1e-3) / 1e9,
                                          "note": "4 ciphertext limbs + 1 special prime, BGV rounding t=65537 (DESIGN.md 2.10)"}}
        ctx5.close()
        del hkey
        # the same ciphertexts with digits of two limbs and two special primes (DESIGN.md 2.11: 24 transforms, a 1.5 MiB key)
        ctx6 = dp.Context(LOG_N, L + 2, device=local_rank)
        dn = ctx6.grouped_digits(2)
        gkey = torch.empty((dn, 2, L + 2, N), dtype=torch.int64, device="cuda")
        ctx6.fill_uniform(SEED + 4, gkey, 2 * dn)
        grp_ms = timed(lambda: ctx6.ct_mul_relin_grouped(2, a, b, gkey, out, B, 65537), k, 2) / k
        extras["ct_mul_relin_grouped"] = {"value": world * B / (grp_ms * 1e-3), "unit": "ct-mult/s", "ms_per_step": grp_ms,
                                          "kernel": "ks_grouped_kernel<13,256,3,MUL_RELIN>", "GBps": B * ALGO_BYTES_CT_MUL / (grp_ms * 1e-3) / 1e9,
                                          "note": "4 ciphertext limbs in 2 digits + 2 special primes, BGV rounding t=65537 (DESIGN.md 2.11)"}
        ctx6.close()
        del gkey
    ctx.ct_mul_relin(a, b, evk, out, B)     # `out` = the reference result for the comparisons below
    torch.cuda.synchronize()

    # end to end through the host-buffer ABI: pinned host memory on this GPU's NUMA node, H2D + D2H inside the timed region
    e2e = None
    host = None
    if not args.no_e2e or (rank == 0 and world == 1 and not args.no_cpu):
        n_words = B * 2 * P_WORDS
        bufs = [ctx.pinned_near(n_words) for _ in range(3)] + [ctx.pinned_near(2 * L * P_WORDS)]
        na, nb, no = (x.array.reshape(shape) for x in bufs[:3])
        nk = bufs[3].array.reshape(L, 2, L, N)
        for dst, src in ((na, a), (nb, b), (nk, evk)):
            torch.from_numpy(dst.view(np.int64)).copy_(src)
        torch.cuda.synchronize()
        host = (na, nb, nk, no, bufs)
    if not args.no_e2e:
        na, nb, nk, no, bufs = host
        ctx.ct_mul_relin_host(na, nb, nk, no)       # warm-up (allocates the staging buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            ctx.ct_mul_relin_host(na, nb, nk, no)
        dt = torch.tensor([(time.perf_counter() - t0) / args.e2e_steps], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_s = float(dt.item())
        ok = bool(torch.equal(torch.from_numpy(no.view(np.int64)).cuda(), out))     # the host path must reproduce the device path bit for bit
        h2d, d2h = 2 * B * CT_BYTES + 2 * L * P_WORDS * 8, B * CT_BYTES
        e2e = {"value": world * B / e2e_s, "unit": "ct-mult/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_s * 1e3, "matches_device_path": ok,
               "pcie": {"h2d_GBps_per_gpu": h2d / e2e_s / 1e9, "d2h_GBps_per_gpu": d2h / e2e_s / 1e9,
                        "note": "both directions run concurrently; the host-to-device stream (two operand batches per result batch) is the bound"},
               "host_memory": {"gpu_numa_node": numa["node"], "pages_placed_on_node": bufs[0].node, "cpus_bound": numa["cpus_bound"],
                               "allocator": "dpfhe_host_alloc_near (mmap + mbind + cudaHostRegister)"},
               "api": "dpfhe_ct_mul_relin_host (pinned host buffers, 3-stage H2D/compute/D2H pipeline; one call per rank, no collective)"}

    # The final result gather.  Every rank's kernel writes its finished output rows straight into rank 0's buffer (opened here
    # through a CUDA IPC handle), so the gather is spread over the compute instead of following it.
    gather = None
    if world > 1 and not args.no_gather:
        ct_words = 2 * P_WORDS
        root_ptr = ctx.device_alloc(world * B * CT_BYTES) if rank == 0 else None
        handles = [ctx.ipc_export(root_ptr) if rank == 0 else None]
        dist.broadcast_object_list(handles, src=0)
        base = root_ptr if rank == 0 else ctx.ipc_open(handles[0])
        mine = base + rank * B * CT_BYTES
        g_ms = timed(lambda: ctx.ct_mul_relin(a, b, evk, mine, B), max(3, args.steps // 2), 2) / max(3, args.steps // 2)
        # verification: rank 0 compares every slice of its buffer with the checksums of the ranks' local results
        def checks(t):
            v = t.view(-1)
            return torch.stack([v.sum(), (v * 0x1E3779B97F4A7C15 - (v >> 17)).sum()])
        local = checks(out)
        allc = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(allc, local)
        verified = None
        if rank == 0:
            root = torch.as_tensor(DevMem(root_ptr, world * B * ct_words), device="cuda")
            verified = all(bool(torch.equal(checks(root[r * B * ct_words:(r + 1) * B * ct_words]), allc[r])) for r in range(world))
        # the collective this replaces: NCCL gather of the finished outputs to rank 0, after the compute
        nb_ = [torch.empty_like(out) for _ in range(world)] if rank == 0 else None
        warm = [torch.empty_like(out[:8]) for _ in range(world)] if rank == 0 else None
        dist.gather(out[:8].contiguous(), warm, dst=0)      # NCCL channel set-up happens on the first call
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        dist.gather(out, nb_, dst=0)
        g1.record()
        barrier()
        nccl_ms = torch.tensor([g0.elapsed_time(g1)], device="cuda", dtype=torch.float64)
        dist.all_reduce(nccl_ms, op=dist.ReduceOp.MAX)
        nccl_ms = float(nccl_ms.item())
        into_root = (world - 1) * B * CT_BYTES
        gather = {"collective": "none: peer stores of the fused kernel into rank 0's IPC-mapped buffer over NVLink (overlapped with the compute)",
                  "ms_per_step_with_gather": g_ms, "value_with_gather": world * B / (g_ms * 1e-3),
                  "bytes_into_root": into_root, "GBps_into_root": into_root / (g_ms * 1e-3) / 1e9,
                  "nvlink_ingress_bound_ms": into_root / 770e9 * 1e3,
                  "verified_against_local_results": verified,
                  "nccl_gather_after_compute": {"ms": nccl_ms, "GBps_into_root": into_root / (nccl_ms * 1e-3) / 1e9,
                                                "value_with_gather": world * B / ((ms_per_step + nccl_ms) * 1e-3),
                                                "collective": "ncclGather via torch.distributed (not overlapped)"}}
        del nb_
        barrier()
        if rank != 0:
            ctx.ipc_close(base)
        barrier()
        if rank == 0:
            ctx.device_free(root_ptr)

    if rank == 0:
        cpu = parity = None
        if not args.no_cpu and world == 1:
            import oracle
            oracle.build()
            o = oracle.Oracle(LOG_N, L)
            threads = pick_threads(o)
            na, nb, nk, _, _ = host
            cpu, parity = cpu_leg(o, threads, na, nb, nk, out.cpu().numpy().view(np.uint64), args.cpu_seconds)
        workload = workload_name(world, args.batch)
        line = {
            "metric": "ct_mult_relin_per_s", "value": value, "unit": "ct-mult/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload,
                       "global_batch": world * B, "parallelism": "batch-sharded x%d, no collective while computing" % world,
                       "moduli": "the %d largest primes k*2^32+1 below 2^60 (default basis, DESIGN.md 2.1)" % L,
                       "l2": "inputs+outputs are %.1f GiB per GPU (>> 126 MB L2), no flush needed" % (3 * B * CT_BYTES / 2**30),
                       "seed": hex(SEED)},
            "roofline": roofline, "ntt": ntt, "extras": extras, "cpu_baseline": cpu, "parity": parity, "e2e": e2e, "gather": gather,
            "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
