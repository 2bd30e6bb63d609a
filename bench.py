#!/usr/bin/env python3
"""bench.py — Ed25519 verifies/s on B200 for BASELINE.json's config[1]:
   "1xB200 batch verify of 2^20 signatures, 512 B msgs" (per GPU; weak scaling across ranks).

A step = one pass of the hot path over one batch: for every record i,
    d_i = Digest(msg_i) = SHA-512(msg_i)[..32]                (mempool/src/processor.rs:30, messages.rs digests)
    verdict_i = Signature::verify(d_i, pk_i)  (verify_strict)  (crypto/src/lib.rs:200-204)
i.e. the reference-shaped use of a 512-byte payload (every message the reference signs is a 32-byte Digest), followed
for N > 1 by the all-gather of the per-rank accept bitmaps.

  value : whole-job verifies/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e   : the same metric through the host-pointer C-ABI call (pinned host buffers, H2D + D2H inside the timed region)
  --impl reference : the CPU path (oracle = restatement of the reference's dalek path; no Rust toolchain here) on all
                     host cores over a bounded sample of the same workload.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: stdout carries exactly one JSON line

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ALGO_BYTES_VERIFY = 128.125   # SURVEY §8(d): 64 B sig + 32 B pk + 32 B digest in, 1 bit out
ALGO_BYTES_DIGEST = 512 + 32  # bytes hashed + digest out
DUMP_MAX_ELEMS = 1 << 22      # per array written by --dump-outputs: 16 MB of float32


def write_outputs(out_dir, **arrays):
    """--dump-outputs: writes each array as out_dir/<name>.npy in float32.  An array of more than DUMP_MAX_ELEMS elements is cut
    down to a fixed sample of its rows (seed 0, in row order), the same in every run with the same arguments, so that two builds
    of the project can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        rows = max(1, DUMP_MAX_ELEMS // max(1, int(np.prod(a.shape[1:]))))
        if a.shape[0] > rows:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


# ------------------------------------------------------------------------------------------------ input synthesis
def make_inputs(n, n_keys, msg_len, seed, corrupt_frac=0.01, engine=None, oracle=None):
    """Synthetic workload of SURVEY §8(d) config 2: n records, n_keys distinct keys (i mod n_keys), msg_len-byte messages
    shaped like the bench client's transactions (node/src/client.rs:112-120: tag byte, u64 counter, padding), signatures
    over Digest(msg), then corrupt_frac of the records get one flipped bit in sig|pk|msg.
    Signing is RFC 8032 (deterministic), so WHO signs does not change the bytes: the GPU arm uses the engine's load-generation
    signer (hs_keygen_batch / hs_sign_digests: 2^20 signatures in milliseconds instead of a minute of host time) and cross-checks
    a sample against OpenSSL; the reference arm (no engine allowed on that path) uses the oracle's signer."""
    import hashlib
    rng = np.random.default_rng(seed)
    seeds = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
    msgs = rng.integers(0, 256, size=(n, msg_len), dtype=np.uint8)
    msgs[:, 0] = 1
    msgs[:, 1:9] = np.arange(n, dtype=">u8").view(np.uint8).reshape(n, 8)
    key_idx = (np.arange(n) % n_keys).astype(np.uint32)
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(msg_len)
    if engine is not None:
        pks = engine.keygen_batch(seeds)
        digests = np.concatenate([engine.digest32_batch(msgs[lo:lo + (1 << 18)].reshape(-1), off[:min(1 << 18, n - lo) + 1])
                                  for lo in range(0, n, 1 << 18)], axis=0)
        sig = engine.sign_digests(seeds, pks, digests, key_idx=key_idx)
        # independent cross-check of the synthesis itself (OpenSSL + hashlib) on a sample
        from cryptography.hazmat.primitives import serialization
        from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
        for i in rng.choice(n, size=min(n, 256), replace=False):
            sk = Ed25519PrivateKey.from_private_bytes(seeds[key_idx[i]].tobytes())
            d = hashlib.sha512(msgs[i].tobytes()).digest()[:32]
            assert d == digests[i].tobytes() and sk.sign(d) == sig[i].tobytes(), "GPU-synthesised input %d differs from OpenSSL" % i
            assert sk.public_key().public_bytes(serialization.Encoding.Raw, serialization.PublicFormat.Raw) == pks[key_idx[i]].tobytes()
    else:
        pks = oracle.keygen_batch(seeds)
        digests = oracle.digest32_batch(msgs.reshape(-1), off, nthreads=host_cores())
        sig = oracle.sign_batch(seeds, pks, key_idx, digests.reshape(-1), np.arange(n + 1, dtype=np.uint64) * 32, nthreads=host_cores())
    pk = pks[key_idx].copy()
    corrupted = np.zeros(n, dtype=bool)
    k = int(n * corrupt_frac)
    if k:
        pos = rng.choice(n, size=k, replace=False)
        where = rng.integers(0, 3, size=k)
        for i, wsel in zip(pos, where):
            if wsel == 0:
                sig[i, int(rng.integers(0, 64))] ^= 1 << int(rng.integers(0, 8))
            elif wsel == 1:
                pk[i, int(rng.integers(0, 32))] ^= 1 << int(rng.integers(0, 8))
            else:
                msgs[i, int(rng.integers(9, msg_len))] ^= 1 << int(rng.integers(0, 8))
        corrupted[pos] = True
    return dict(sig=sig, pk=pk, msgs=msgs, pks=pks, key_idx=key_idx, corrupted=corrupted)


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if mx and x > 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def host_cores():
    """Cores this process may actually use: min(visible CPUs, affinity mask, cgroup cpu.max quota)."""
    c = os.cpu_count() or 1
    try:
        c = min(c, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            c = min(c, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return c


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def cpu_reference_step(oracle, inp, lo, hi, nthreads):
    """The reference's CPU path on records [lo, hi): Digest(msg) then Signature::verify, all host threads."""
    msgs = inp["msgs"][lo:hi]
    n = hi - lo
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(msgs.shape[1])
    t0 = time.perf_counter()
    d = oracle.digest32_batch(msgs.reshape(-1), off, nthreads=nthreads)
    recs = np.concatenate([inp["sig"][lo:hi], inp["pk"][lo:hi], d], axis=1)
    ok = oracle.verify_rec128(recs, mode=0, nthreads=nthreads)
    return time.perf_counter() - t0, ok


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle_api import Oracle
    oracle = Oracle()
    cores = host_cores()
    sample = min(args.n, args.ref_sample)
    inp = make_inputs(sample, min(args.keys, sample), args.msg_len, seed=1234, corrupt_frac=0.01, oracle=oracle)
    for _ in range(args.warmup):
        cpu_reference_step(oracle, inp, 0, min(sample, 4096), cores)
    times = []
    for _ in range(args.steps):
        dt, ok = cpu_reference_step(oracle, inp, 0, sample, cores)
        times.append(dt)
        assert int(ok.sum()) == sample - int(inp["corrupted"].sum())
    total = float(np.sum(times))
    v = sample * args.steps / total
    line = {
        "impl": "reference", "metric": "Ed25519 verifies/s", "value": v, "unit": "verifies/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": workload_config(args, 1) | {"reference_sample": "%d records per step" % sample},
        "cpu_baseline": {"value": v, "unit": "verifies/s", "cores": cores, "kind": "port",
                         "sample": "%d records/step x %d steps: Digest(512 B) + verify_strict on %d pthreads (oracle = C restatement of the dalek path; reference Rust cannot be built here)" % (sample, args.steps, cores)},
        "e2e": {"value": v, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, world):
    coll = "none (1 rank)" if world == 1 else ("fused peer-store all-gather in the finish kernel (NVLink P2P)" if args.collective == "peer" else "ncclAllGather")
    return {"collective": coll,"workload": "config[1]: 2^20 signatures per GPU, 512 B msgs: Digest(msg)=SHA-512[..32] on GPU then verify_strict over the digest",
            "records_per_gpu": args.n, "msg_len": args.msg_len, "distinct_keys": args.keys, "corrupted_frac": 0.01,
            "key_mode": args.key_mode, "l2": "inputs (%.0f MB/GPU) larger than the 126 MB L2" % (args.n * (96 + args.msg_len) / 1e6),
            "parallelism": "records sharded across %d rank(s); all-gather of accept bitmaps" % world}


# ------------------------------------------------------------------------------------------------ QC workload (configs 2/3)
def make_qc_inputs(eng, n_val, n_qc, votes_per_qc, seed):
    """Committee of n_val validators; n_qc QCs, each with votes_per_qc distinct signers over QC::digest =
    SHA-512(hash || round_le)[..32] (consensus/src/messages.rs:201-208).  1 % of the votes get one flipped signature bit.
    Keys and signatures come from the engine's load-generation signer (RFC 8032, cross-checked against OpenSSL on a sample)."""
    import hashlib
    from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
    rng = np.random.default_rng(seed)
    seeds = rng.integers(0, 256, size=(n_val, 32), dtype=np.uint8)
    pks = eng.keygen_batch(seeds)
    pre = np.zeros((n_qc, 40), dtype=np.uint8)
    pre[:, :32] = rng.integers(0, 256, size=(n_qc, 32), dtype=np.uint8)
    pre[:, 32:] = np.arange(1, n_qc + 1, dtype="<u8").view(np.uint8).reshape(n_qc, 8)
    digests = np.array([np.frombuffer(hashlib.sha512(pre[j].tobytes()).digest()[:32], dtype=np.uint8) for j in range(n_qc)])
    n = n_qc * votes_per_qc
    vidx = np.concatenate([rng.choice(n_val, size=votes_per_qc, replace=False) for _ in range(n_qc)]).astype(np.uint32)
    midx = np.repeat(np.arange(n_qc, dtype=np.uint32), votes_per_qc)
    sig = eng.sign_digests(seeds, pks, digests[midx], key_idx=vidx)
    for i in rng.choice(n, size=64, replace=False):
        assert Ed25519PrivateKey.from_private_bytes(seeds[vidx[i]].tobytes()).sign(digests[midx[i]].tobytes()) == sig[i].tobytes()
    bad = rng.choice(n, size=n // 100, replace=False)
    sig[bad, rng.integers(0, 64, bad.shape[0])] ^= (1 << rng.integers(0, 8, bad.shape[0])).astype(np.uint8)
    corrupted = np.zeros(n, dtype=bool)
    corrupted[bad] = True
    return dict(pks=pks, pre=pre, digests=digests, vidx=vidx, midx=midx, sig=sig, corrupted=corrupted)


def qc_leg(eng, torch, dist, dev, rank, world, committee, qcs, votes_per_qc, steps, warmup, collective):
    """One QC-verification measurement: QC::digest for every certificate, the verify_batch condition per vote of THIS rank's
    shard, all-gather of the vote bitmaps (fused peer stores or ncclAllGather), per-QC AND over the gathered bitmap — every rank
    ends with every QC verdict.  STRONG scaling: the total number of votes is fixed.  Engine kernels only inside the timed region."""
    from hotstuff_b200.sharding import shard_range, all_gather_bitmap
    inp = make_qc_inputs(eng, committee, qcs, votes_per_qc, seed=4321)   # identical on every rank (seeded)
    n = inp["sig"].shape[0]
    lo, hi, per = shard_range(n, rank, world)
    assert eng.committee_register(inp["pks"]).all()
    d_pre = torch.from_numpy(inp["pre"].reshape(-1)).to(dev)
    d_dig = torch.empty((qcs, 32), dtype=torch.uint8, device=dev)
    d_sig = torch.from_numpy(inp["sig"][lo:hi]).to(dev)
    d_vidx = torch.from_numpy(inp["vidx"][lo:hi].astype(np.int32)).to(dev)
    d_midx = torch.from_numpy(inp["midx"][lo:hi].astype(np.int32)).to(dev)
    d_midx_all = torch.from_numpy(inp["midx"].astype(np.int32)).to(dev)
    words_local = (hi - lo + 31) // 32
    d_bm = torch.zeros(max(1, per // 32), dtype=torch.int32, device=dev)
    d_full = torch.zeros((per // 32) * world, dtype=torch.int32, device=dev)
    d_qc = torch.zeros((qcs + 31) // 32, dtype=torch.int32, device=dev)
    pag = None
    if world > 1 and collective == "peer":
        from hotstuff_b200.sharding import PeerAllGather
        try:
            pag = PeerAllGather(eng, n, rank, world)
        except RuntimeError as ex:
            if rank == 0:
                print("peer all-gather unavailable, using ncclAllGather: %s" % ex, file=sys.stderr)

    # deferred-results mode: the finish kernel (+ peer exchange) and the per-QC AND of pass i run on the engine's tail stream beside the
    # main kernel of pass i+1; hs_results_wait() closes the timed region.  (Not with ncclAllGather: the collective needs the bitmap on torch's stream.)
    deferred = world == 1 or pag is not None
    eng.set_deferred(deferred)

    def step():
        eng.digest32_fixed_dev(d_pre, 40, d_dig, qcs)                                       # QC::digest for every certificate
        if pag is not None:
            pag.arm()
        eng.verify_qc_votes_dev(d_dig, d_sig, d_midx, d_bm, hi - lo, d_vidx=d_vidx)          # verify_batch condition per vote (this shard)
        if pag is not None:
            full = pag.bitmap()
        elif world > 1:
            dist.all_gather_into_tensor(d_full, d_bm)
            full = d_full
        else:
            full = d_bm
        eng.qc_and_dev(full, d_midx_all, n, qcs, d_qc)                                      # per-QC AND over ALL votes, on every rank
        return full

    for _ in range(max(3, warmup)):
        full = step()
    if deferred:
        eng.results_wait()
    torch.cuda.synchronize()
    bits = np.unpackbits(full.cpu().numpy().view(np.uint8), bitorder="little")[:n].astype(bool)
    assert (bits == ~inp["corrupted"]).all(), "vote verdicts differ from the expected pattern"
    want_qc = np.ones(qcs, dtype=bool)
    np.logical_and.at(want_qc, inp["midx"], ~inp["corrupted"])
    got_qc = np.unpackbits(d_qc.cpu().numpy().view(np.uint8), bitorder="little")[:qcs].astype(bool)
    assert (got_qc == want_qc).all(), "per-QC AND differs"
    l0 = eng.kernel_launches
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    if deferred:
        eng.results_wait()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    wa, wb = eng.window_bits
    eng.set_deferred(False)
    return {"votes": n, "deferred_results": deferred, "committee": committee, "qcs": qcs, "votes_per_qc": votes_per_qc, "ms_per_step": ms / steps, "votes_per_s": n * steps / (ms * 1e-3),
            "gpu_launches_per_step": int(eng.kernel_launches - l0) // steps, "window_bits": {"key": wa, "base": wb}, "votes_per_rank": per,
            "collective": "none (1 rank)" if world == 1 else ("fused peer-store all-gather inside the finish kernel (NVLink P2P)" if pag is not None else "ncclAllGather"),
            "scaling": "strong"}


def run_qc(args):
    import torch
    import torch.distributed as dist
    from hotstuff_b200 import Engine, build
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    build.build_engine()
    eng = Engine(local_rank, base_window=args.base_window)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    r = qc_leg(eng, torch, dist, dev, rank, world, args.committee, args.qcs, args.votes_per_qc, args.steps, args.warmup, args.collective)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        print(json.dumps({
            "metric": "Ed25519 verifies/s", "value": r["votes_per_s"], "unit": "verifies/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "gpu_launches": r["gpu_launches_per_step"] * args.steps, "clocks": clocks,
            "config": {"workload": "QC verification: committee=%d, %d QCs x %d votes = %d votes (BASELINE config[%d]); QC::digest on GPU, "
                                   "verify_batch condition per vote, all-gather of accept bitmaps, per-QC AND" % (
                                       args.committee, args.qcs, args.votes_per_qc, r["votes"], 2 if args.committee <= 1000 else 3),
                       "votes": r["votes"], "shard": "contiguous ranges of %d votes per rank" % r["votes_per_rank"], "window_bits": r["window_bits"],
                       "collective": r["collective"],
                       "l2": "per-key tables (%d keys) far larger than L2; inputs %.0f MB" % (args.committee, r["votes"] * 72 / 1e6)}}))
    if world > 1:
        dist.destroy_process_group()
    eng.close()


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--keys", type=int, default=4096)
    ap.add_argument("--msg-len", type=int, default=512)
    ap.add_argument("--key-mode", default="committee", choices=["committee", "indexed", "generic", "cache"],
                    help="committee: the signer keys are registered once (epoch set-up, untimed); records carry 32-byte keys that the "
                         "engine resolves through its device hash table.  indexed: records carry validator indices.  generic: nothing registered, "
                         "every key is decompressed per record (key cache off).  cache: nothing registered, the engine learns the keys during warm-up")
    ap.add_argument("--ref-sample", type=int, default=1 << 18)
    ap.add_argument("--cpu-sample", type=int, default=1 << 18)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="experiments only: skip the host-pointer leg")
    ap.add_argument("--workload", default="msgs", choices=["msgs", "qc"],
                    help="msgs: BASELINE config[1] (default, the driver's headline).  qc: BASELINE config[2]/[3] — a committee of --committee "
                         "validators, --qcs quorum certificates of --votes-per-qc votes each, verify_batch semantics per vote + per-QC AND; "
                         "with --gpus N the votes are sharded across ranks (strong scaling) and the bitmaps all-gathered")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the per-rank accept bitmaps reach every rank.  peer: the verify finish kernel stores its words straight "
                         "into every rank's buffer over NVLink (fused all-gather, hs_peer_*).  nccl: ncclAllGather after the kernel (baseline)")
    ap.add_argument("--base-window", type=int, default=24,
                    help="comb window of the base-point table in bits: 24 = the library default (11 windows, 8.9 GB).  26 (10 windows, 32 GB: one "
                         "mixed addition fewer) was measured on B200 and buys nothing — 2.361 vs 2.371 ms for the main kernel — because the gathers "
                         "from the 3.6x larger table miss L2/TLB more often (profiles/r02_bench_base_window_26.json)")
    ap.add_argument("--key-window", type=int, default=0, help="force the per-key comb window (bits); 0 = widest that fits the table budget. "
                    "E.g. --base-window 20 --key-window 12 is the ~18 GB configuration for a shared GPU (DESIGN.md §5c)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling QC leg (BASELINE config[3]) reported next to the headline")
    ap.add_argument("--committee", type=int, default=1000)
    ap.add_argument("--qcs", type=int, default=10000)
    ap.add_argument("--votes-per-qc", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float32): accept.npy = the 0/1 verdict "
                         "of every record of every rank, digest.npy = rank 0's 32-byte digests (a fixed sample of rows above 2^22 values)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "msgs"):
        ap.error("--dump-outputs applies to the GPU arm's msgs workload")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "qc":
        return run_qc(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    from hotstuff_b200 import Engine, build
    if not os.environ.get("HS_CRYPTO_LIB"):
        build.build_engine()
    eng = Engine(local_rank, key_cache=(args.key_mode != "generic"), base_window=args.base_window, key_window=args.key_window)
    n, L = args.n, args.msg_len
    inp = make_inputs(n, args.keys, L, seed=1234 + rank, corrupt_frac=0.01, engine=eng)
    n_bad = int(inp["corrupted"].sum())

    # ---- resident buffers
    d_sig = torch.from_numpy(inp["sig"]).to(dev)
    d_pk = torch.from_numpy(inp["pk"]).to(dev)
    d_msgs = torch.from_numpy(inp["msgs"].reshape(-1)).to(dev)
    d_vidx = torch.from_numpy(inp["key_idx"].astype(np.int32)).to(dev)
    d_digest = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    words = (n + 31) // 32
    d_bitmap = torch.zeros(words, dtype=torch.int32, device=dev)
    d_all = torch.zeros(words * world, dtype=torch.int32, device=dev)
    if args.key_mode in ("committee", "indexed"):
        assert eng.committee_register(inp["pks"]).all()
    indexed = args.key_mode == "indexed"

    pag = None
    if world > 1 and args.collective == "peer":
        from hotstuff_b200.sharding import PeerAllGather
        try:
            pag = PeerAllGather(eng, n * world, rank, world)
        except RuntimeError as ex:     # raised on every rank together: fall back to the NCCL collective
            args.collective = "nccl"
            if rank == 0:
                print("peer all-gather unavailable, using ncclAllGather: %s" % ex, file=sys.stderr)

    def step_resident():
        if pag is not None:
            pag.arm()   # the finish kernel of the next call writes this rank's words into every rank's buffer + signals
        eng.verify_msgs_dev(d_sig, d_msgs, L, d_digest, d_bitmap, n, d_pk=None if indexed else d_pk, d_vidx=d_vidx if indexed else None)
        if world > 1 and pag is None:
            dist.all_gather_into_tensor(d_all, d_bitmap)

    def expected_bits():
        if indexed:
            # index mode ignores corrupted pk *bytes* (the registered key is used), so those records verify
            pk_ok = (inp["pk"] == inp["pks"][inp["key_idx"]]).all(axis=1)
            return ~(inp["corrupted"] & pk_ok)
        return ~inp["corrupted"]

    def check(bm_words):
        bits = np.unpackbits(bm_words.view(np.uint8), bitorder="little")[:n].astype(bool)
        assert (bits == expected_bits()).all(), "GPU verdicts differ from the expected accept pattern"

    for _ in range(args.warmup):
        step_resident()
    if args.key_mode == "cache":          # the cache learns at most 1,024 keys per call: warm up until every signer key has its table
        for _ in range(16):
            if eng.cached_keys >= args.keys:
                break
            step_resident()
    torch.cuda.synchronize()
    if world > 1:
        # every rank must hold every rank's verdicts: check this rank's slice of the gathered bitmap, and that the other
        # slices are populated (each rank's inputs differ only by seed, ~1 % rejected everywhere)
        full = (pag.full if pag is not None else d_all).cpu().numpy()
        check(full[rank * words:(rank + 1) * words].copy())
        for r in range(world):
            ones = int(np.unpackbits(full[r * words:(r + 1) * words].view(np.uint8)).sum())
            assert 0.98 * n < ones < n, "rank %d sees no plausible bitmap from rank %d" % (rank, r)
        if pag is not None:
            assert not eng.lib.hs_peer_timed_out(eng.h), "peer wait timed out"
    else:
        check(d_bitmap.cpu().numpy())

    d_arange = torch.arange(n, dtype=torch.int32, device=dev)
    d_recs = torch.empty((n, 128), dtype=torch.uint8, device=dev)
    d_recs[:, :64] = d_sig
    d_recs[:, 64:96] = d_pk
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for s_ in range(args.steps):
        step_resident()
        ev[s_ + 1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if args.dump_outputs and rank == 0:
        # taken before the kernel timings below overwrite d_bitmap and d_digest
        words_all = (pag.full if pag is not None else d_all) if world > 1 else d_bitmap
        accept = np.unpackbits(words_all.cpu().numpy().view(np.uint8).reshape(world, -1), axis=1, bitorder="little")[:, :n].reshape(-1)
        write_outputs(args.dump_outputs, accept=accept, digest=d_digest.cpu().numpy())
    total_ms = ev[0].elapsed_time(ev[-1])
    launches = eng.kernel_launches - launches0
    # dominant kernel timed on its own (same stream, CUDA events around the verify pass only: digests already computed)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern = []
    for _ in range(3):
        k0.record()
        if indexed:
            eng.verify_committee_dev(d_vidx, d_sig, d_digest, d_bitmap, n, d_midx=d_arange)
        else:
            d_recs[:, 96:] = d_digest
            k0.record()  # re-record after the untimed digest scatter
            eng.verify_rec128_dev(d_recs, d_bitmap, n)
        k1.record()
        torch.cuda.synchronize()
        kern.append(k0.elapsed_time(k1))
    kern_ms = float(np.median(kern))
    # the dominant kernel alone: CUDA events recorded by the engine around k_verify_main<committee> on the stream it is launched on
    main_ms = None
    if args.key_mode != "generic" and eng.lib.hs_profile_enable(eng.h, 1) == 0:
        ms_ = []
        for _ in range(5):
            if indexed:
                eng.verify_committee_dev(d_vidx, d_sig, d_digest, d_bitmap, n, d_midx=d_arange)
            else:
                eng.verify_rec128_dev(d_recs, d_bitmap, n)
            ms_.append(float(eng.lib.hs_profile_main_ms(eng.h)))
        eng.lib.hs_profile_enable(eng.h, 0)
        main_ms = float(np.median(ms_[1:]))
    head_wa, head_wb = eng.window_bits
    head_cached = eng.cached_keys
    dig = []
    for _ in range(3):   # the Digest kernel on its own (same stream, CUDA events)
        k0.record()
        eng.digest32_fixed_dev(d_msgs, L, d_digest, n)
        k1.record()
        torch.cuda.synchronize()
        dig.append(k0.elapsed_time(k1))
    dig_ms = float(np.median(dig))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * n * args.steps / (total_ms * 1e-3)

    # ---- end to end through the host-pointer C ABI (pinned host buffers; H2D + D2H inside the timed region)
    h_sig = torch.from_numpy(inp["sig"]).pin_memory()
    h_pk = torch.from_numpy(inp["pk"]).pin_memory()
    h_msgs = torch.from_numpy(inp["msgs"].reshape(-1)).pin_memory()
    h_vidx = torch.from_numpy(inp["key_idx"].astype(np.int32)).pin_memory()
    h_bitmap = torch.zeros(words, dtype=torch.int32).pin_memory()
    h_bytes = h_sig.numel() + h_msgs.numel() + (h_vidx.numel() * 4 if indexed else h_pk.numel())

    def step_e2e():
        rc = eng.lib.hs_verify_msgs(eng.h, h_sig.data_ptr(), None if indexed else h_pk.data_ptr(), h_vidx.data_ptr() if indexed else None,
                                    h_msgs.data_ptr(), L, n, 0, h_bitmap.data_ptr())
        assert rc == 0, eng.lib.hs_last_error(eng.h)

    for _ in range(0 if args.no_e2e else 2):
        step_e2e()
    if not args.no_e2e:
        check(h_bitmap.numpy())
    if world > 1:
        dist.barrier()
    launches_e2e0 = eng.kernel_launches
    e2e_steps = 1 if args.no_e2e else args.steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e = {"value": world * n * e2e_steps / float(t.item()), "unit": "verifies/s", "h2d_bytes_per_step": int(h_bytes), "d2h_bytes_per_step": int(words * 4),
           "api": "hs_verify_msgs (host pointers, pinned)", "gpu_launches": int(eng.kernel_launches - launches_e2e0)}
    clocks = sampler.stop() if rank == 0 else None

    # ---- CPU baseline on the box's host cores (rank 0, N = 1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle_api import Oracle
        oracle = Oracle()
        cores = host_cores()
        m = min(n, args.cpu_sample)
        cpu_reference_step(oracle, inp, 0, min(m, 2048), cores)
        dt, ok = cpu_reference_step(oracle, inp, 0, m, cores)
        assert (ok == ~inp["corrupted"][:m]).all(), "oracle disagrees with the expected accept pattern"
        cpu = {"value": m / dt, "unit": "verifies/s", "cores": cores, "kind": "port",
               "sample": "first %d records of the same workload: Digest(512 B) + verify_strict, %d pthreads, %.2f s" % (m, cores, dt)}

    # ---- strong-scaling leg next to the weak headline: BASELINE config[3] (committee 10,000, 150 QCs x 6,667 votes = 1 M votes in
    # total, sharded across the ranks, every rank ends with every verdict).  Re-registers the committee (untimed, epoch set-up).
    strong = None
    if not args.no_strong:
        strong = qc_leg(eng, torch, dist, dev, rank, world, 10000, 150, 6667, args.steps, args.warmup, args.collective)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        dom_ms = main_ms if main_ms and main_ms > 0 else kern_ms
        achieved = ALGO_BYTES_VERIFY * n / (dom_ms * 1e-3) / 1e9
        # dram__bytes_read + dram__bytes_write and pipe utilisation of the kernels from THIS round's ncu --set full capture at the same
        # 2^20 records per launch (tools/run_all_gpu.sh -> tools/ncu_traffic.py -> profiles/r02_traffic.json); not measured in this run
        tr = {}
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        except Exception:
            pass
        traffic = (tr.get("k_verify_main_bytes_per_record", 0) * n) or None
        wa, wb = head_wa, head_wb

        def ndig(w):
            r = 253 % w
            return (253 + w - 1) // w + (1 if r in (0, w - 1) else 0)
        adds = (ndig(wa) if wa else 64) + ndig(wb)
        # SASS counts of the hot loop (tools/sass_hist.py, profiles/r02_sass_mainloop.txt): per mixed addition 336 IMAD.WIDE.U32.X (carry-in form,
        # measured issue rate 32 lanes/clk/SM) + 171 IMAD.WIDE.U32 (54 lanes/clk/SM) + 129 other FMA-pipe instructions (64 lanes/clk/SM)
        fma_clk_per_add = 336 / 32.0 + 171 / 54.0 + 129 / 64.0          # SM-clocks of FMA-pipe time per mixed addition per lane-group
        sm_clk = (clocks or {}).get("sm_mhz") or 1965.0
        fma_floor_ms = adds * fma_clk_per_add * n / (148 * sm_clk * 1e6) * 1e3 if wa else None
        fe_muls = adds * 7 + 10 + (0 if wa else 252 * (3 + 4 * 0.7) + 64 * 8 + 254 * 0.7 + 20)
        line = {
            "metric": "Ed25519 verifies/s", "value": value, "unit": "verifies/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic", "config": workload_config(args, world), "gpu_launches": int(launches), "clocks": clocks,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "kernel": "k_verify_main<committee>" if args.key_mode != "generic" else "k_verify_main<generic>", "cached_keys": head_cached,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s", "traffic": traffic,
                         "traffic_source": "profiles/r02_traffic.json: ncu --set full of this round at 2^20 records per launch (dram__bytes_read.sum + dram__bytes_write.sum); "
                                           "table gathers, by design ~41x the algorithmic bytes" if traffic else None,
                         "kernel_ms": dom_ms, "kernel_ms_covers": "k_verify_main<committee> alone (CUDA events recorded by the engine on its launch stream)" if main_ms else
                                                                    "lookup + main + finish kernels of one verify pass",
                         "verify_pass_ms": kern_ms, "verify_pass_covers": "lookup + main + finish kernels over 2^20 resident records",
                         "digest_kernel_ms": dig_ms, "digest_algorithmic_GBps": ALGO_BYTES_DIGEST * n / (dig_ms * 1e-3) / 1e9,
                         "digest_alu_pipe_pct_ncu": tr.get("k_digest32_fixed_alu_pipe_pct"),
                         "algorithmic_bytes_per_verify": ALGO_BYTES_VERIFY,
                         "note": "integer-ALU bound path: 128 B of compulsory I/O per ~30 k INT32 instructions; the HBM fraction is necessarily << 1 (SURVEY §0.7): "
                                 "see alu_roofline for the resource that binds"},
            "alu_roofline": {"bound": "integer-multiply (FMA-heavy / IMAD) pipe — the resource that actually binds k_verify_main",
                             "fmaheavy_pipe_busy_pct_ncu": tr.get("k_verify_main_fmaheavy_pipe_pct"),
                             "fmaheavy_source": "profiles/r02_traffic.json (sm__pipe_fmaheavy_cycles_active, this round's ncu capture at 2^20 records)",
                             "issue_floor_ms": fma_floor_ms, "issue_floor_frac": (fma_floor_ms / dom_ms) if fma_floor_ms else None,
                             "issue_floor_basis": "mixed additions x (336 IMAD.WIDE.X / 32 + 171 IMAD.WIDE / 54 + 129 other / 64 lanes per clk per SM): raw issue "
                                                  "rates from profiles/r01_pipes.txt and r01_widex.txt, instruction counts from profiles/r02_sass_mainloop.txt",
                             "field_muls_per_s": fe_muls * n / (dom_ms * 1e-3), "field_mul_microbench_peak": 1.138e11,
                             "field_mul_frac": fe_muls * n / (dom_ms * 1e-3) / 1.138e11,
                             "field_mul_peak_source": "best fe_mul rate of tools/microbench/febench.cu on this GPU (profiles/r01_febench.txt, 2,048 threads/SM)",
                             "field_muls_per_verify": fe_muls, "mixed_additions_per_verify": adds, "window_bits": {"key": wa, "base": wb}},
            "cpu_baseline": cpu,
            "strong_scaling_config3": strong,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    eng.close()


if __name__ == "__main__":
    main()
