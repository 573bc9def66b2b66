#!/usr/bin/env python
"""Benchmark: EmailVerifier proofs/sec (witness + Groth16 prove) on B200 - BASELINE.json's metric.

Workload (config.workload): BASELINE.json configs[2] - a batch of 64 synthetic 1024-byte-body emails, default circuit
EmailVerifier(1024, 1536, 121, 17), full witness + Groth16 prove (N = 2^22 H multi-exponentiation + six 2^22 NTTs per
proof).  One "step" = one pass of the hot path over one batch.  With N GPUs every rank proves its own batch of 64
(weak scaling, no data-path collective - SURVEY 8(e)(i)); the ranks only meet at the timing barrier.

  value  : whole-job proofs/s with the packed inputs already resident in HBM when the timed region starts
  e2e    : the same through the C-ABI with pinned HOST buffers (H2D of inputs, D2H of proofs inside the timed region)
  Both arms drive the K timed steps through the pipelined form of fullprove (zke_fullprove_submit / _collect, at most
  two batches in flight): the latency-bound witness kernel of step k + 1 runs under the proving kernels of step k.
  Every step's witness + proving work, its copies and its host tail lie inside the timed region.
  roofline: the dominant kernel (bucket accumulation of the H multi-exponentiation) timed live with CUDA events;
            achieved = algorithmic bytes (N x (64-byte point + 32-byte scalar), SURVEY 8(d)) / kernel time vs the
            measured HBM copy peak.  The kernel is bound by the integer (IMAD) pipe, not HBM - see DESIGN.md.
  cpu_baseline: the CPU oracle port (oracle/zkref_*.c, all host threads) timed on ONE email of the same workload.
  The inputs are seeded (RSA signing key, emails, proving key, blinding scalars r and s): the proofs repeat from run to
  run, and `--dump-outputs DIR` writes those of the last timed step as .npy files for comparing two builds.

`--impl reference` times that CPU path alone (the reference's snarkjs/circom stack is not runnable offline - DESIGN.md).
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "zk-email-verify_b200", "host"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

BATCH = 64
CIRCUIT = ("EmailVerifier", [1024, 1536, 121, 17])
KEY_SEED = 20260923


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag = gpu_index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def make_inputs(z, circuit, count, key):
    packed = []
    for i in range(count):
        em = z.synthetic.make_signed_email(i, key)
        dk = z.verify_dkim_signature(em, resolver=lambda n, t: [z.synthetic.key_record(key)])
        packed.append(circuit.pack_inputs(z.generate_email_verifier_inputs_from_dkim_result(dk)))
    return packed


def dump_outputs(out_dir, proofs, publics, status, batch, npub):
    """What one fullprove step returns, as .npy files: every 256-bit field element as its eight little-endian 32-bit
    limbs in float64 (exact), so that the outputs of two builds can be compared element for element.
      proofs.npy  [batch, 8, 8]     A.x, A.y, B.x.c0, B.x.c1, B.y.c0, B.y.c1, C.x, C.y of each proof
      publics.npy [batch, npub, 8]  public signals
      status.npy  [batch]           -1 = constraints satisfied, else the first violated constraint"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def limbs(raw, shape):
        return np.frombuffer(raw, dtype="<u4").reshape(shape).astype(np.float64)

    np.save(os.path.join(out_dir, "proofs.npy"), limbs(proofs, (batch, 8, 8)))
    np.save(os.path.join(out_dir, "publics.npy"), limbs(publics, (batch, npub, 8)))
    np.save(os.path.join(out_dir, "status.npy"), np.asarray(status, dtype=np.float64))


def cpu_reference_proof(z, circuit, zk, packed_one, threads, rs=None):
    """One witness + Groth16 proof on the host cores with the CPU oracle; returns (seconds, proof bytes, witness)."""
    import zkutil
    sec = zkutil.product_sections(zk)          # key material: generated once by the setup, not part of the timed path
    rc = zkutil.ref_view(circuit)
    total = circuit.info.n_vars + circuit.info.n_temps
    wbuf = ctypes.create_string_buffer(32 * total)
    r, s = rs if rs else (12345, 67890)
    t0 = time.perf_counter()
    assert zkutil.ref.zkref_witness(ctypes.byref(rc), packed_one, wbuf) == 0
    assert zkutil.ref.zkref_check_r1cs(ctypes.byref(rc), wbuf) < 0
    proof = zkutil.oracle_prove(circuit, sec, wbuf.raw[: 32 * circuit.info.n_vars], r, s, threads=threads)
    dt = time.perf_counter() - t0
    return dt, proof, wbuf.raw[: 32 * circuit.info.n_vars]


def extra_configs(z, torch, dist, rank, local_rank, world, key):
    """Driver-visible numbers for the other GPU configurations of BASELINE.json (not part of `value`).  Every rank proves
    its own share (batch parallelism, as the headline); with N > 1 one proof of the config-[4] circuit is also computed
    by all ranks together (zkemail_b200.parallel.prove_sharded: NCCL all-to-all + all-gather) and compared bit for bit
    with the single-GPU proof."""
    out = {}

    def sync_max(dt):
        if dist is None:
            return dt
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def measure(label, template, params, batch, steps, make_packed, want):
        circuit = z.Circuit(template, params)
        zk = z.Zkey(circuit, seed=KEY_SEED + len(params) + batch, device=local_rank)
        ctx = z.Context(circuit, zk, device=local_rank, max_batch=batch)
        packed_list = [make_packed(circuit, i) for i in range(batch)]
        packed = b"".join(packed_list)
        ctx.fullprove(packed, batch)                                # warm-up
        barrier()
        t0 = time.perf_counter()
        ctx.submit(packed, batch)
        for _ in range(steps - 1):
            ctx.submit(packed, batch)
            ctx.collect()
        proofs, publics, status = ctx.collect()
        dt = sync_max(time.perf_counter() - t0)
        npub = circuit.info.n_public
        proof, pubs = z.proof_to_json(proofs[:256], publics[: 32 * npub], npub)
        ok = status == [-1] * batch and z.verify(zk.vkey(), pubs, proof)
        out[label] = {"workload": want, "n_gpus": world, "batch_per_gpu": batch, "steps": steps, "proofs_per_s": world * batch * steps / dt,
                      "ms_per_step": 1e3 * dt / steps, "n_constraints": circuit.info.n_constraints, "domain": "2^%d" % circuit.info.domain_log2,
                      "proofs_verify": bool(ok), "parallelism": "batch-dp%d" % world}
        return circuit, zk, ctx, packed_list

    def email_inputs(maxh, maxb, body_len):
        def f(circuit, i):
            em = z.synthetic.make_signed_email(1000 + i, key, body_len=body_len)
            dk = z.verify_dkim_signature(em, resolver=lambda n, t: [z.synthetic.key_record(key)])
            return circuit.pack_inputs(z.generate_email_verifier_inputs_from_dkim_result(dk, {"maxHeadersLength": maxh, "maxBodyLength": maxb}))
        return f

    def twitter_inputs(circuit, i):
        em = z.synthetic.make_signed_email(2000 + i, key, marker="This email was meant for @user%04d" % i)
        dk = z.verify_dkim_signature(em, resolver=lambda n, t: [z.synthetic.key_record(key)])
        return circuit.pack_inputs(z.generate_twitter_verifier_inputs_from_dkim_result(dk, 0x1234567890ABCDEF1234567890ABCDEF12345678 + i))

    # the headline statement on the optimised front end: EmailVerifier(1024, 1536) with the compact regex shape (regex.cpp) is
    # the same relation over the same public signals in 1.78 M constraints, so its Groth16 domain is 2^21.  Reported beside
    # the headline, not as it: configs[2] names the 2^22 domain of the zk-regex-shaped circuit.
    _, zkc, ctxc, packed_c = measure("config2_compact_regex", "EmailVerifier", [1024, 1536, 121, 17, 0, 0, 0, 0, 0, 1], 64, 4, email_inputs(1024, 1536, 1024),
                              "configs[2]'s statement (EmailVerifier default parameters, batch 64 per GPU, witness + prove) with the compact "
                              "regex circuit shape: same public signals, domain 2^21 instead of 2^22")
    lat = []
    for _ in range(5):                                               # single-email fullProve on the same context, host buffers, wall clock
        t0 = time.perf_counter()
        ctxc.fullprove(packed_c[0], 1)
        lat.append(1e3 * (time.perf_counter() - t0))
    out["config2_compact_regex"]["single_email_fullprove_latency_ms"] = sorted(lat)[len(lat) // 2]
    ctxc.close()
    del ctxc, zkc
    if world in (1, 4):
        _, zk4, ctx4, _ = measure("config3_twitter", "TwitterVerifier", [1024, 1536, 121, 17], 64, 2, twitter_inputs,
                                  "configs[3]: Proof-of-Twitter circuit (EmailVerifier + body regex + packing + address), batch 256 over 4 "
                                  "GPUs = 64 per GPU; proofs sharded across GPUs (no intra-proof exchange at this size)")
        ctx4.close()
        del ctx4, zk4
        _, zk4, ctx4, _ = measure("config3_twitter_compact_regex", "TwitterVerifier", [1024, 1536, 121, 17, 1], 64, 2, twitter_inputs,
                                  "configs[3]'s statement with the compact regex circuit shape (header and body regex): domain 2^21 instead of 2^22")
        ctx4.close()
        del ctx4, zk4
    if world in (1, 2, 8):
        circuit5, zk5, ctx5, packed5 = measure("config4_body16384", "EmailVerifier", [1024, 16384, 121, 17], 8, 2, email_inputs(1024, 16384, 12288),
                                               "configs[4]: EmailVerifier(1024, 16384) - 10.2 M constraints, domain 2^24 - batch 8 per GPU "
                                               "(1024 over 8 GPUs = 128 per GPU in sub-batches of 8)")
        if dist is not None and world in (2, 4, 8):
            from zkemail_b200.parallel import prove_sharded
            rs = (0xA5A5A5A5).to_bytes(32, "little") + (0x5A5A5A5A5A).to_bytes(32, "little")
            one = [packed5[0]]
            dist.broadcast_object_list(one, src=0)                       # every rank proves rank 0's email
            prove_sharded(ctx5, one[0], rs)                              # warm-up: NCCL communicators, buffers
            barrier()
            t0 = time.perf_counter()
            proof_sh, pub_sh, _ = prove_sharded(ctx5, one[0], rs)
            torch.cuda.synchronize()
            dt_sh = sync_max(time.perf_counter() - t0)
            # the proving part alone (the witness resident on every GPU): what the sharding actually divides
            ctx5.witness(one[0], 1, want_witness=False)
            barrier()
            t0 = time.perf_counter()
            prove_sharded(ctx5, None, rs)
            torch.cuda.synchronize()
            dt_sh_prove = sync_max(time.perf_counter() - t0)
            same = None
            dt_1 = dt_1_prove = None
            if rank == 0:
                ctx5.witness(one[0], 1, want_witness=False)
                t1 = time.perf_counter()
                ctx5.witness(one[0], 1, want_witness=False)
                t2 = time.perf_counter()
                proof_1, pub_1, _ = ctx5.prove(1, rs)
                dt_1, dt_1_prove = time.perf_counter() - t1, time.perf_counter() - t2
                same = proof_1 == proof_sh and pub_1 == pub_sh
            n = 1 << circuit5.info.domain_log2
            out["sharded_proof"] = {"workload": "ONE proof of the configs[4] circuit computed by all %d GPUs together (4-step NTT split, "
                                                "point-sharded multi-exponentiations)" % world, "n_gpus": world,
                                    "latency_ms": 1e3 * dt_sh, "single_gpu_latency_ms": None if dt_1 is None else 1e3 * dt_1,
                                    "prove_only_latency_ms": 1e3 * dt_sh_prove,
                                    "single_gpu_prove_only_latency_ms": None if dt_1_prove is None else 1e3 * dt_1_prove,
                                    "bit_identical_to_single_gpu": same,
                                    "collectives": {"all_to_all_bytes_per_gpu_total": 6 * 32 * (n // world) * (world - 1) // world,
                                                    "all_gather_bytes_per_gpu": 388,
                                                    "limiting": "no collective (each all-to-all moves < 60 MB per GPU over NVLink): the witness kernel is replicated "
                                                                "(latency_ms - prove_only_latency_ms, a dependency chain more GPUs cannot shorten) and the proving part "
                                                                "is a chain of short kernels with two host round trips between the three engine steps"}}
        ctx5.close()
        del ctx5, zk5
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extra-configs", action="store_true",
                    help="do not measure BASELINE configs[3] / configs[4] / the sharded proof after the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (proofs, public signals, status) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" and rank != 0:
        return 0

    import torch
    import zkemail_b200 as z
    if not torch.cuda.is_available() or z.device_count() == 0:
        print(json.dumps({"error": "no CUDA device: this benchmark has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1 and args.impl == "b200":
        import datetime
        import torch.distributed as dist
        # a bounded collective timeout: a rank that fails inside the optional extras must not hang the others for ever
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=600))

    circuit = z.Circuit(*CIRCUIT)
    info = circuit.info
    N = 1 << info.domain_log2
    host_threads = os.cpu_count() or 1
    key = z.synthetic.generate_key(seed=KEY_SEED)
    zk = z.Zkey(circuit, seed=KEY_SEED, device=local_rank)
    config = {"workload": "configs[2]: batch of %d synthetic 1024-byte-body emails per GPU, EmailVerifier(1024,1536,121,17), "
                          "witness + full Groth16 prove" % args.batch,
              "batch_per_gpu": args.batch, "n_constraints": info.n_constraints, "n_vars": info.n_vars,
              "domain": "2^%d" % info.domain_log2, "parallelism": "batch-dp%d" % world,
              "l2": "working set per step (>= 4.9 GB of witnesses + 1.3 GB key) exceeds the 126 MB L2"}

    if args.impl == "reference":
        packed = make_inputs(z, circuit, 1, key)
        times = []
        for it in range(args.warmup + args.steps):
            dt, _, _ = cpu_reference_proof(z, circuit, zk, packed[0], host_threads)
            if it >= args.warmup:
                times.append(dt)
        total = sum(times)
        val = len(times) / total
        line = {"impl": "reference", "metric": "EmailVerifier proofs/sec (witness+prove)", "value": val, "unit": "proofs/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u256 (BN254 Fr/Fq integers)",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": host_threads, "kind": "port",
                                 "sample": "1 email (witness + prove) per step; CPU oracle port of the snarkjs algorithm - "
                                           "node/circom/snarkjs are not installable offline"},
                "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    batch = args.batch
    ctx = z.Context(circuit, zk, device=local_rank, max_batch=batch)
    packed_list = make_inputs(z, circuit, batch, key)
    packed = b"".join(packed_list)
    # pinned host staging for the e2e arm
    pinned_in = torch.empty(len(packed), dtype=torch.uint8).pin_memory()
    pinned_in.copy_(torch.frombuffer(bytearray(packed), dtype=torch.uint8))
    npub = info.n_public
    pinned_proofs = torch.empty(256 * batch, dtype=torch.uint8).pin_memory()
    pinned_pub = torch.empty(max(1, 32 * npub * batch), dtype=torch.uint8).pin_memory()
    status = (ctypes.c_int32 * batch)()
    err = ctypes.create_string_buffer(4096)
    L = z._lib
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    # seeded blinding scalars (r, s) of every proof, in place of fresh randomness: the proofs repeat from run to run
    blinding = b"".join((int.from_bytes(hashlib.sha256(b"bench %d %d" % (KEY_SEED, j)).digest(), "little") % z.FR_MODULUS).to_bytes(32, "little")
                  for j in range(2 * batch))

    def step(inputs_ptr):
        rc = L.zke_fullprove(ctx.handle, inputs_ptr, batch, blinding, pinned_proofs.data_ptr(), pinned_pub.data_ptr(), status, err, 4096)
        if rc != 0:
            raise RuntimeError("zke_fullprove failed: %d %s" % (rc, err.value.decode()))

    def submit(inputs_ptr):
        if L.zke_fullprove_submit(ctx.handle, inputs_ptr, batch, blinding, err, 4096) != 0:
            raise RuntimeError("zke_fullprove_submit failed: %s" % err.value.decode())

    def collect():
        rc = L.zke_fullprove_collect(ctx.handle, pinned_proofs.data_ptr(), pinned_pub.data_ptr(), status, err, 4096)
        if rc != 0:
            raise RuntimeError("zke_fullprove_collect failed: %d %s" % (rc, err.value.decode()))

    def pipelined(inputs_ptr, steps):
        submit(inputs_ptr)
        for _ in range(steps - 1):
            submit(inputs_ptr)
            collect()
        collect()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(inputs_ptr, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        pipelined(inputs_ptr, steps)
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    # ---- device-resident arm (value)
    ctx.upload_inputs(packed, batch)
    for _ in range(args.warmup):
        step(None)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.zke_kernel_launches()
    ms_value = timed(None, args.steps)
    launches = L.zke_kernel_launches() - launches0
    # ---- end-to-end arm (host buffers through the C ABI)
    for _ in range(1):
        step(pinned_in.data_ptr())
    ms_e2e = timed(pinned_in.data_ptr(), args.steps)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    pr_raw, pb_raw = bytes(pinned_proofs.numpy()), bytes(pinned_pub.numpy())[: 32 * npub * batch]
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, pr_raw, pb_raw, list(status), batch, npub)
    # ---- every proof of the last end-to-end batch is verified (outside the timed region): the batch verifier checks them
    #      with one randomised product of pairings and falls back to one-by-one to name offenders
    proofs_verified = None
    if rank == 0:
        try:
            t0 = time.perf_counter()
            items = [z.proof_to_json(pr_raw[256 * k: 256 * (k + 1)], pb_raw[32 * npub * k: 32 * npub * (k + 1)], npub) for k in range(batch)]
            oks = z.verify_batch(zk.vkey(), [it[1] for it in items], [it[0] for it in items])
            proofs_verified = {"n": batch, "valid": int(sum(oks)), "status_ok": all(int(x) == -1 for x in status),
                               "how": "zke_verify_batch_json: n + 3 Miller loops, one final exponentiation (host)",
                               "ms": 1e3 * (time.perf_counter() - t0)}
        except Exception as e:
            proofs_verified = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    # ---- roofline pass: one extra step with per-stage CUDA events (single lane: no overlap, so the dominant kernel is
    #      timed alone on its launching stream); not part of `value`
    ctx.profile(True)
    step(None)
    prof = ctx.profile_get()
    ctx.profile(False)
    # ---- extra lines (not part of `value`): BASELINE configs[1] = witness generation only for the same batch, and the
    #      latency of a single-email fullProve (the reference's generateProof is a one-email call)
    extra = {}
    if rank == 0:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            rc = L.zke_witness(ctx.handle, None, batch, None, status, err, 4096)
            if rc != 0:
                raise RuntimeError("zke_witness failed: %s" % err.value.decode())
        dtw = (time.perf_counter() - t0) / reps
        lat = []
        one_in = pinned_in.data_ptr()
        for _ in range(5):
            t0 = time.perf_counter()
            rc = L.zke_fullprove(ctx.handle, one_in, 1, None, pinned_proofs.data_ptr(), pinned_pub.data_ptr(), status, err, 4096)
            if rc != 0:
                raise RuntimeError("zke_fullprove failed: %s" % err.value.decode())
            lat.append(time.perf_counter() - t0)
        lat.sort()
        extra = {"config1_witness_only": {"workload": "configs[1]: batch of %d, calculateWitness + checkConstraints (zke_witness), inputs resident" % batch,
                                          "emails_per_s": batch / dtw, "ms_per_batch": 1e3 * dtw,
                                          "witness_kernel_ms_per_batch": prof["witness"]["ms"] / max(1, prof["witness"]["count"])},
                 "single_email_fullprove_latency_ms": {"median": 1e3 * lat[len(lat) // 2], "min": 1e3 * lat[0],
                                                       "what": "zke_fullprove(batch = 1) with host buffers, wall clock"}}
    cpu_baseline = None
    if rank == 0 and not args.skip_cpu_baseline:
        dt, proof_cpu, _ = cpu_reference_proof(z, circuit, zk, packed_list[0], host_threads, rs=(12345, 67890))
        # same email, same (r, s) on the GPU: full-size bit-exact parity check on the side
        rs = (12345).to_bytes(32, "little") + (67890).to_bytes(32, "little")
        ctx.witness(packed_list[0], 1, want_witness=False)
        proofs_gpu, _, _ = ctx.prove(1, rs)
        cpu_baseline = {"value": 1.0 / dt, "unit": "proofs/s", "cores": host_threads, "kind": "port",
                        "sample": "1 email of the workload (witness + full prove), %.1f s" % dt,
                        "gpu_proof_bit_exact": proofs_gpu[:256] == proof_cpu}

    # ---- BASELINE configs[3] (Proof-of-Twitter circuit, 4 GPUs) and configs[4] (maxBodyLength 16384, domain 2^24, 8 GPUs):
    #      batch-parallel throughput of each rank's share, and ONE config-[4] proof sharded across all ranks (N > 1)
    other = {}
    if not args.skip_extra_configs:
        ctx.close()
        del ctx, zk
        try:
            other = extra_configs(z, torch, dist, rank, local_rank, world, key)
        except Exception as e:          # the headline line must survive a failure of the optional measurements
            other = {"extra_configs_error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
        dist = None

    if rank != 0:
        return 0
    extra.update(other)

    proofs_total = world * batch * args.steps
    value = proofs_total / (ms_value / 1e3)
    e2e_value = proofs_total / (ms_e2e / 1e3)
    peaks, peak_kind = load_peaks()
    hb = prof["msm_h_buckets"]
    kernel_ms = hb["ms"] / max(1, hb["count"])
    alg_bytes = N * (64 + 32)
    achieved = alg_bytes / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else 0.0
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed `ncu --set full` capture
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            t = json.load(f)
        traffic = float(t["dram_bytes_read"]) + float(t["dram_bytes_write"])
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "chunk_sum_kernel<Fq> (H MSM bucket accumulation, 2^%d points)" % info.domain_log2,
                "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "peak_source": peak_kind, "traffic": traffic, "kernel_ms": kernel_ms, "algorithmic_bytes": alg_bytes,
                "note": "bound by the integer multiply pipe, not HBM: 13 windows x ~10 Fq products per 64-byte point "
                        "(fmaheavy pipe 85 % busy in the ncu capture); traffic = 13 table levels gathered at 64 B per "
                        "entry, see DESIGN.md section 5"}
    # the pipe that actually bounds the kernel: integer multiply (IMAD.WIDE).  achieved = executed fmaheavy warp
    # instructions of one launch (ncu capture, profiles/roofline_traffic.json) / live kernel time; peak = the measured
    # IMAD.WIDE rate of this GPU inside the Montgomery product (scripts/field_peaks.cu -> profiles/field_peaks_r02.json)
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            t = json.load(f)
        with open(os.path.join(ROOT, "profiles", "field_peaks_r02.json")) as f:
            pk = json.load(f)["results"]["mul_cios"]["giga_warp_imad_wide_per_s"]
        ach = float(t["fmaheavy_warp_instr"]) / (kernel_ms / 1e3) / 1e9
        roofline["imad"] = {"achieved": ach, "peak": pk, "unit": "G warp-IMAD.WIDE/s", "frac": ach / pk,
                            "warp_instr_per_launch": float(t["fmaheavy_warp_instr"])}
    except Exception:
        roofline["imad"] = None
    stages = {k: (v["ms"] / max(1, v["count"])) for k, v in prof.items()}

    line = {"metric": "EmailVerifier proofs/sec (witness+prove)", "value": value, "unit": "proofs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u256 (BN254 Fr/Fq integers, 8x32-bit limbs)", "data": "synthetic",
            "config": config, "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "proofs/s", "h2d_bytes_per_step": len(packed),
                    "d2h_bytes_per_step": 256 * batch + 32 * npub * batch + 4 * batch},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "stage_ms": stages, "proofs_verified": proofs_verified, "extra": extra,
            "pipelining": "steps driven through zke_fullprove_submit/_collect, <= 2 batches in flight"}
    cc = (extra or {}).get("config2_compact_regex") if isinstance(extra, dict) else None
    if cc:
        # NOT the headline (`value` is the 2^22-domain circuit BASELINE configs[2] names): the same statement compiled with
        # the compact regex shape of the front end, whose Groth16 domain is 2^21 - what a deployment would choose
        line["compact_circuit"] = {"value": cc["proofs_per_s"], "unit": "proofs/s", "domain": cc["domain"], "n_constraints": cc["n_constraints"],
                                   "proofs_verify": cc["proofs_verify"], "see": "extra.config2_compact_regex, DESIGN.md section 2"}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
