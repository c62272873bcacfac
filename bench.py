#!/usr/bin/env python3
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

A "step" is one pass of the hot path over one batch of synthetic input:
  * headline (`value`): best_multiexp over 2^20 (scalar, base) pairs per GPU on Pallas
    (BASELINE.json configs[2]; for N > 1 each rank owns its own contiguous 2^20-pair shard --
    weak scaling -- and the per-rank 96-byte partial points are all-gathered over NCCL and summed,
    SURVEY.md section 8(e)).  Inputs are resident in HBM when the timed region starts.
  * `extra.ntt`: best_fft at 2^20 over Fp (configs[1]; single GPU by the north star).
  * `e2e`: the same MSM through the reference-facing C-ABI call h2_msm with HOST (pinned)
    buffers -- H2D of scalars + bases and D2H of the result inside the timed region.
  * `roofline`: the dominant kernel (msm_accum0_kernel), algorithmic bytes (96 B per pair,
    SURVEY.md section 8(d)) / its CUDA-event duration measured live, against the measured HBM peak.
  * `cpu_baseline`: the C restatement of the reference algorithm (oracle/halo2_oracle.c, "port":
    the Rust reference cannot be built here) on all host cores, same workload (N = 1 only).
  * more single-GPU side measurements under `extra` (N = 1 only, each next to the C restatement): `create_proof_k14_replay`
    (the prover's hot-path call schedule, SURVEY.md Appendix C), `resident_column_k14`, `params_lagrange_k14` (Params::new's
    EC-FFT), `poly_reductions_k14` (eval_polynomial / kate_division), `quotient_pipeline_k14` (coeff_to_extended -> Ast ->
    divide_by_vanishing_poly -> extended_to_coeff on resident polynomials), `create_proof_k14_replay.verify` (the verifier's side of the
    same proof: multiopen MSM, the opening, compute_s on the device, one multiexp over the resident generators),
    `golden_proofs_verify_k11` (the reference's fifteen stored k = 11 proofs verified through the engine under their pinned keys),
    `create_proof_k14_real` (a real proof of the reference's benchmark circuit through the engine's API, verified through the engine).

`--impl reference` times that CPU restatement alone (the reference arm).
`--dump-outputs DIR` writes what the last timed step computed, from inputs that are the same on every run, so that two builds
can be compared output for output.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = 20
SEED = 0x48414C4F32
CURVE, SCALAR_FIELD = "pallas", "fq"
MSM_BYTES_PER_PAIR = 96      # 32 B scalar + 64 B affine base, each read once (SURVEY.md 8(d))
NTT_BYTES_PER_ELEM = 64      # 32 B read + 32 B written, one ideal pass

Q_MOD = 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001
P_MOD = 0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, arrays):
    """Writes each named array of 32-byte canonical field elements as out_dir/<name>.npy: float64, one column per
    little-endian 32-bit limb (float64 holds every limb exactly, so two runs compare bit for bit)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.uint8).view("<u4").astype(np.float64))


def rand_canonical_scalars(torch, n, seed, device):
    """n uniform-ish canonical scalars (< 2^254 < modulus) as an (n, 8) int32 tensor."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randint(-2**31, 2**31 - 1, (n, 8), dtype=torch.int32, device=device, generator=g)
    x[:, 7] &= 0x3FFFFFFF
    return x


# =================================================================================================
# reference arm: the reference's CPU algorithm (C restatement) on the host cores
# =================================================================================================
def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import cref
    n = 1 << LOG_N
    threads = os.cpu_count() or 1
    kb = cref.gen_scalars(SCALAR_FIELD, SEED + 3, n)
    pb = cref.gen_points(CURVE, SEED + 33, n)
    for _ in range(min(args.warmup, 1)):
        cref.best_multiexp(CURVE, kb, pb, threads)
    t0 = time.time()
    for _ in range(args.steps):
        got = cref.best_multiexp(CURVE, kb, pb, threads)
    dt = (time.time() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"msm": got.reshape(2, 32)})
    value = n / dt
    sample = f"{args.steps} x full 2^{LOG_N}-pair best_multiexp (window-parallel, c=ceil(ln n)=14, 19 window tasks)"
    line = {
        "impl": "reference", "metric": "msm_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (255-bit modular integers)", "data": "synthetic",
        "config": {"workload": f"best_multiexp 2^{LOG_N} pairs, Pallas (configs[2]), CPU restatement of arithmetic.rs:143-180"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# =================================================================================================
# create_proof k=14 schedule replay (SURVEY.md Appendix C): the hot-path CALLS the unchanged prover
# makes for the benches/plonk.rs circuit (3 advice, 4 fixed, 3-column permutation, degree 5 =>
# ext_k = 16; Vesta, Fp scalars), in order, through the reference-facing host API.  It is a replay,
# not the Rust prover (no Rust toolchain here): witness synthesis, the h(X) evaluator, transcript,
# the IPA generator fold and the 2-term MSMs stay on the CPU in the real prover and are not timed.
# =================================================================================================
PROVER_K, PROVER_J = 14, 5


def prover_replay(h2, cref, threads, reps=3, k=None):
    """create_proof k=14 (BASELINE configs[3]) as a proof-shaped replay with the reference's Blake2b transcript in both arms
    (tests/prover_replay.py): the GPU arm through the reference-facing API on device-resident polynomials, wall-clock per
    proof including the Python glue and the host-side transcript; the CPU arm through the C restatement, counting ONLY its
    hot-path calls (commits, transforms, eval_polynomial, kate_division, the IPA loop).  The proof bytes of the two arms are
    compared: every commitment, evaluation and opening round enters the transcript and every challenge feeds back."""
    from oracle import pasta
    from tests import prover_replay as R
    k = PROVER_K if k is None else k
    n = 1 << k
    pts = cref.gen_points("vesta", SEED + 50, n + 2)           # g || w || u: seeded stand-ins (a real Params::new(14) hashes 2^14 messages)
    g, w, u = pts[:n], pts[n:n + 1], pts[n + 1:n + 2]
    gl = h2.lagrange_generators("vesta", k, g)                 # g_lagrange as Params::new derives it (EC-iFFT on the device)
    inp = R.replay_inputs(cref, k, SEED + 14)
    omega = pasta.omega_for_k("fp", k)
    t0 = time.time()
    gpu = R.GpuArm(h2, k, g, gl, w, u)
    setup_s = time.time() - t0
    try:
        proof = R.run(gpu, inp, k, omega)                      # warm-up: pools, twiddles, graph capture
        gpu.free()
        R.run(gpu, inp, k, omega)
        gpu.free()
        t0 = time.time()
        for _ in range(reps):
            proof_t = R.run(gpu, inp, k, omega)
            gpu.free()
        gdt = (time.time() - t0) / reps
        # the verifier's side of the same proof (tests/prover_replay.verify): multiopen MSM from the proof's commitments, the opening,
        # ONE multiexp over all 2^k generators with compute_s built on the device -- against the resident table the prover used
        gver = R.GpuVerifierArm(h2, k, g, gl, w, u, params=gpu.params)
        v_ok = R.verify(gver, proof, k, omega)                 # warm-up
        t0 = time.time()
        for _ in range(reps):
            v_ok = R.verify(gver, proof_t, k, omega) and v_ok
        vdt = (time.time() - t0) / reps
        bad = bytearray(proof)
        bad[len(bad) - 40] ^= 1                                # one bit of c
        v_rej = not R.verify(gver, bytes(bad), k, omega)
        # per-kind attribution: one more pass with a device sync after every arm call (perturbs the total; not the headline)
        by_kind = {}
        class Timed:
            def __init__(self, arm): self.arm = arm
            def __getattr__(self, name):
                f = getattr(self.arm, name)
                if name in ("sync", "free", "close") or not callable(f):
                    return f
                def wrap(*a, **kw):
                    t1 = time.time()
                    r = f(*a, **kw)
                    self.arm.sync()
                    key = {"commit": "commit", "l2c": "lagrange_to_coeff", "c2e": "coeff_to_extended", "e2c": "extended_to_coeff",
                           "evals": "eval_polynomial", "kate": "kate_division", "ipa": "ipa"}.get(name, "glue (uploads, Ast programs, copies)")
                    by_kind[key] = by_kind.get(key, 0.0) + (time.time() - t1) * 1e3
                    return r
                return wrap
        R.run(Timed(gpu), inp, k, omega)
    finally:
        gpu.close()
    cpu = R.CpuArm(cref, pasta, k, g, gl, w, u, threads)
    # parallelize() (arithmetic.rs:345-362) falls back to ONE chunk when len / threads < threads, which serialises
    # parallel_generator_collapse on a many-core host: give the CPU arm's IPA its best thread count
    cpu.ipa_threads = min(threads, 16)
    t0 = time.time()
    proof_c = R.run(cpu, inp, k, omega)
    cpu_wall = time.time() - t0
    cver = R.CpuVerifierArm(cref, pasta, k, g, gl, w, u, threads)
    t0 = time.time()
    cv_ok = R.verify(cver, proof_c, k, omega)
    cver_wall = time.time() - t0
    verify = {"metric": "ms_per_verification", "value": vdt * 1e3, "unit": "ms", "higher_is_better": False, "accepted": bool(v_ok),
              "tampered_rejected": bool(v_rej),
              "cpu_baseline": {"value": cver.hot_s * 1e3, "unit": "ms", "cores": threads, "kind": "port", "accepted": bool(cv_ok),
                               "wall_ms_incl_glue": cver_wall * 1e3,
                               "sample": "1 verification: compute_s (serial doubling loop, verifier.rs:156-171) and the final best_multiexp over "
                                         "2^k + 2 + ~40 terms (msm.rs:175); parsing, the transcript and the scalar glue are not counted"},
              "note": "the multiopen + opening checks of plonk::verify_proof's tail on the replay's proof (poly/multiopen/verifier.rs:29-140, "
                      "poly/commitment/verifier.rs:67-141, SingleVerifier plonk/verifier.rs:53-62); GPU arm: wall-clock through halo2_b200.verifier "
                      "incl. point decompression on the device, the host-side transcript and glue"}
    return {
        "verify": verify,
        "metric": "hot_path_ms_per_proof", "value": gdt * 1e3, "unit": "ms", "higher_is_better": False, "k": k,
        "transcript_identical": bool(proof == proof_c and proof_t == proof_c), "proof_bytes": len(proof_c),
        "proof_blake2b": __import__("hashlib").blake2b(proof_c, digest_size=16).hexdigest(),
        "cpu_baseline": {"value": cpu.hot_s * 1e3, "unit": "ms", "cores": threads, "kind": "port", "ipa_threads": cpu.ipa_threads,
                         "ms_by_kind": {k_: v * 1e3 for k_, v in cpu.by_kind.items()}, "wall_ms_incl_glue": cpu_wall * 1e3,
                         "sample": "1 proof: the hot-path calls only (11 commitments, 4 + 4 + 1 transforms, 18 eval_polynomial, 2 kate_division, "
                                   "the 14-round opening); elementwise glue and the transcript are not counted"},
        "params_setup_ms": setup_s * 1e3, "gpu_ms_by_kind_synced": by_kind,
        "note": "proof-shaped replay of plonk::create_proof's hot path for the benches/plonk.rs circuit shape (Vesta, k=14, extended_k=16; "
                "SURVEY.md Appendix C) with the reference's Blake2bWrite / Challenge255 transcript in both arms and every challenge fed back "
                "(tests/prover_replay.py).  NOT the Rust prover: the columns, the h(X) expression and the multiopen sets are stand-ins of the "
                "same shape and size.  GPU arm: wall-clock per proof through the Python host API on device-resident polynomials, "
                "glue and host-side transcript included.  CPU arm: C restatement, hot-path calls only."}


def prover_replay_inputs(cref):
    n = 1 << PROVER_K
    gl = cref.gen_points("vesta", SEED + 50, n + 1)
    g = cref.gen_points("vesta", SEED + 51, n + 2)       # g || w || u
    g[n] = gl[n]                                         # same w
    polys = [cref.gen_scalars("fp", SEED + 60 + i, n) for i in range(4)]
    ext = cref.gen_scalars("fp", SEED + 70, n << 2)
    return g, gl, polys, ext


def params_lagrange_ms(h2, cref, threads, reps=3):
    """Params::new's g -> g_lagrange derivation at k=14 (poly/commitment.rs:74-101: EC-iFFT = best_fft at G = curve point,
    * 2^-k, batch_normalize) through h2_params_lagrange, host generators in / host g_lagrange out, next to the C
    restatement on the host cores (at k=12 when the box has < 32 threads, to keep the run bounded)."""
    from oracle import pasta
    k = PROVER_K
    g = cref.gen_points("vesta", SEED + 80, 1 << k)
    out = h2.lagrange_generators("vesta", k, g)
    t0 = time.time()
    for _ in range(reps):
        out = h2.lagrange_generators("vesta", k, g)
    gpu_ms = (time.time() - t0) / reps * 1e3
    kc = k if threads >= 32 else 12
    r = pasta.VESTA.r
    t0 = time.time()
    want = cref.params_lagrange("vesta", g[:1 << kc], kc, pasta.inv(pasta.omega_for_k("fp", kc), r), pow(pasta.inv(2, r), kc, r), threads)
    cpu_ms = (time.time() - t0) * 1e3
    res = {"k": k, "gpu_ms": gpu_ms, "scalar_muls": (k << (k - 1)) + 1,   # k n/2 - (n - 1) twiddle products + n scalings
           "cpu_baseline": {"k": kc, "ms": cpu_ms, "cores": threads, "kind": "port"}}
    if kc == k:
        res["same_result"] = bool((out == want).all())
    return res


def poly_reductions_ms(h2, cref, reps=5):
    """The prover's coefficient-form reductions at k=14 on resident polynomials -- 16 eval_polynomial (one batch, own points) and
    4 kate_division (arithmetic.rs:297-341; serial loops in the reference, hence 1 core) -- next to the C restatement."""
    import numpy as np
    n = 1 << PROVER_K
    polys = [cref.gen_scalars("fp", SEED + 90 + i, n) for i in range(16)]
    pts = cref.bytes_to_ints(cref.gen_scalars("fp", SEED + 89, 16))
    res = [h2.ResidentPoly("fp", n, p) for p in polys]
    quot = [h2.ResidentPoly("fp", n - 1) for _ in range(4)]
    out = {}
    for name, fn in (("eval_x16", lambda: h2.eval_polynomial_resident(res, pts)),
                     ("kate_division_x4", lambda: (h2.kate_division_resident(res[:4], pts[:4], dst=quot), quot[3].download(1)))):
        fn()
        t0 = time.time()
        for _ in range(reps):
            got = fn()
        out[name] = {"gpu_ms": (time.time() - t0) / reps * 1e3}
    t0 = time.time()
    want = [cref.eval_polynomial("fp", p, x) for p, x in zip(polys, pts)]
    out["eval_x16"]["cpu_baseline"] = {"ms": (time.time() - t0) * 1e3, "cores": 1, "kind": "port"}
    out["eval_x16"]["same_result"] = h2.eval_polynomial_resident(res, pts) == want
    t0 = time.time()
    wq = [cref.kate_division("fp", p, x) for p, x in zip(polys[:4], pts[:4])]
    out["kate_division_x4"]["cpu_baseline"] = {"ms": (time.time() - t0) * 1e3, "cores": 1, "kind": "port"}
    out["kate_division_x4"]["same_result"] = bool(all((q.download(n - 1) == w).all() for q, w in zip(quot, wq)))
    for r in res + quot:
        r.close()
    return out


def lookup_permute_ms(h2, cref, reps=5):
    """The lookup argument's permuted columns (permute_expression_pair, plonk/lookup/prover.rs:563-647) at k=14 on resident
    columns -- a 2^10-value table, inputs drawn from it -- next to the C restatement (serial like the reference: sort + ordered map)."""
    import numpy as np
    n = 1 << PROVER_K
    u = n - 6
    rng = np.random.default_rng(SEED & 0xffffffff)
    pool = cref.gen_scalars("fp", SEED + 120, 1 << 10)
    tab = pool[np.concatenate([np.arange(1 << 10), rng.integers(0, 1 << 10, n - (1 << 10))])]
    inp = tab[rng.integers(0, u, n)]
    a, t = h2.ResidentPoly("fp", n, inp), h2.ResidentPoly("fp", n, tab)
    oa, ot = h2.ResidentPoly("fp", n), h2.ResidentPoly("fp", n)
    h2.permute_expression_pair_resident(a, t, u, oa, ot)
    t0 = time.time()
    for _ in range(reps):
        h2.permute_expression_pair_resident(a, t, u, oa, ot)
    gpu_ms = (time.time() - t0) / reps * 1e3
    t0 = time.time()
    want = cref.permute_expression_pair(inp, tab, u)
    cpu_ms = (time.time() - t0) * 1e3
    same = bool((oa.download(u) == want[0]).all() and (ot.download(u) == want[1]).all())
    for r in (a, t, oa, ot):
        r.close()
    return {"k": PROVER_K, "usable_rows": u, "gpu_ms": gpu_ms, "cpu_baseline": {"ms": cpu_ms, "cores": 1, "kind": "port"}, "same_result": same}


def golden_proofs_verify_ms(h2, cref, threads):
    """The reference's fifteen stored k = 11 proofs (halo2_gadgets/src/test_circuits/circuit_data/proof_*.bin: ECC chip, Sinsemilla,
    Merkle, range checks) verified through the engine under their pinned keys (tests/plonk_verifier.py restates plonk::verify_proof
    around the path).  Reported: acceptance; per proof, the wall time of the whole verification through the Python host mirror and
    the share of the path's own tail -- Guard::use_challenges (compute_s on the device) + MSM::eval (one multiexp over the 2^11
    resident generators) -- next to the same two hot calls on the C restatement; and the BatchVerifier shape
    (plonk/verifier/batch.rs:83-131): all fifteen MSMs scaled and accumulated on the device, ONE eval."""
    from oracle import pasta
    from tests import plonk_verifier as PV
    cases = [c for c in PV.load_golden_proofs() if c["name"] != "plonk_api"]
    k = 11
    delta = PV.scalar_delta(pasta.P_MOD)
    prm = h2.Params.new("vesta", k)
    g_bytes, w_xy, u_xy = prm.g.copy(), prm.w.copy(), prm.u.copy()

    class TimedArm(PV.EngineArm):
        tail_s = 0.0
        keep = None

        def finish(self, guard):
            t0 = time.time()
            if self.keep is not None:                              # batch mode: hand the MSM over instead of evaluating it
                self.keep.append(guard.use_challenges())
                ok = True
            else:
                ok = PV.EngineArm.finish(self, guard)
            self.tail_s += time.time() - t0
            return ok

    arm = TimedArm(h2, "vesta", k, prm.g, prm.g_lagrange, prm.w, prm.u)
    prm.close()
    keys = [PV.PinnedKey(c["key_text"]) for c in cases]
    try:
        ok = all(PV.verify_proof(arm, vk, c["proof"], c["instances"], delta) for vk, c in zip(keys, cases))     # warm-up
        arm.tail_s = 0.0
        t0 = time.time()
        ok = all(PV.verify_proof(arm, vk, c["proof"], c["instances"], delta) for vk, c in zip(keys, cases)) and ok
        wall = time.time() - t0
        tail = arm.tail_s
        bad = bytearray(cases[0]["proof"])
        bad[-40] ^= 1
        rejected = not PV.verify_proof(arm, keys[0], bytes(bad), cases[0]["instances"], delta)
        # batch: every proof's MSM into one accumulator, one eval
        factors = cref.bytes_to_ints(cref.gen_scalars("fp", SEED + 130, len(cases)))
        arm.keep = []
        t0 = time.time()
        for vk, c in zip(keys, cases):
            PV.verify_proof(arm, vk, c["proof"], c["instances"], delta)
        t_guard = time.time() - t0
        t0 = time.time()
        acc = h2.MSM(arm.params)
        for f, m_i in zip(factors, arm.keep):
            acc.scale_add_msm(f, m_i)
        batch_ok = acc.eval()
        batch_tail = time.time() - t0
        for m_i in arm.keep:
            m_i.close()
        acc.close()
    finally:
        arm.close()
    # the C restatement's two hot calls per proof (compute_s, the multiexp), on the MSMs the oracle's verifier builds
    class CpuArm(PV.OracleArm):
        hot_s = 0.0

        def finish(self, guard):
            t0 = time.time()
            s = cref.compute_s("fp", guard.u, guard.neg_c)
            self.hot_s += time.time() - t0
            msm = guard.msm
            if msm.g_scalars is not None:
                for i, gv in enumerate(msm.g_scalars):
                    if gv:
                        s[i] = cref.ints_to_bytes([(int.from_bytes(s[i].tobytes(), "little") + gv) % pasta.P_MOD])[0]
            msm.g_scalars = None
            sc, bs = msm.terms()
            import numpy as np
            scalars = np.concatenate([cref.ints_to_bytes(sc), s])
            bases = np.concatenate([cref.affines_to_bytes(bs), g_bytes])
            t0 = time.time()
            res = cref.best_multiexp("vesta", scalars, bases, threads)
            self.hot_s += time.time() - t0
            return not res.any()

    carm = CpuArm("vesta", k, g_bytes[:1], g_bytes[:1], w_xy, u_xy)          # the generators stay in g_bytes (bytes): no 2^11 tuple conversions
    carm.g = [None] * (1 << k)
    cpu_ok = all(PV.verify_proof(carm, vk, c["proof"], c["instances"], delta) for vk, c in zip(keys, cases))
    n = len(cases)
    return {"k": k, "proofs": n, "accepted": bool(ok), "tampered_rejected": bool(rejected),
            "gpu_ms_per_proof_wall": wall / n * 1e3, "gpu_ms_per_proof_path_tail": tail / n * 1e3,
            "batch": {"accepted": bool(batch_ok), "gpu_ms_accumulate_and_eval": batch_tail * 1e3, "gpu_ms_guards_wall": t_guard * 1e3},
            "cpu_baseline": {"ms_per_proof_hot": carm.hot_s / n * 1e3, "accepted": bool(cpu_ok), "cores": threads, "kind": "port",
                             "sample": "compute_s (verifier.rs:156-171) + the final best_multiexp (msm.rs:175) of each of the 15 proofs; the "
                                       "plonk::verify_proof glue around them is the same Python code in both arms and is not counted here"},
            "note": "reference-held proofs and keys (tests/golden/golden_proofs.json.gz); wall = everything incl. the Python restatement of "
                    "plonk::verify_proof, the Blake2b transcript and per-point decompression calls; path tail = use_challenges + eval"}


def real_proof_ms(h2, cref, k=None, reps=3, threads=None):
    """A REAL proof of the reference's benchmark circuit (benches/plonk.rs: StandardPlonk, 3 advice columns under one permutation,
    4 fixed columns, one gate, minimum degree 5, every usable row filled; rebuilt in tests/bench_circuit.py) at k = 14 on the GPU:
    plonk::create_proof composed from the engine's reference-facing API (tests/plonk_prover.create_proof_engine -- resident
    polynomials, device transforms, Ast programs, batch_invert + running product, fixed-base commits, one batched evaluation call,
    the multi-point opening and the opening argument), with a key generated here (commit_lagrange of the fixed / permutation
    columns) and the proving key's polynomials resident between proofs; the proof is then VERIFIED through the engine
    (tests/plonk_verifier.verify_proof: the verifier the reference's sixteen golden proofs pin).  Wall-clock per proof through the
    Python composition, witness columns given as byte arrays.  CPU arm: the same prover on the C restatement
    (tests/plonk_prover.CrefProver, validated bit for bit against the big-integer oracle prover at small k), same randomness, counting
    ONLY its hot-path calls (commitments, transforms, eval_polynomial, kate_division, the opening's round loop) like the replay's CPU
    arm; the two proofs are compared byte for byte (`transcript_identical`)."""
    from tests import bench_circuit as BC
    from tests import multiopen_cases as MC
    from tests import plonk_prover as PP
    from tests import plonk_verifier as PV
    from tests import prover_replay as R
    k = PROVER_K if k is None else k
    n = 1 << k
    m = P_MOD
    zeta = pow(5, (m - 1) // 3, m)
    delta = PV.scalar_delta(m)
    pts = cref.gen_points("vesta", SEED + 50, n + 2)
    g, w, u = pts[:n], pts[n:n + 1], pts[n + 1:n + 2]
    t0 = time.time()
    gl = h2.lagrange_generators("vesta", k, g)
    prm = h2.Params("vesta", k, g, gl, w, u=u)
    D = h2.EvaluationDomain("fp", BC.DEGREE, k, zeta)
    fixed, sigma, adv = BC.columns(k, m, D.omega, delta, 2834758237 * zeta % m)
    to_b = PV._ints_to_bytes
    fixed_b, sigma_b, adv_b = [to_b(c_) for c_ in fixed], [to_b(c_) for c_ in sigma], [to_b(c_) for c_ in adv]
    xy = lambda col: h2.batch_normalize(prm.commit_lagrange(col, h2.Blind(1)).reshape(1, 96), "vesta")[0]           # keygen.rs:233-236
    as_pt = lambda b: (int.from_bytes(bytes(b[:32]), "little"), int.from_bytes(bytes(b[32:]), "little"))
    vk = PV.PinnedKey(BC.pinned_key_text(k, D.extended_k, 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001, m, D.omega,
                                         [as_pt(xy(c_)) for c_ in fixed_b], [as_pt(xy(c_)) for c_ in sigma_b]))
    pk = {}
    setup_s = time.time() - t0
    try:
        def prove(seed):
            T = R.Blake2bTranscript(m)
            PP.create_proof_engine(h2, prm, vk, fixed_b, sigma_b, [adv_b], [[]], MC.SeededRng("fp", SEED + seed, True), T, zeta, delta, pk=pk)
            return bytes(T.proof)
        proof = prove(200)                                         # warm-up: the proving key's polynomials, pools, graphs
        prove(201)
        t0 = time.time()
        for r_ in range(reps):
            proof = prove(202 + r_)
        dt = (time.time() - t0) / reps
        arm = PV.EngineArm(h2, "vesta", k, params=prm)
        t0 = time.time()
        accepted = PV.verify_proof(arm, vk, proof, [[]], delta)
        verify_ms = (time.time() - t0) * 1e3
        bad = bytearray(proof)
        bad[len(bad) // 2] ^= 1
        rejected = not PV.verify_proof(arm, vk, bytes(bad), [[]], delta)
    finally:
        PP.close_proving_key(pk)
        prm.close()
    threads = threads or (os.cpu_count() or 1)
    cp = PP.CrefProver(cref, "vesta", "fp", g, gl, w, u, threads)
    Tc = R.Blake2bTranscript(m)
    t0 = time.time()
    cp.create_proof(vk, fixed_b, sigma_b, [adv_b], [[]], MC.SeededRng("fp", SEED + 202 + reps - 1, True), Tc, zeta, delta)
    cpu_wall = time.time() - t0
    return {"metric": "ms_per_real_proof", "value": dt * 1e3, "unit": "ms", "higher_is_better": False, "k": k, "proof_bytes": len(proof),
            "transcript_identical": bool(bytes(Tc.proof) == proof),
            "cpu_baseline": {"value": cp.hot_s * 1e3, "unit": "ms", "cores": threads, "kind": "port", "ms_by_kind": {k_: v * 1e3 for k_, v in cp.by_kind.items()},
                             "wall_ms_incl_glue": cpu_wall * 1e3,
                             "sample": "1 real proof on the C restatement: the hot-path calls only (11 commitments, 4 + 4 + 1 transforms, 13 + 4 eval_polynomial, "
                                       "3 kate_division, the 14-round opening); expressions, products and folds are not counted"},
            "accepted_by_the_verifier": bool(accepted), "tampered_rejected": bool(rejected), "verify_ms": verify_ms, "setup_ms": setup_s * 1e3,
            "circuit": "benches/plonk.rs StandardPlonk: 3 advice columns, 1 permutation set, 4 fixed columns, 1 gate, degree 5, 2^k - 6 rows",
            "note": "a real proof (not the replay): plonk::create_proof composed from the engine's API (tests/plonk_prover.create_proof_engine), "
                    "verified through the engine by the pinned-key-driven verifier (tests/plonk_verifier.py).  Wall-clock per proof incl. the "
                    "Python composition; CPU arm: the same prover on the C restatement, hot-path calls only."}


def quotient_pipeline_ms(h2, cref, threads, reps=5):
    """The quotient pipeline of plonk/vanishing/prover.rs:81-88 at k=14, extended_k=16, resident on the device: coeff_to_extended of
    four columns, an h(X)-shaped Ast over them (two gates, a permutation-style product with the linear term, folded by powers of
    y: poly/evaluator.rs:129-228), divide_by_vanishing_poly, extended_to_coeff -- next to the same steps on the C restatement
    (all host threads).  The circuit-specific Ast of benches/plonk.rs is the caller's; this one has its shape and size."""
    import numpy as np
    from halo2_b200.evaluator import Ast, AstLeaf, compile_ast
    zeta = pow(5, (P_MOD - 1) // 3, P_MOD)
    d = h2.EvaluationDomain("fp", PROVER_J, PROVER_K, zeta)
    n = d.n
    cols = [cref.gen_scalars("fp", SEED + 95 + i, n) for i in range(4)]
    y, theta = cref.bytes_to_ints(cref.gen_scalars("fp", SEED + 99, 2))

    def expr(a, b, c, q):
        gate0 = (a * b - c) * q
        gate1 = (a.with_rotation(1) - a) * (b.with_rotation(-1) + Ast.constant_term(7)) * 3
        perm = (c + Ast.linear_term(theta) + Ast.constant_term(11)) * (a.with_rotation(-2) + b * theta)
        return Ast.distribute_powers([gate0, gate1, -perm, q.with_rotation(3)], y)

    res = [h2.ResidentPoly("fp", n, c_) for c_ in cols]
    ext = [h2.ResidentPoly("fp", d.extended_len()) for _ in cols]
    hx = h2.ResidentPoly("fp", d.extended_len())
    out = h2.ResidentPoly("fp", n * d.quotient_poly_degree)
    ev = h2.Evaluator(d, "extended")
    ast = expr(*[ev.register_poly(e) for e in ext])

    def run():
        for r, e in zip(res, ext):
            d.coeff_to_extended_resident(r, out=e)
        ev.evaluate(ast, out=hx)
        d.divide_by_vanishing_poly_resident(hx)
        d.extended_to_coeff_resident(hx, out=out)
        return out.download(1)          # synchronises
    run()
    t0 = time.time()
    for _ in range(reps):
        run()
    gpu_ms = (time.time() - t0) / reps * 1e3
    got = out.download()
    # CPU restatement: same steps, all threads
    code, consts = compile_ast(expr(*[AstLeaf(i) for i in range(4)]), P_MOD, 1 << (d.extended_k - d.k))
    t0 = time.time()
    ext_c = np.stack([cref.coeff_to_extended("fp", c_, PROVER_K, d.extended_k, zeta, d.extended_omega, threads) for c_ in cols])
    h_c = cref.ast_eval("fp", ext_c, d.extended_k, code, consts, d.extended_omega, zeta, threads)
    tev = cref.ints_to_bytes(d.t_evaluations)
    h_i = (np.arange(d.extended_len()) % len(d.t_evaluations))
    t1 = time.time()
    # divide_by_vanishing_poly: an elementwise multiply (domain.rs:329-348) -- through the same interpreter: POLY 0, POLY 1, MUL
    tfull = tev[h_i]
    h_c = cref.ast_eval("fp", np.stack([h_c, tfull]), d.extended_k, np.array([[0, 0, 0, 0], [0, 1, 0, 0], [4, 0, 0, 0]], dtype=np.uint32), [],
                        d.extended_omega, zeta, threads)
    want = cref.extended_to_coeff("fp", h_c, d.extended_k, d.extended_omega_inv, d.extended_ifft_divisor, zeta, n * d.quotient_poly_degree, threads)
    cpu_ms = (time.time() - t0) * 1e3
    same = bool((got == want).all())
    for r in res + ext + [hx, out]:
        r.close()
    return {"k": PROVER_K, "extended_k": d.extended_k, "columns": 4, "ast_instructions": int(code.shape[0]), "gpu_ms": gpu_ms,
            "cpu_baseline": {"ms": cpu_ms, "cores": threads, "kind": "port"}, "same_result": same}


def resident_column_ms(h2, cref, reps=5):
    """One advice column's trip through the hot path at k=14 -- commit_lagrange, lagrange_to_coeff, commit,
    coeff_to_extended, extended values back to the host -- with host buffers per call vs device-resident handles."""
    n, k = 1 << PROVER_K, PROVER_K
    g, gl, polys, _ = prover_replay_inputs(cref)
    params = h2.Params("vesta", k, g[:n], gl[:n], g[n:n + 1])
    dom = h2.EvaluationDomain("fp", PROVER_J, k, pow(5, (P_MOD - 1) // 3, P_MOD))
    blind = h2.Blind(7)
    ext_buf = h2.ResidentPoly("fp", dom.extended_len())

    def host():
        v = polys[0]
        params.commit_lagrange(v, blind)
        cf = dom.lagrange_to_coeff(v)
        params.commit(cf, blind)
        return dom.coeff_to_extended(cf)

    def resident():
        r = h2.ResidentPoly("fp", n, polys[0])
        params.commit_resident([r], [blind], lagrange=True)
        dom.lagrange_to_coeff_resident(r)
        params.commit_resident([r], [blind])
        out = dom.coeff_to_extended_resident(r, ext_buf).download()
        r.close()
        return out

    res = {}
    ref_out = None
    for name, fn in (("host_buffers", host), ("resident", resident)):
        out = fn()
        if ref_out is None:
            ref_out = out
        same = bool((out == ref_out).all())
        t0 = time.time()
        for _ in range(reps):
            fn()
        res[name] = {"ms": (time.time() - t0) / reps * 1e3, "same_result": same}
    ext_buf.close()
    params.close()
    return res


# =================================================================================================
# our arm
# =================================================================================================

# =================================================================================================
# BASELINE configs[4]: MSM 2^24 Pallas pairs TOTAL, sharded over the ranks (strong scaling), bases pre-resident.
# The 2^24 pairs are eight seeded blocks of 2^21, so the problem -- and the point the oracle computes -- is the same
# for every N; rank r of N owns blocks [8 r / N, 8 (r + 1) / N).
# =================================================================================================
C5_LOG_TOTAL, C5_BLOCKS = 24, 8


def config5_strong(torch, dist, L, lib, msm_step, result_affine, barrier, rank, world, dev, sp, cid, steps, with_oracle):
    if C5_BLOCKS % world:
        return {"skipped": f"world size {world} does not divide {C5_BLOCKS} blocks"}
    blk = (1 << C5_LOG_TOTAL) // C5_BLOCKS
    mine = range(rank * C5_BLOCKS // world, (rank + 1) * C5_BLOCKS // world)
    n5 = blk * len(mine)
    sc = torch.cat([rand_canonical_scalars(torch, blk, SEED + 5000 + b, dev) for b in mine])
    bs = torch.empty((n5, 16), dtype=torch.int32, device=dev)
    for j, b in enumerate(mine):
        L.check(lib.h2_dev_gen_points(cid, SEED + 55, ctypes.c_uint64(b * blk), ctypes.c_size_t(blk),
                                      ctypes.c_void_p(bs[j * blk:].data_ptr()), sp))
    for _ in range(2):
        msm_step(sc, bs, n5)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(torch.cuda.current_stream())
    for _ in range(steps):
        msm_step(sc, bs, n5)
    e1.record(torch.cuda.current_stream())
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms /= steps
    out = {"metric": "msm_pairs_per_s", "value": (1 << C5_LOG_TOTAL) / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "n_gpus": world,
           "scaling": "strong", "steps": steps, "pairs_total": 1 << C5_LOG_TOTAL, "pairs_per_gpu": n5,
           "config": {"workload": f"best_multiexp 2^{C5_LOG_TOTAL} Pallas pairs in total (BASELINE configs[4]), contiguous shards of "
                                  f"2^{C5_LOG_TOTAL}/N pairs per rank, bases and scalars resident, NCCL all-gather of the 96 B partials + "
                                  "on-device G-term sum inside the timed step; inputs 1.5 GiB / N per rank (> L2)"}}
    if with_oracle:
        got = result_affine()
        if rank == 0:
            from oracle import cref
            ks, ps = [], []
            for b in range(C5_BLOCKS):
                ks.append(rand_canonical_scalars(torch, blk, SEED + 5000 + b, dev).cpu().numpy().view(np.uint8).reshape(blk, 32))
                t_b = torch.empty((blk, 16), dtype=torch.int32, device=dev)
                L.check(lib.h2_dev_gen_points(cid, SEED + 55, ctypes.c_uint64(b * blk), ctypes.c_size_t(blk), ctypes.c_void_p(t_b.data_ptr()), sp))
                L.check(lib.h2_dev_convert(L.FIELD_ID[L.BASE_FIELD[CURVE]], ctypes.c_void_p(t_b.data_ptr()), ctypes.c_size_t(2 * blk), 0, sp))
                torch.cuda.synchronize()
                ps.append(t_b.cpu().numpy().view(np.uint8).reshape(blk, 64))
                del t_b
            t0 = time.time()
            want = cref.best_multiexp(CURVE, np.concatenate(ks), np.concatenate(ps), os.cpu_count() or 1)
            cdt = time.time() - t0
            out["parity_vs_oracle"] = bool((got == want).all())
            out["cpu_baseline"] = {"value": (1 << C5_LOG_TOTAL) / cdt, "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
                                   "sample": f"1 x full 2^{C5_LOG_TOTAL}-pair best_multiexp (C restatement, c = 17, 16 window tasks)", "ms_per_step": cdt * 1e3}
        barrier()
    del sc, bs
    torch.cuda.empty_cache()
    return out


def window_sweep_and_skew(torch, L, lib, dev, sp, cid, scal0, bases0, n):
    """BASELINE configs[2] "window-size sweep" (c = 8 ... 20, device-resident 2^20 pairs) and the skew cases of SURVEY.md
    section 8(d).3: all-zero, all-one, all-equal, 0/1 mix, top-bit-heavy scalars -- ms per call each."""
    out_dev = torch.zeros(24, dtype=torch.int32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(sc_t, c, reps=3):
        def run():
            L.check(lib.h2_msm_dev(cid, ctypes.c_void_p(sc_t.data_ptr()), L.REPR_CANONICAL, ctypes.c_void_p(bases0.data_ptr()),
                                   ctypes.c_size_t(n), c, ctypes.c_void_p(out_dev.data_ptr()), sp))
        run()
        torch.cuda.synchronize()
        e0.record(torch.cuda.current_stream())
        for _ in range(reps):
            run()
        e1.record(torch.cuda.current_stream())
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    sweep = {}
    for c in range(8, 21):
        try:
            sweep[str(c)] = timed(scal0, c)
        except Exception as e:  # noqa: BLE001
            sweep[str(c)] = f"error: {e}"
    sweep["auto"] = timed(scal0, 0)
    skew = {}
    z = torch.zeros_like(scal0)
    skew["all_zero"] = timed(z, 0)
    one = z.clone(); one[:, 0] = 1
    skew["all_one"] = timed(one, 0)
    eq = scal0[:1].expand(n, 8).contiguous()
    skew["all_equal"] = timed(eq, 0)
    g = torch.Generator(device=dev).manual_seed(SEED + 9)
    mix = z.clone(); mix[:, 0] = torch.randint(0, 2, (n,), dtype=torch.int32, device=dev, generator=g)
    skew["zero_one_mix"] = timed(mix, 0)
    top = z.clone(); top[:, 7] = 0x3FFFFFFF; top[:, 6] = scal0[:, 6]
    skew["top_bit_heavy"] = timed(top, 0)
    skew["uniform"] = sweep["auto"]
    return {"window_sweep_ms": sweep, "skew_ms": skew, "n": n,
            "note": "device-resident h2_msm_dev, ms per call; skewed inputs overflow the single-pass bins and take the exact counting sort"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy: msm (the affine x, y of "
                         "the MSM result) and, for the ours arm, ntt_fp / ntt_fq (a fixed sample of the transforms' outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from halo2_b200 import lib as L

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (halo2_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout: rank 0 prints one JSON line
        dist.init_process_group("nccl", device_id=dev)
    lib = L.init(local_rank)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    cid, n = L.CURVE_ID[CURVE], 1 << LOG_N

    # ---- synthetic inputs, resident in HBM.  Rotating 4 scalar sets + 2 base sets = 256 MiB > L2.
    n_sc, n_bs = 4, 2
    scal = [rand_canonical_scalars(torch, n, SEED + 100 * rank + i, dev) for i in range(n_sc)]
    bases = []
    for i in range(n_bs):
        b = torch.empty((n, 16), dtype=torch.int32, device=dev)
        L.check(lib.h2_dev_gen_points(cid, SEED + 7 + i, ctypes.c_uint64(rank * n), ctypes.c_size_t(n),
                                      ctypes.c_void_p(b.data_ptr()), sp))
        bases.append(b)
    out_dev = torch.zeros(24, dtype=torch.int32, device=dev)
    gathered = torch.zeros(24 * world, dtype=torch.int32, device=dev) if world > 1 else None
    final_dev = torch.zeros(24, dtype=torch.int32, device=dev)

    def msm_step(sc_t, bs_t, count):
        """The whole path on the device: per-rank Pippenger, then (N > 1) the one exchange -- 96-byte Jacobian partials
        all-gathered over NCCL -- and the G-term EC sum on the same stream (h2_point_sum_dev).  No host round trip."""
        L.check(lib.h2_msm_dev(cid, ctypes.c_void_p(sc_t.data_ptr()), L.REPR_CANONICAL, ctypes.c_void_p(bs_t.data_ptr()),
                               ctypes.c_size_t(count), 0, ctypes.c_void_p(out_dev.data_ptr()), sp))
        if world > 1:
            dist.all_gather_into_tensor(gathered, out_dev)
            L.check(lib.h2_point_sum_dev(cid, ctypes.c_void_p(gathered.data_ptr()), ctypes.c_size_t(world),
                                         ctypes.c_void_p(final_dev.data_ptr()), sp))

    def step(i):
        msm_step(scal[i % n_sc], bases[i % n_bs], n)

    def result_affine():
        """The affine canonical bytes of the last step's result (Montgomery Jacobian on the device)."""
        from oracle import cref                       # checker only: normalises a point for comparison
        r = (final_dev if world > 1 else out_dev).clone()
        L.check(lib.h2_dev_convert(L.FIELD_ID[L.BASE_FIELD[CURVE]], ctypes.c_void_p(r.data_ptr()), ctypes.c_size_t(3), 0, sp))
        torch.cuda.synchronize()
        return cref.jac_to_affine(CURVE, r.cpu().numpy().view(np.uint8).reshape(96))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    launches0 = L.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    barrier()
    t_wall1 = time.time()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = L.launch_count() - launches0
    dumps = {}
    if args.dump_outputs and rank == 0:
        dumps["msm"] = result_affine().reshape(2, 32)
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * n / (ms_step * 1e-3)

    # ---- N > 1: the point all ranks computed together against the CPU oracle on the same N x 2^20 pairs (rank 0 regenerates
    # every rank's seeded shard on its own GPU, copies it to the host and runs the C restatement once, outside the timed region)
    parity_multi = None
    if world > 1 and not args.no_cpu_baseline:
        step(0)
        got_aff = result_affine()
        if rank == 0:
            from oracle import cref
            ks, ps = [], []
            for r in range(world):
                ks.append(rand_canonical_scalars(torch, n, SEED + 100 * r + 0, dev).cpu().numpy().view(np.uint8).reshape(n, 32))
                b = torch.empty((n, 16), dtype=torch.int32, device=dev)
                L.check(lib.h2_dev_gen_points(cid, SEED + 7, ctypes.c_uint64(r * n), ctypes.c_size_t(n), ctypes.c_void_p(b.data_ptr()), sp))
                L.check(lib.h2_dev_convert(L.FIELD_ID[L.BASE_FIELD[CURVE]], ctypes.c_void_p(b.data_ptr()), ctypes.c_size_t(2 * n), 0, sp))
                torch.cuda.synchronize()
                ps.append(b.cpu().numpy().view(np.uint8).reshape(n, 64))
                del b
            t0 = time.time()
            want = cref.best_multiexp(CURVE, np.concatenate(ks), np.concatenate(ps), os.cpu_count() or 1)
            parity_multi = {"parity_vs_oracle": bool((got_aff == want).all()), "pairs": world * n, "oracle_s": time.time() - t0,
                            "what": "MSM per rank + NCCL all-gather + on-device G-term sum vs the C restatement on all N x 2^20 pairs"}
            del ks, ps
        barrier()

    # ---- roofline of the dominant kernel, CUDA events on its launch stream
    L.check(lib.h2_profile_enable(1))
    for i in range(5):
        step(i)
    torch.cuda.synchronize()
    tot, cnt = ctypes.c_float(), ctypes.c_uint32()
    L.check(lib.h2_profile_read(0, ctypes.byref(tot), ctypes.byref(cnt)))
    L.check(lib.h2_profile_enable(0))
    hbm_peak, peak_src = measured_peaks()
    k_ms = tot.value / max(cnt.value, 1)
    achieved = MSM_BYTES_PER_PAIR * n / (k_ms * 1e-3) / 1e9
    traffic, traffic_src, ntt_traffic, ntt_traffic_src = None, None, None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")   # dram read+write bytes per launch from the committed ncu --set full captures
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_src = tj.get("msm_accum0_kernel", {}).get("dram_bytes_per_launch"), tj.get("msm_accum0_kernel", {}).get("source")
        ntt_traffic, ntt_traffic_src = tj.get("ntt_pass_kernel", {}).get("dram_bytes_per_launch"), tj.get("ntt_pass_kernel", {}).get("source")
    # the pipe that actually bounds it: 255-bit modular multiplies on the INT32 multiply-add pipe.  Peak = the multiply
    # microbenchmark measured live at full occupancy (h2_bench_field_mul: 4 dependent-chain multiplies per thread and
    # iteration, 64 warps per SM); achieved = multiplies the kernel must execute / its duration.
    # One mixed addition = 8M + 2S; one addition per (point, window) reference: 2 x 8 windows per pair with the GLV split.
    mm = ctypes.c_float()
    L.check(lib.h2_bench_field_mul(0, 256, 148 * 8, 2000, ctypes.byref(mm)))
    peak_gmul = 256 * 148 * 8 * 2000 * 4 / (mm.value * 1e-3) / 1e9
    refs_per_pair = 16
    achieved_gmul = n * refs_per_pair * 10 / (k_ms * 1e-3) / 1e9
    compute = {"pipe": "INT32 multiply-add (fmaheavy)", "unit": "G modmul/s", "achieved": achieved_gmul, "peak": peak_gmul,
               "frac": achieved_gmul / peak_gmul, "modmul_per_launch": n * refs_per_pair * 10,
               "peak_source": "h2_bench_field_mul measured in this run (Montgomery multiply microbenchmark, 64 warps/SM)"}
    roofline = {"kernel": "msm_accum0_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "compute": compute,
                "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": MSM_BYTES_PER_PAIR * n, "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_step,
                "peak_source": peak_src,
                "note": "255-bit modular integer work: the limiter is the INT32 multiply-add pipe, not HBM (DESIGN.md section 5)"}

    # ---- e2e: reference-facing host call, pinned host buffers, copies inside the timed region;
    # every rank pushes its own shard through h2_msm, then the 96 B partials are exchanged
    sc_host = [torch.empty((n, 8), dtype=torch.int32).pin_memory() for _ in range(2)]
    bs_host = [torch.empty((n, 16), dtype=torch.int32).pin_memory() for _ in range(2)]
    for i in range(2):
        sc_host[i].copy_(scal[i])
        tmp = bases[i].clone()   # generator output is Montgomery; the reference hands over canonical coordinates
        L.check(lib.h2_dev_convert(L.FIELD_ID[L.BASE_FIELD[CURVE]], ctypes.c_void_p(tmp.data_ptr()), ctypes.c_size_t(2 * n), 0, sp))
        bs_host[i].copy_(tmp)
    torch.cuda.synchronize()
    res = np.zeros(96, dtype=np.uint8)
    res_t = torch.zeros(96, dtype=torch.uint8, device=dev)
    res_all = [torch.zeros(96, dtype=torch.uint8, device=dev) for _ in range(world)] if world > 1 else None

    def e2e_step(i):
        L.check(lib.h2_msm(cid, ctypes.c_void_p(sc_host[i % 2].data_ptr()), ctypes.c_void_p(bs_host[i % 2].data_ptr()),
                           ctypes.c_size_t(n), L.REPR_CANONICAL, L.ptr(res)))
        if world > 1:
            res_t.copy_(torch.from_numpy(res))
            dist.all_gather(res_all, res_t)
            torch.cuda.synchronize()

    for i in range(2):
        e2e_step(i)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.time()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_dt = (time.time() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    e2e_pinned = {"value": world * n / e2e_dt, "unit": "pairs/s", "ms_per_step": e2e_dt * 1e3, "host_memory": "pinned (cudaHostAlloc)"}

    # The same call with PAGEABLE caller memory -- what a Rust Vec or a numpy array is.  The library stages it through its
    # pinned ring (host threads copy slot-sized pieces while the DMA engine drains the previous ones; the uploads run on their
    # own thread so that chunk j is sorted / accumulated while chunk j + 1 is staged).  This is the headline e2e: it is the
    # memory the reference's callers hand over.  `pageable_plain` switches the ring off (plain cudaMemcpyAsync).
    sc_pg = [np.empty((n, 32), dtype=np.uint8) for _ in range(2)]
    bs_pg = [np.empty((n, 64), dtype=np.uint8) for _ in range(2)]
    for i in range(2):
        sc_pg[i][:] = sc_host[i].numpy().view(np.uint8).reshape(n, 32)
        bs_pg[i][:] = bs_host[i].numpy().view(np.uint8).reshape(n, 64)

    def e2e_pg_step(i):
        L.check(lib.h2_msm(cid, L.ptr(sc_pg[i % 2]), L.ptr(bs_pg[i % 2]), ctypes.c_size_t(n), L.REPR_CANONICAL, L.ptr(res)))
        if world > 1:
            res_t.copy_(torch.from_numpy(res))
            dist.all_gather(res_all, res_t)
            torch.cuda.synchronize()

    def time_pg():
        for i in range(2):
            e2e_pg_step(i)
        barrier()
        t0 = time.time()
        for i in range(e2e_steps):
            e2e_pg_step(i)
        barrier()
        dt = (time.time() - t0) / e2e_steps
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt
    pg_dt = time_pg()
    L.check(lib.h2_test_set_staging(0))
    pg_plain_dt = time_pg()
    L.check(lib.h2_test_set_staging(1))
    e2e = {"value": world * n / pg_dt, "unit": "pairs/s", "h2d_bytes_per_step": n * 96, "d2h_bytes_per_step": 96,
           "ms_per_step": pg_dt * 1e3, "host_memory": "pageable (numpy), staged through the library's pinned ring",
           "api": "h2_msm (host buffers, canonical repr) per rank + all-gather of results", "n_gpus": world,
           "pinned": e2e_pinned,
           "pageable_plain": {"value": world * n / pg_plain_dt, "unit": "pairs/s", "ms_per_step": pg_plain_dt * 1e3,
                              "host_memory": "pageable, plain cudaMemcpyAsync (staging ring off)"}}
    del sc_pg, bs_pg

    # ---- BASELINE configs[4]: 2^24 pairs in total, strong scaling over the ranks (every N, oracle-checked)
    c5 = None
    try:
        c5 = config5_strong(torch, dist, L, lib, msm_step, result_affine, barrier, rank, world, dev, sp, cid, max(3, min(args.steps, 5)),
                            not args.no_cpu_baseline)
    except Exception as e:  # noqa: BLE001
        c5 = {"error": f"{type(e).__name__}: {e}"}
        if world > 1:
            raise

    if rank == 0:
        # ---- NTT (configs[1]) on this GPU
        extra = {}
        a = rand_canonical_scalars(torch, n, SEED + 1, dev)
        L.check(lib.h2_dev_convert(L.FIELD_ID["fp"], ctypes.c_void_p(a.data_ptr()), ctypes.c_size_t(n), 1, sp))
        bufs = [a.clone() for _ in range(5)]   # 5 x 32 MiB rotating > L2
        outs = [torch.empty_like(a) for _ in range(5)]
        omega = pow(5, (P_MOD - 1) >> 32, P_MOD)
        for _ in range(LOG_N, 32):
            omega = omega * omega % P_MOD
        ob = L.fe_bytes(omega)

        def ntt_step(i):
            L.check(lib.h2_ntt_dev(L.FIELD_ID["fp"], ctypes.c_void_p(bufs[i % 5].data_ptr()), ctypes.c_void_p(outs[i % 5].data_ptr()),
                                   L.ptr(ob), L.REPR_CANONICAL, LOG_N, sp))
        for i in range(3):
            ntt_step(i)
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(args.steps):
            ntt_step(i)
        e1.record(stream)
        torch.cuda.synchronize()
        ntt_ms = e0.elapsed_time(e1) / args.steps

        def ntt_sample(field, out):
            """4096 fixed positions of a transform's output (256 KiB instead of 32 MiB), Montgomery -> canonical."""
            s = out[torch.randperm(n, generator=torch.Generator().manual_seed(SEED))[:4096].sort().values.to(dev)]
            L.check(lib.h2_dev_convert(L.FIELD_ID[field], ctypes.c_void_p(s.data_ptr()), ctypes.c_size_t(s.shape[0]), 0, sp))
            return s.cpu().numpy().view(np.uint8)
        if args.dump_outputs:
            dumps["ntt_fp"] = ntt_sample("fp", outs[(args.steps - 1) % 5])
        L.check(lib.h2_profile_enable(1))
        for i in range(5):
            ntt_step(i)
        torch.cuda.synchronize()
        L.check(lib.h2_profile_read(1, ctypes.byref(tot), ctypes.byref(cnt)))
        L.check(lib.h2_profile_enable(0))
        pass_ms = tot.value / max(cnt.value, 1)
        ntt_ach = NTT_BYTES_PER_ELEM * n / (pass_ms * 1e-3) / 1e9
        # host-buffer e2e for the NTT
        ah = torch.empty((n, 8), dtype=torch.int32).pin_memory()
        ah.copy_(rand_canonical_scalars(torch, n, SEED + 2, dev))
        torch.cuda.synchronize()
        for _ in range(2):
            L.check(lib.h2_ntt(L.FIELD_ID["fp"], ctypes.c_void_p(ah.data_ptr()), L.ptr(ob), LOG_N, L.REPR_CANONICAL))
        t0 = time.time()
        for _ in range(5):
            L.check(lib.h2_ntt(L.FIELD_ID["fp"], ctypes.c_void_p(ah.data_ptr()), L.ptr(ob), LOG_N, L.REPR_CANONICAL))
        ntt_e2e = (time.time() - t0) / 5
        extra["ntt"] = {
            "metric": "ntt_elems_per_s", "value": n / (ntt_ms * 1e-3), "unit": "elems/s", "ms_per_step": ntt_ms,
            "config": {"workload": f"best_fft 2^{LOG_N} over Fp (configs[1]), twiddles cached per (omega, log_n), "
                                   "5 rotating 32 MiB buffers (> L2)"},
            "roofline": {"kernel": "ntt_pass_kernel", "bound": "hbm", "achieved": ntt_ach, "peak": hbm_peak, "unit": "GB/s",
                         "frac": ntt_ach / hbm_peak, "traffic": ntt_traffic, "traffic_source": ntt_traffic_src, "kernel_ms": pass_ms, "passes_per_step": 3,
                         "compute": {"pipe": "INT32 multiply-add (fmaheavy)", "unit": "G modmul/s", "achieved": (LOG_N * n / 2) / (ntt_ms * 1e-3) / 1e9,
                                     "peak": peak_gmul, "frac": (LOG_N * n / 2) / (ntt_ms * 1e-3) / 1e9 / peak_gmul,
                                     "note": "log_n * n / 2 butterflies, one multiply each, over the whole transform"}},
            "e2e": {"value": n / ntt_e2e, "unit": "elems/s", "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": n * 32,
                    "ms_per_step": ntt_e2e * 1e3, "api": "h2_ntt (host buffers, canonical repr)"},
        }

        # ---- the same transform over Fq (configs[1] names the Vesta scalar field Fq; both fields are measured)
        q_omega = pow(5, (Q_MOD - 1) >> 32, Q_MOD)
        for _ in range(LOG_N, 32):
            q_omega = q_omega * q_omega % Q_MOD
        qb = L.fe_bytes(q_omega)
        aq = rand_canonical_scalars(torch, n, SEED + 11, dev)
        L.check(lib.h2_dev_convert(L.FIELD_ID["fq"], ctypes.c_void_p(aq.data_ptr()), ctypes.c_size_t(n), 1, sp))
        qbufs = [aq.clone() for _ in range(5)]

        def nttq_step(i):
            L.check(lib.h2_ntt_dev(L.FIELD_ID["fq"], ctypes.c_void_p(qbufs[i % 5].data_ptr()), ctypes.c_void_p(outs[i % 5].data_ptr()),
                                   L.ptr(qb), L.REPR_CANONICAL, LOG_N, sp))
        for i in range(3):
            nttq_step(i)
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(args.steps):
            nttq_step(i)
        e1.record(stream)
        torch.cuda.synchronize()
        nttq_ms = e0.elapsed_time(e1) / args.steps
        if args.dump_outputs:
            dumps["ntt_fq"] = ntt_sample("fq", outs[(args.steps - 1) % 5])
        extra["ntt_fq"] = {"metric": "ntt_elems_per_s", "value": n / (nttq_ms * 1e-3), "unit": "elems/s", "ms_per_step": nttq_ms,
                           "config": {"workload": f"best_fft 2^{LOG_N} over Fq (configs[1] as written: the Vesta scalar field)"}}
        del qbufs, aq
        # pageable host buffers for the NTT e2e as well (32 MiB up, 32 MiB down)
        ap_ = np.empty((n, 32), dtype=np.uint8)
        ap_[:] = ah.numpy().view(np.uint8).reshape(n, 32)
        for _ in range(2):
            L.check(lib.h2_ntt(L.FIELD_ID["fp"], L.ptr(ap_), L.ptr(ob), LOG_N, L.REPR_CANONICAL))
        t0 = time.time()
        for _ in range(5):
            L.check(lib.h2_ntt(L.FIELD_ID["fp"], L.ptr(ap_), L.ptr(ob), LOG_N, L.REPR_CANONICAL))
        ntt_pg = (time.time() - t0) / 5
        extra["ntt"]["e2e"]["pinned"] = {"value": extra["ntt"]["e2e"]["value"], "ms_per_step": extra["ntt"]["e2e"]["ms_per_step"]}
        extra["ntt"]["e2e"].update({"value": n / ntt_pg, "ms_per_step": ntt_pg * 1e3,
                                    "host_memory": "pageable (numpy), staged through the library's pinned ring both ways"})
        del ap_
        try:
            extra["msm_window_sweep_and_skew"] = window_sweep_and_skew(torch, L, lib, dev, sp, cid, scal[0], bases[0], n)
        except Exception as e:  # noqa: BLE001
            extra["msm_window_sweep_and_skew"] = {"error": f"{type(e).__name__}: {e}"}

        # ---- CPU baseline: the reference algorithm restated in C, all host cores, same workload
        cpu = None
        if not args.no_cpu_baseline and world == 1:   # the CPU arm and the single-GPU side measurements: N = 1 only
            from oracle import cref
            threads = os.cpu_count() or 1
            kb = cref.gen_scalars(SCALAR_FIELD, SEED + 3, n)
            pb = cref.gen_points(CURVE, SEED + 33, n)
            cref.best_multiexp(CURVE, kb[:4096], pb[:4096], threads)
            t0 = time.time()
            reps = 2
            for _ in range(reps):
                want = cref.best_multiexp(CURVE, kb, pb, threads)
            cdt = (time.time() - t0) / reps
            cpu = {"value": n / cdt, "unit": "pairs/s", "cores": threads, "kind": "port",
                   "sample": f"{reps} x full 2^{LOG_N}-pair best_multiexp (reference algorithm, C restatement, "
                             f"{threads} threads; window-parallel so at most 19 are busy)", "ms_per_step": cdt * 1e3}
            # and a parity spot check of the e2e path on the very same input
            got = np.zeros(96, dtype=np.uint8)
            L.check(lib.h2_msm(cid, L.ptr(kb), L.ptr(pb), ctypes.c_size_t(n), L.REPR_CANONICAL, L.ptr(got)))
            cpu["parity_vs_gpu"] = bool((cref.jac_to_affine(CURVE, got) == want).all())
            a_c = cref.gen_scalars("fp", SEED + 2, n)
            t0 = time.time()
            cref.best_fft("fp", a_c, omega, LOG_N, threads)
            extra["ntt"]["cpu_baseline"] = {"value": n / (time.time() - t0), "unit": "elems/s", "cores": threads, "kind": "port",
                                            "sample": f"1 x full 2^{LOG_N} best_fft (serial bit-reversal + twiddle scan, "
                                                      "join-recursion; includes canonical<->Montgomery conversion)"}
            import halo2_b200 as h2
            extra["resident_column_k14"] = resident_column_ms(h2, cref)
            def guarded(fn, *a):     # a failing side measurement must not take the headline line down with it
                try:
                    return fn(*a)
                except Exception as e:  # noqa: BLE001
                    return {"error": f"{type(e).__name__}: {e}"}
            extra["params_lagrange_k14"] = guarded(params_lagrange_ms, h2, cref, threads)
            extra["poly_reductions_k14"] = guarded(poly_reductions_ms, h2, cref)
            extra["quotient_pipeline_k14"] = guarded(quotient_pipeline_ms, h2, cref, threads)
            extra["lookup_permute_k14"] = guarded(lookup_permute_ms, h2, cref)
            extra["golden_proofs_verify_k11"] = guarded(golden_proofs_verify_ms, h2, cref, threads)
            extra["create_proof_k14_replay"] = guarded(prover_replay, h2, cref, threads)
            # the top of the reference's own bench range (benches/plonk.rs: k = 8..16): the passes stop being latency-bound
            extra["create_proof_k16_replay"] = guarded(prover_replay, h2, cref, threads, 2, 16)
            # a REAL proof of the reference's benchmark circuit through the engine's API, verified through the engine (after the replays,
            # whose timings it must not perturb)
            extra["create_proof_k14_real"] = guarded(real_proof_ms, h2, cref, None, 3, threads)

        extra["msm_2p24_strong"] = c5
        line = {
            "metric": "msm_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32x8 (255-bit modular integers)", "data": "synthetic",
            "config": {"workload": f"best_multiexp 2^{LOG_N} pairs per GPU, Pallas (BASELINE configs[2]); "
                                   f"N>1: contiguous 2^{LOG_N}-pair shard per rank + NCCL all-gather of 96 B partials + on-device G-term EC sum, all inside the timed step "
                                   "(the 2^24-total strong-scaling config is extra.msm_2p24_strong)",
                       "pairs_per_gpu": n, "window_bits": "auto", "l2": "inputs rotate over 4 scalar + 2 base buffers (256 MiB > L2)",
                       "parallelism": f"shard x{world}"},
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "gpu_launches": int(launches),
            "multi_gpu_parity": parity_multi, "extra": extra,
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
