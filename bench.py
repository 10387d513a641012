#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for the B200-native PlonK proving backend.

Headline (BASELINE.json metric, first clause; configs[3]): proofs/sec of the VALID-MATCH-class
TurboPlonk statement — a synthetic circuit of n = 2^16 gates with 17 public inputs standing in for
`IntentAndBalancePrivateSettlementCircuit` (SURVEY.md §0.1; the reference's Rust circuit synthesis
cannot run here) — proved by the device prover behind `b200_plonk_prove`.  A "step" is one full
proof: witness table in, 1152-byte proof out.  `value` has the witness table resident in HBM;
`e2e` passes it from pinned host memory through the same C-ABI call (H2D inside the timed region).

Second clause (configs[1]): a 2^20-point BN254 G1 MSM per GPU, reported in the `msm` object of the
same JSON line as achieved GB/s of algorithmic bytes (96 B per (point, scalar) pair, SURVEY §8(d)).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--concurrency C] [--dump-outputs DIR]

N > 1 (under torchrun, one rank per GPU): proofs are independent jobs — one proof stream per GPU,
no data-path collective (weak scaling); the MSM leg shards one N*2^20-point MSM by point range
and finishes with one NCCL all_gather of 72-byte partial sums + a k-term G1 sum (EC addition is
not an NCCL reduce op).

--impl reference times the CPU restatement of the reference's prover (oracle/: the reference is
Rust with un-vendored crates and cannot be built here) on all host cores, same circuit.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# A prover pool keeps 3 streams per worker busy; with the default 8 hardware queues unrelated streams share a queue and
# wait for each other.  Must be in the environment before the process's first CUDA call (profiles/r2r_max_connections.log:
# +3 % on the 2^12 statement and the bundle, nothing at 2^16).  A host application sets it the same way.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))  # host_circuits: caller-side restatement of the reference's circuits

LOG_N = 16                 # "~2^16 constraints"
NUM_INPUTS = 17            # IntentAndBalancePrivateSettlementStatement (SURVEY.md §2.1)
CIRCUIT_SEED = 0xB200
MSM_LOG_N = 20
BYTES_PER_PAIR = 96        # 64 B affine base + 32 B scalar (SURVEY.md §8(d))
SEED_BASES, SEED_SCALARS, SEED_SRS = 0xB200, 0x5CA1A8, 0x7A0
METRIC = "proofs/sec, VALID-MATCH-class TurboPlonk proof (n = 2^16 gates, BN254/KZG)"
WORKLOAD = ("synthetic TurboPlonk circuit, n = 2^16 gates, 17 public inputs, 5 wire columns, 13 selector columns "
            "(stand-in for IntentAndBalancePrivateSettlementCircuit, BASELINE.json configs[3]); "
            "13 KZG commitments of ~2^16 points and a degree-(5n+7) quotient per proof (the reference: 8n-point coset FFTs; "
            "this library: 6 cosets of n points, same coefficients)")


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_proof(out_dir, proof):
    """`--dump-outputs`: one <field>.npy per field of the proof, float64.  Coordinates and evaluations are 256-bit
    integers (Montgomery form, as the C ABI returns them); each is stored as its eight 32-bit little-endian words, which
    float64 holds exactly, so two builds can be compared bit for bit: shape (..., 16) per G1 point, (..., 8) per Fr."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, _ in type(proof)._fields_:
        limbs = np.ctypeslib.as_array(getattr(proof, name))
        words = np.ascontiguousarray(limbs, dtype="<u8").view("<u4")
        np.save(os.path.join(out_dir, name + ".npy"), words.astype(np.float64))


def make_circuit(kind, log_n, seed):
    """The proved circuit.  "synthetic" (default): renegade_b200/synth.py, random gates of the reference's mix.
    "merkle": as many height-10 Poseidon2 Merkle openings (the reference's gadgets restated in
    examples/host_circuits/circuit.py, public roots) as fit the domain — 27 at n = 2^16; same prover work, real constraints."""
    from renegade_b200 import synth
    if kind == "synthetic":
        return synth.synth_circuit(log_n, num_inputs=NUM_INPUTS, seed=seed)
    import random
    from host_circuits import circuit as cb
    rnd = random.Random(seed)
    cs = cb.PlonkCircuit()
    per_opening = 2400  # 11 sponge hashes of 195-gate permutations plus selects and additions
    while cs.num_gates + per_opening + 1 <= (1 << log_n):
        leaf = [rnd.randrange(cb.R) for _ in range(4)]
        opening = cb.MerkleOpening([rnd.randrange(cb.R) for _ in range(10)], [rnd.random() < 0.5 for _ in range(10)])
        root = cs.create_public_variable(cb.native_merkle_root(leaf, opening))
        op = cb.MerkleOpeningVar([cs.create_variable(v) for v in opening.elems],
                                 [cs.create_boolean_variable(b) for b in opening.indices])
        cb.PoseidonMerkleHashGadget.compute_and_constrain_root([cs.create_variable(v) for v in leaf], op, root, cs)
    return cs.finalize_for_arithmetization(min_log_n=log_n)


def real_statement_leg(pool, ctx, d_srs_ptr, conc, steps, srs_host=None, cpu_baseline=False):
    """The reference's own statements at their own sizes (restated in examples/host_circuits/valid_balance_create.py and
    private_settlement.py: n = 2^13 and 2^12, not the 2^16 BASELINE.json quotes): one proof alone, and proofs/s end
    to end from pinned host memory through the pool.  Reported beside the headline, never instead of it."""
    import numpy as np
    import torch
    from host_circuits import private_settlement as ps
    from renegade_b200 import synth
    from host_circuits import valid_balance_create as vbc
    from renegade_b200.backend import PlonkKzgSnark, prove_raw
    w, st = vbc.create_witness_statement(1)
    parties, st2 = ps.create_witness_statement(1)
    circuits = [("valid_balance_create (BASELINE.json configs[0])", vbc.ValidBalanceCreate.build(w, st)),
                ("intent_and_balance_private_settlement (the statement of configs[3])",
                 ps.IntentAndBalancePrivateSettlementCircuit.build(parties, st2))]
    res = {}
    for name, cs in circuits:
        circ = cs.finalize_for_arithmetization()
        bases = ctx.load_bases_device(d_srs_ptr, circ.n + 3)
        pk = PlonkKzgSnark.preprocess(ctx, bases, circ.log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
        h_w = torch.from_numpy(circ.wires.view(np.int64)).pin_memory()
        bl = [synth.splitmix_blinders(5000 + i) for i in range(8)]
        for i in range(3):
            prove_raw(ctx, pk, h_w.data_ptr(), circ.pub_inputs, bl[i])
        t = time.perf_counter()
        for i in range(5):
            prove_raw(ctx, pk, h_w.data_ptr(), circ.pub_inputs, bl[i])
        single_ms = (time.perf_counter() - t) / 5 * 1e3
        rate = None
        if pool is not None:
            def run(count):
                tickets = [pool.submit_prove(pk, h_w.data_ptr(), circ.pub_inputs, bl[i % 8]) for i in range(count)]
                for tk in tickets:
                    pool.wait(tk)
            run(8 * conc)  # steady state: every worker has its buffers sized and its rounds captured as graphs
            l0, h0 = ctx._lib.b200_kernel_launches(), ctx._lib.b200_launch_host_ns()
            t = time.perf_counter()
            run(steps)
            rate = steps / (time.perf_counter() - t)
            launches = (ctx._lib.b200_kernel_launches() - l0) / steps
            launch_host_us = (ctx._lib.b200_launch_host_ns() - h0) / steps / 1e3
        cpu = None
        if cpu_baseline:  # the oracle prover on the same tables, SRS and blinders — the only use of oracle/ in this leg
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import oracle_c
            oracle_c.autotune_threads()
            srs_np = srs_host[:circ.n + 3]
            opk = oracle_c.plonk_preprocess(circ.log_n, circ.selectors, circ.perm, circ.k, srs_np)
            t = time.perf_counter()
            rc, oproof, _, _ = oracle_c.plonk_prove(circ.log_n, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs, bl[0], srs_np)
            cdt = time.perf_counter() - t
            gproof = prove_raw(ctx, pk, h_w.data_ptr(), circ.pub_inputs, bl[0])
            cpu = {"value": 1.0 / cdt, "unit": "proofs/s", "cores": oracle_c.num_threads(), "kind": "port",
                   "sample": "1 proof of the same circuit, SRS and blinders (%.3f s)" % cdt,
                   "bit_exact_vs_gpu": bool(rc == 0 and bytes(oproof) == bytes(gproof))}
        res[name] = {"log_n": circ.log_n, "gates": circ.n_gates, "num_inputs": circ.num_inputs,
                     "ms_one_proof_in_flight": single_ms, "proofs_per_s_e2e": rate, "in_flight": conc, "steps": steps,
                     "launches_per_proof": launches if pool is not None else None,
                     "launch_host_us_per_proof": launch_host_us if pool is not None else None,
                     "cpu_baseline": cpu}
        pk.free()
        bases.free()
    return res


def private_match_bundle_leg(pool, ctx, d_srs_ptr, conc, bundles, srs_host=None, cpu_baseline=False):
    """What the reference proves for one private match (native_proof_manager.rs:526-584, 726-782), with the restated
    circuits: both parties' INTENT AND BALANCE VALIDITY (n = 2^14) and OUTPUT BALANCE VALIDITY (n = 2^13) proofs, the
    PRIVATE SETTLEMENT proof (n = 2^12) and the four link proofs — `bundles` of them through the pool, end to end from
    pinned host memory."""
    import numpy as np
    import torch
    from host_circuits import intent_and_balance_validity as val
    from host_circuits import output_balance_validity as obv
    from host_circuits import private_settlement as ps
    from renegade_b200 import synth
    from renegade_b200.backend import GroupLayout, LinkingHint, PlonkKzgSnark
    if pool is None:
        return {"skipped": "needs the pool (concurrency > 1)"}
    parties, _ = ps.create_witness_statement(seed=61)
    validity = [val.create_witness_statement(seed=70 + i, intent=parties[i].intent, balance=parties[i].input_balance)
                for i in (0, 1)]
    out_validity = [obv.create_witness_statement(80 + i, parties[i].output_balance) for i in (0, 1)]
    parties, statement = ps.create_witness_statement(
        seed=61, linked=[(validity[i][0].new_amount_public_share, validity[i][0].post_match_balance_shares,
                          out_validity[i][0].post_match_balance_shares) for i in (0, 1)])
    settlement_cs = ps.IntentAndBalancePrivateSettlementCircuit.build(parties, statement)
    layouts = settlement_cs.get_circuit_layout()
    circs = [settlement_cs.finalize_for_arithmetization()] + \
            [val.IntentAndBalanceValidityCircuit.build(w, st, layouts).finalize_for_arithmetization() for w, st in validity] + \
            [obv.OutputBalanceValidityCircuit.build(w, st, layouts).finalize_for_arithmetization() for w, st in out_validity]
    bases = ctx.load_bases_device(d_srs_ptr, (1 << 14) + 3)
    pks = [PlonkKzgSnark.preprocess(ctx, bases, c.log_n, c.num_inputs, c.selectors, c.perm, c.k) for c in circs]
    wires = [torch.from_numpy(c.wires.view(np.int64)).pin_memory() for c in circs]
    bl = [synth.splitmix_blinders(7000 + i) for i in range(8)]
    # (validity proof index, link group): party groups link proofs 1, 2; output-balance groups link proofs 3, 4
    link_plan = [(1 + p, GroupLayout(layouts[g].alignment, layouts[g].offset, layouts[g].size))
                 for p, g in enumerate(ps.PARTY_LINKS)] + \
                [(3 + p, GroupLayout(layouts[g].alignment, layouts[g].offset, layouts[g].size))
                 for p, g in enumerate(ps.OUTPUT_LINKS)]

    def run(count):
        # one ticket per bundle: the five proofs, then the four link proofs forked inside the pool (b200_pool_submit_bundle)
        tickets = [pool.submit_bundle(bases, [(pks[j], wires[j].data_ptr(), circs[j].pub_inputs, bl[(5 * b + j) % 8]) for j in range(5)],
                                      [(j, 0, lay) for j, lay in link_plan]) for b in range(count)]
        return [pool.wait(tk) for tk in tickets]
    run(max(2, 6 * conc))  # steady state: every worker has proved every key twice (buffers sized, rounds captured as graphs)
    t = time.perf_counter()
    res = run(bundles)
    dt = time.perf_counter() - t
    # CPU baseline: the oracle prover (the restated reference algorithm) on the same five tables and the same four
    # links, one bundle, all host cores — the only place this leg touches oracle/
    cpu = None
    if cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_c
        oracle_c.autotune_threads()
        srs_np = srs_host
        opks = [oracle_c.plonk_preprocess(c.log_n, c.selectors, c.perm, c.k, srs_np[:c.n + 3]) for c in circs]
        t0 = time.perf_counter()
        oproofs, olinks = [], []
        for j, c in enumerate(circs):
            rc, op, _, olink = oracle_c.plonk_prove(c.log_n, c.num_inputs, c.k, opks[j], c.wires, c.pub_inputs, bl[j % 8],
                                                    srs_np[:c.n + 3], True)
            assert rc == 0
            oproofs.append((op, olink))
        for j, lay in link_plan:
            rc, olp, _ = oracle_c.plonk_link(oproofs[j][1], oproofs[0][1], oproofs[j][0].to_array()[:8].copy(),
                                             oproofs[0][0].to_array()[:8].copy(), lay.alignment, lay.offset, lay.size, srs_np)
            assert rc == 0
            olinks.append(olp)
        cdt = time.perf_counter() - t0
        # bundle 0 of the timed run used blinders bl[j % 8]: its proofs and link proofs must be the oracle's, byte for byte
        g_proofs, _, g_links = res[0] if bundles >= 1 else (None, None, None)
        exact = all(bytes(g_proofs[j]) == bytes(oproofs[j][0]) for j in range(5)) and \
            all(bytes(g_links[i]) == bytes(olinks[i]) for i in range(4))
        cpu = {"value": 1.0 / cdt, "unit": "bundles/s", "cores": oracle_c.num_threads(), "kind": "port",
               "sample": "1 whole bundle (5 proofs + 4 link proofs) on the same tables, SRS and blinders (%.2f s)" % cdt,
               "bit_exact_vs_gpu": bool(exact)}
    for pk in pks:
        pk.free()
    bases.free()
    return {"bundles_per_s_e2e": bundles / dt, "ms_per_bundle": dt / bundles * 1e3, "bundles": bundles, "in_flight": conc,
            "cpu_baseline": cpu,
            "proofs_per_bundle": {"intent_and_balance_validity (n = 2^14)": 2, "output_balance_validity (n = 2^13)": 2,
                                  "private_settlement (n = 2^12)": 1, "link proofs": 4}}


def collaborative_leg(pool, ctx, d_srs_ptr, conc, count, srs_host=None, cpu_baseline=False):
    """VALID MATCH MPC in the metric's own words: the VALID-MATCH-class settlement statement (n = 2^12) proved JOINTLY by two
    parties holding additive shares of the witness table (renegade_b200/collaborative.py on the device backend: share-wise
    NTT / MSM, Beaver multiplications for the 26 quotient products and the round-2 products).  Host-orchestrated, one
    proof at a time; the opened proof must equal the single-prover proof of the same witness and blinders."""
    import numpy as np
    from host_circuits import private_settlement as ps
    from renegade_b200 import collaborative as co
    from renegade_b200 import synth
    from renegade_b200.backend import PlonkKzgSnark
    parties, statement = ps.create_witness_statement(seed=61)
    circ = ps.IntentAndBalancePrivateSettlementCircuit.build(parties, statement).finalize_for_arithmetization()
    bases = ctx.load_bases_device(d_srs_ptr, circ.n + 3, window_bits=1)
    be = co.DeviceBackend(ctx, bases)
    t = time.perf_counter()
    cpk = co.CollaborativeProvingKey.build(be, circ.log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    setup_s = time.perf_counter() - t
    bl = synth.splitmix_blinders(4242)
    shares = co.share_table(np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), 2, seed=1)
    bsh = co.share_table(np.asarray(bl, dtype=np.uint64).reshape(-1, 4), 2, seed=2)
    co.MultiproverPlonkKzgSnark.prove_with_link_hint(be, cpk, shares, circ.pub_inputs, bsh)  # warm-up
    ts = []
    for _ in range(count):
        t = time.perf_counter()
        proof, _, fab = co.MultiproverPlonkKzgSnark.prove_with_link_hint(be, cpk, shares, circ.pub_inputs, bsh)
        ts.append(time.perf_counter() - t)
    pk = PlonkKzgSnark.preprocess(ctx, bases, circ.log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    single, _ = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, bl)
    pk.free()
    bases.free()
    ts.sort()
    return {"statement": "intent_and_balance_private_settlement, n = 2^12, 2 parties", "ms_per_joint_proof": ts[len(ts) // 2] * 1e3,
            "joint_proofs_per_s": 1.0 / ts[len(ts) // 2], "opened_proof_equals_single_prover_proof": bytes(proof) == bytes(single),
            "beaver_multiplications": fab.multiplications, "opened_field_elements": fab.opened_elements, "key_setup_s": setup_s,
            "note": "arithmetic of the protocol with the transport collapsed to in-process sums; host-orchestrated (Python), "
                    "so the figure is an upper bound on latency, not a tuned throughput"}


def run_extras(args):
    """`--extras-only`: the restated statements at their own sizes and the private-match bundle, on device 0, as one JSON
    object on stdout (bench.py's main run calls this in a subprocess)."""
    import numpy as np
    import torch
    import renegade_b200 as rb
    from renegade_b200.backend import ProverPool
    conc = max(1, args.concurrency)
    torch.cuda.set_device(0)
    pool = ProverPool(0, workers=conc) if conc > 1 else None
    ctx = pool.context(0) if pool else rb.Context(0)
    n_srs = (1 << 14) + 3
    d_srs = torch.empty((n_srs, 8), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.known_dlog_bases_device(SEED_SRS, n_srs, d_srs.data_ptr())
    extras = {}
    srs_host = d_srs.cpu().numpy().view(np.uint64)
    for key, leg, count in (("real_statements", real_statement_leg, 600), ("private_match_bundle", private_match_bundle_leg, 160),
                            ("valid_match_mpc_collaborative", collaborative_leg, 5)):
        if key in os.environ.get("B200_BENCH_SKIP_LEGS", "").split(","):  # tools/small_proof_sweep.sh
            continue
        try:
            extras[key] = leg(pool, ctx, d_srs.data_ptr(), conc, count, srs_host, not args.no_cpu_baseline)
        except Exception as e:
            extras[key] = {"error": repr(e)[:300]}
    print(json.dumps(extras), flush=True)
    os._exit(0)  # skip interpreter teardown: the parent only needs the line above


def multi_plan(multi, mbases):
    """Window plan of local device 0's shard of a sharded set of bases."""
    import ctypes as C
    plan = (C.c_int * 4)()
    multi._lib.b200_multi_bases_plan(mbases._h, 0, C.byref(plan))
    return {"window_bits": plan[0], "digits": plan[1], "physical_windows": plan[2], "tables": plan[3]}


def shared_config(args):
    """The `config` object BOTH arms print, key for key (the driver compares them)."""
    return {"workload": WORKLOAD, "log_n": LOG_N, "num_inputs": NUM_INPUTS, "circuit": args.circuit}


def base_line(args, world):
    return {"metric": METRIC, "unit": "proofs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 (256-bit Montgomery integers; Fr and Fq of BN254)", "data": "synthetic"}


def run_reference(args, rank, world):
    """CPU arm: the oracle's restatement of the reference prover, all host cores (OpenMP)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c
    from renegade_b200 import synth
    t0 = time.perf_counter()
    cores = oracle_c.autotune_threads()  # all logical CPUs unless a subset is faster on this (shared) host
    log_n = LOG_N
    while True:
        n = 1 << log_n
        circ = make_circuit(args.circuit, log_n, CIRCUIT_SEED)
        srs = oracle_c.known_dlog_bases(SEED_SRS, n + 3)
        pk = oracle_c.plonk_preprocess(log_n, circ.selectors, circ.perm, circ.k, srs)
        bl = synth.splitmix_blinders(1)
        t = time.perf_counter()
        rc, _, _, _ = oracle_c.plonk_prove(log_n, circ.num_inputs, circ.k, pk, circ.wires, circ.pub_inputs, bl, srs)
        probe = time.perf_counter() - t
        assert rc == 0
        # bounded sample: the whole --steps/--warmup run must end within a few minutes
        if probe * (args.steps + args.warmup) <= 240.0 or log_n <= 12:
            break
        log_n -= 1
    for i in range(args.warmup):
        oracle_c.plonk_prove(log_n, circ.num_inputs, circ.k, pk, circ.wires, circ.pub_inputs, bl, srs)
    t = time.perf_counter()
    for i in range(args.steps):
        oracle_c.plonk_prove(log_n, circ.num_inputs, circ.k, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(i), srs)
    dt = (time.perf_counter() - t) / max(args.steps, 1)
    scale = float(1 << (LOG_N - log_n))  # a 2^k-times smaller circuit stands for 1/2^k of a proof
    value = 1.0 / (dt * scale)
    sample = "1 full proof of the same circuit per step" if log_n == LOG_N else \
        f"one proof of a 2^{log_n}-gate circuit per step, counted as 1/{int(scale)} proof"
    out = base_line(args, args.gpus)
    out.update({
        "impl": "reference", "value": value, "ms_per_step": dt * 1e3,
        "config": shared_config(args), "sample": sample,
        "cpu_baseline": {"value": value, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "restated CPU prover (C + OpenMP; arkworks msm_bigint / radix-2 FFT algorithms, "
                                 "jellyfish TurboPlonk rounds) — not the Rust reference itself"},
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "setup_s": time.perf_counter() - t0,
    })
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--concurrency", type=int, default=int(os.environ.get("B200_BENCH_CONCURRENCY", "6")),
                    help="proofs in flight per GPU (one context + stream each), like the reference's rayon pool "
                         "of concurrent proof jobs (native_proof_manager.rs:187-192)")
    ap.add_argument("--msm-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-msm", action="store_true")
    ap.add_argument("--extras-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-real-statements", action="store_true",
                    help="skip the extra leg that proves the restated VALID BALANCE CREATE and PRIVATE SETTLEMENT circuits")
    ap.add_argument("--circuit", choices=("synthetic", "merkle"), default="synthetic",
                    help="synthetic: random gates of the reference's mix (default); merkle: height-10 Poseidon2 Merkle "
                         "openings built with the reference's gadgets (examples/host_circuits/circuit.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed proofs, write the last one (the proof a caller receives) to DIR as one "
                         ".npy per field; the inputs depend on the arguments only, so two builds can be compared")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device prover's proof; the reference arm has none")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.extras_only:
        run_extras(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import renegade_b200 as rb
    from renegade_b200 import synth
    from renegade_b200.backend import PlonkKzgSnark, ProverPool, plonk_last_timings, prove_raw
    from renegade_b200.sharded import MultiGpu

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(dt):
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        return dt

    # ---------------------------------------------------------------------------------------------
    # setup: circuit, SRS, proving key (device resident), witness tables
    # ---------------------------------------------------------------------------------------------
    t_setup = time.perf_counter()
    n = 1 << LOG_N
    conc = max(1, args.concurrency)
    # conc > 1: the library's own prover pool (b200_pool: FIFO queue + `conc` worker threads, one context
    # each, keys shared) — the same C-ABI object a relayer's proof manager would hold
    pool = ProverPool(local_rank, workers=conc) if conc > 1 else None
    ctxs = [pool.context(i) for i in range(conc)] if pool else [rb.Context(local_rank)]
    ctx = ctxs[0]
    circ = make_circuit(args.circuit, LOG_N, CIRCUIT_SEED + rank)
    d_srs = torch.empty((n + 3, 8), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    # any n + 3 valid G1 points cost the same as a powers-of-tau SRS (the reference's real SRS file
    # is not on the GPU box); known-dlog points are generated on the device
    ctx.known_dlog_bases_device(SEED_SRS, n + 3, d_srs.data_ptr())
    srs = ctx.load_bases_device(d_srs.data_ptr(), n + 3)
    pk = PlonkKzgSnark.preprocess(ctx, srs, LOG_N, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    h_wires = torch.from_numpy(circ.wires.view(np.int64)).pin_memory()
    d_wires = h_wires.to(dev)
    torch.cuda.synchronize()
    blinders = [synth.splitmix_blinders(1000 * rank + i) for i in range(max(args.steps + args.warmup, args.warmup * conc, 2 * conc) + 8)]
    setup_s = time.perf_counter() - t_setup

    def run_proofs(count, wires_ptr, first_blinder, collect=None):
        """`count` proofs, `conc` in flight (pool workers, one context/stream each)."""
        if conc == 1:
            for i in range(count):
                proof = prove_raw(ctx, pk, wires_ptr, circ.pub_inputs, blinders[first_blinder + i])
                if collect is not None:
                    collect.append(plonk_last_timings(ctx))
            return proof
        tickets = [pool.submit_prove(pk, wires_ptr, circ.pub_inputs, blinders[first_blinder + i]) for i in range(count)]
        proof = None
        for tk in tickets:
            proof = pool.wait(tk)
        return proof

    # ---- proofs, witness resident in HBM ---------------------------------------------------------------
    for c in ctxs:  # CUDA-event timing of the dominant kernel over the timed region, every context; switched on BEFORE the
        c.msm_timing(True)  # warm-up: the timing events are nodes of the captured graphs, toggling it later would re-capture
    # warm-up in waves of `conc` (one proof per worker, all waited for): after W >= 3 waves every worker has run the key
    # eagerly, captured its rounds as CUDA graphs and replayed them at least once, so the timed region is steady state
    for wave in range(max(args.warmup, 3)):
        run_proofs(conc, d_wires.data_ptr(), (wave * conc) % max(1, len(blinders) - conc))
    for c in ctxs:
        c.msm_timing_totals(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    phases = []
    barrier()
    launches0 = ctx._lib.b200_kernel_launches()  # the library counts every kernel it launches (replayed graph nodes included)
    graphs0 = ctx._lib.b200_graph_launches()
    t = time.perf_counter()
    proof = run_proofs(args.steps, d_wires.data_ptr(), args.warmup, phases)
    barrier()
    dt = max_over_ranks(time.perf_counter() - t)
    gpu_launches = int(ctx._lib.b200_kernel_launches() - launches0)
    graph_launches = int(ctx._lib.b200_graph_launches() - graphs0)
    clocks = sampler.stop() if rank == 0 else None
    acc_tot = [c.msm_timing_totals(reset=True) for c in ctxs]
    if args.dump_outputs and rank == 0:
        dump_proof(args.dump_outputs, proof)  # the proof of the last timed step (blinders[warmup + steps - 1])
    # ---- the same through the public call with HOST buffers (e2e) ---------------------------------------
    run_proofs(2 * conc, h_wires.data_ptr(), 0)
    barrier()
    t = time.perf_counter()
    proof_e2e = run_proofs(args.steps, h_wires.data_ptr(), args.warmup)
    barrier()
    dt_e2e = max_over_ranks(time.perf_counter() - t)
    if conc == 1:
        assert bytes(proof) == bytes(proof_e2e)  # same witness + blinders -> identical proof
    # the same from PAGEABLE host memory (a plain numpy buffer): what an unregistered Rust Vec<Fr> costs
    p_wires = np.ascontiguousarray(circ.wires, dtype=np.uint64).copy()
    run_proofs(2 * conc, p_wires.ctypes.data, 0)
    barrier()
    t = time.perf_counter()
    run_proofs(args.steps, p_wires.ctypes.data, args.warmup)
    barrier()
    dt_pg = max_over_ranks(time.perf_counter() - t)
    e2e_pageable = {"value": world * args.steps / dt_pg, "unit": "proofs/s"}
    # steady state: a K-step run with `conc` in flight ramps up and drains (about one wave of `conc` proofs at each end);
    # the same loop over >= 200 proofs shows the rate without that edge
    steady = None
    if args.steps < 200:
        ss_steps = 200
        ss_bl = [synth.splitmix_blinders(77000 + i) for i in range(ss_steps)]

        def run_ss():
            if conc == 1:
                for i in range(ss_steps):
                    prove_raw(ctx, pk, d_wires.data_ptr(), circ.pub_inputs, ss_bl[i])
                return
            tks = [pool.submit_prove(pk, d_wires.data_ptr(), circ.pub_inputs, ss_bl[i]) for i in range(ss_steps)]
            for tk in tks:
                pool.wait(tk)
        barrier()
        t = time.perf_counter()
        run_ss()
        barrier()
        dt_ss = max_over_ranks(time.perf_counter() - t)
        steady = {"value": world * ss_steps / dt_ss, "unit": "proofs/s", "steps": ss_steps,
                  "note": "same loop, witness resident in HBM, 200 proofs: the K-step figure above includes ramp-up and drain"}

    # ---- kernel-level numbers of the dominant kernel inside a proof --------------------------------------
    # bucket accumulation of the batched commitments, timed with CUDA events on the library's stream
    ctx.msm_timing(True)
    msm_ms = []
    d_polys = torch.empty((5, n + 4, 4), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    for b in range(5):
        ctx.splitmix_fr_device(0xC0FFEE + b, n + 2, d_polys[b].data_ptr(), montgomery=True)
    import ctypes as C
    from renegade_b200 import _lib
    out5 = np.zeros((5, 8), dtype=np.uint64)
    for i in range(6):
        _lib.check(ctx._lib.b200_msm_batch_device(ctx._h, srs._h, 0, C.c_void_p(d_polys.data_ptr()), n + 2, n + 4, 5, 1,
                                                  out5.ctypes.data_as(C.c_void_p), None))
        if i >= 2:
            msm_ms.append(ctx.msm_timing(True))
    acc_ms_alone = sum(p["accumulate"] for p in msm_ms) / len(msm_ms)
    peak, peak_src = measured_peak_hbm()
    # live, over the timed region: algorithmic bytes of all accumulate launches / their summed event durations
    # (with several proofs in flight the launches share the SMs, so this is the in-situ figure)
    live_ms = sum(t["accumulate_ms"] for t in acc_tot)
    live_pairs = sum(t["pairs"] for t in acc_tot)
    live_launches = sum(t["launches"] for t in acc_tot)
    achieved = live_pairs * BYTES_PER_PAIR / (live_ms * 1e-3) / 1e9
    achieved_alone = 5 * (n + 2) * BYTES_PER_PAIR / (acc_ms_alone * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "msm_accumulate_traffic.json")) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    except Exception:
        pass

    # ---- single-proof latency (one proof in flight) and its phases -----------------------------------------
    lat_phases = []
    for i in range(8):
        prove_raw(ctx, pk, d_wires.data_ptr(), circ.pub_inputs, blinders[i])
        if i >= 2:
            lat_phases.append(plonk_last_timings(ctx))
    single = {k: sum(p[k] for p in lat_phases) / len(lat_phases) for k in lat_phases[0]}
    single_ms = sum(single.values())

    # ---- configs[2]: 2^20 NTT + iNTT round trip (device resident, CUDA events in the library) ------------
    ntt = None
    if not args.no_msm:
        nn = 1 << 20
        d_x = torch.empty((nn, 4), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        ctx.splitmix_fr_device(0x1177, nn, d_x.data_ptr(), montgomery=True)
        ref = d_x.clone()
        f_ms, i_ms = [], []
        for i in range(8):
            ctx.ntt_device(d_x.data_ptr(), 20, inverse=False)
            f = ctx.ntt_last_ms()
            ctx.ntt_device(d_x.data_ptr(), 20, inverse=True)
            if i >= 3:
                f_ms.append(f)
                i_ms.append(ctx.ntt_last_ms())
        rt_ms = min(f_ms) + min(i_ms)
        ntt = {"workload": "2^20-element BN254-Fr NTT + iNTT round trip (BASELINE.json configs[2])",
               "round_trip_ms": rt_ms, "fwd_ms": min(f_ms), "inv_ms": min(i_ms), "round_trip_ok": bool(torch.equal(d_x, ref)),
               "roofline": {"bound": "hbm", "achieved": nn * 128 / (rt_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": nn * 128 / (rt_ms * 1e-3) / 1e9 / peak, "kernel": "ntt_pass_kernel",
                            "note": "64 B per element per transform (SURVEY 8(d)); the kernel is bound by the integer "
                                    "pipe: 10 Fr products per element per transform"}}

    # ---- second clause: 2^20-point MSM per GPU, sharded across ranks -------------------------------------
    msm = None
    msm_traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "msm_accumulate_traffic_2_20.json")) as f:
            msm_traffic = json.load(f).get("dram_bytes_per_launch")
    except Exception:
        pass
    if not args.no_msm:
        nm = 1 << MSM_LOG_N
        first = rank * nm
        # the whole leg runs behind the C ABI: b200_multi_* = local Pippenger per GPU + ncclAllGather of the
        # 128-byte partials + W-term sum on every device (world = 1: the same code without the collective)
        multi = MultiGpu.from_torch_distributed(local_rank) if world > 1 else MultiGpu.single_process([local_rank])
        mctx = multi.ctx(0)
        mctx.msm_timing(True)
        mbases = multi.known_dlog_bases(SEED_BASES, world * nm)
        assert mbases.shard(0) == (first, first + nm)
        d_sc = torch.empty((nm, 4), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        mctx.splitmix_fr_device(SEED_SCALARS, nm, d_sc.data_ptr(), montgomery=False, first=first)
        h_sc = torch.empty((nm, 4), dtype=torch.int64).pin_memory()
        h_sc.copy_(d_sc)
        torch.cuda.synchronize()

        def msm_step(host):
            return multi.msm_local(mbases, [h_sc.data_ptr() if host else d_sc.data_ptr()], on_device=not host, montgomery=False)
        for _ in range(3):
            msm_step(False)
        mph = []
        barrier()
        t = time.perf_counter()
        for _ in range(args.msm_steps):
            r0 = msm_step(False)
            mph.append(mctx.msm_timing(True))
        barrier()
        mdt = max_over_ranks(time.perf_counter() - t) / args.msm_steps
        for _ in range(2):
            msm_step(True)
        barrier()
        t = time.perf_counter()
        for _ in range(args.msm_steps):
            r1 = msm_step(True)
        barrier()
        mdt_e2e = max_over_ranks(time.perf_counter() - t) / args.msm_steps
        assert (r0[0] == r1[0]).all()
        # closed form: the bases are a_i * G, so the result must be (sum a_i s_i mod r) * G.  Every rank folds its own
        # 2^20 products (device field multiplier, exact limb sums on the host), rank 0 adds them and checks with one
        # scalar multiplication — product code only, no oracle
        R_MOD = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
        d_a = torch.empty((nm, 4), dtype=torch.int64, device=dev)
        d_sm = torch.empty((nm, 4), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        mctx.splitmix_fr_device(SEED_BASES, nm, d_a.data_ptr(), montgomery=True, first=first)
        mctx.splitmix_fr_device(SEED_SCALARS, nm, d_sm.data_ptr(), montgomery=True, first=first)
        prod = mctx.field_op(0, 0, d_a.cpu().numpy().view(np.uint64), d_sm.cpu().numpy().view(np.uint64))  # mont(a_i s_i)
        cols = prod.view(np.uint32).reshape(-1, 8).astype(np.uint64).sum(axis=0)
        part = sum(int(cols[j]) << (32 * j) for j in range(8)) % R_MOD
        parts = [part]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, part)
        k_dlog = sum(parts) * pow(1 << 256, -1, R_MOD) % R_MOD  # out of Montgomery form
        Q_MOD = 0x30644e72e131a029b85045b68181585d97816a916871ca8d3c208c16d87cfd47
        gen = np.zeros((1, 8), dtype=np.uint64)  # G = (1, 2), coordinates in Montgomery form
        for off, v in ((0, 1), (4, 2)):
            mv = (v << 256) % Q_MOD
            gen[0, off:off + 4] = [(mv >> (64 * j)) & 0xffffffffffffffff for j in range(4)]
        gb = mctx.load_bases(gen)
        kk = np.array([[(k_dlog >> (64 * j)) & 0xffffffffffffffff for j in range(4)]], dtype=np.uint64)
        exp_xy, exp_inf = mctx.msm(gb, kk, montgomery=False)
        msm_verified = bool((not exp_inf) and (not r0[1]) and (r0[0] == exp_xy).all())
        gb.free()
        del d_a, d_sm
        macc = sum(p["accumulate"] for p in mph) / len(mph)
        mplan = multi_plan(multi, mbases)
        msm = {
            "workload": "2^20-point BN254 G1 Pippenger MSM per GPU (BASELINE.json configs[1]); N GPUs = one "
                        "N*2^20-point MSM sharded by point range behind the C ABI (b200_multi_msm_local): local Pippenger, "
                        "ncclAllGather of the 128-byte partial sums, W-term addition on every device",
            "verified": msm_verified,
            "verified_how": "result == (sum a_i s_i mod r) * G for the N*2^20 known-discrete-log bases (closed form, product code only)",
            "value": world * nm * BYTES_PER_PAIR / mdt / 1e9, "unit": "GB/s", "ms_per_step": mdt * 1e3,
            "points_per_sec": world * nm / mdt, "steps": args.msm_steps,
            "e2e": {"value": world * nm * BYTES_PER_PAIR / mdt_e2e / 1e9, "unit": "GB/s", "h2d_bytes_per_step": nm * 32,
                    "d2h_bytes_per_step": 128},
            "device_phases_ms": {k: sum(p[k] for p in mph) / len(mph) for k in ("total", "sort", "accumulate", "reduce")},
            "plan": mplan,
            "roofline": {"bound": "hbm", "achieved": nm * BYTES_PER_PAIR / (macc * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": nm * BYTES_PER_PAIR / (macc * 1e-3) / 1e9 / peak, "kernel": "msm_accumulate_kernel",
                         "traffic": msm_traffic,
                         # what actually bounds the kernel: Fq products on the IMAD.WIDE pipe.  A mixed addition is
                         # 8M + 2S with one fused pair = 9.5 product-equivalents of 128 IMAD.WIDE each; the pipe issues
                         # one warp-wide IMAD.WIDE per ~4 clk per SM sub-partition (tools/microbench.cu).
                         "int_pipe": {"achieved_gmul_per_s": nm * mplan["digits"] * 9.5 / (macc * 1e-3) / 1e9,
                                      "peak_gmul_per_s": 148 * 4 * 32 / (128 * 4.0) * 1.965,
                                      "frac": nm * mplan["digits"] * 9.5 / (macc * 1e-3) / 1e9 / (148 * 4 * 32 / (128 * 4.0) * 1.965),
                                      "measured_multiplier_gmul_per_s": 66.6}},
            "l2": "window tables %.0f MB + 32 MB of scalars per step vs 126 MB of L2" % (mplan["tables"] * nm * 64 / 1e6),
        }

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_step = dt / args.steps * 1e3
    out = base_line(args, world)
    out.update({
        "value": world * args.steps / dt, "ms_per_step": ms_step,
        "config": shared_config(args),
        "run": {"gates_used": circ.n_gates, "concurrency_per_gpu": conc,
                "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"),
                "prover_rounds": "replayed as CUDA graphs from the second proof of a key on a worker (B200_GRAPHS=%s)" % os.environ.get("B200_GRAPHS", "1"),
                "parallelism": "one proof stream per GPU (replicas, no collective)", "msm_plan": srs.plan,
                "l2": "working set > L2: shared key tables 227 MB + SRS window tables 67 MB, plus per proof in flight "
                      "7 x 12.6 MB extended polynomials and ~100 MB of MSM scratch, vs 126 MB of L2",
                "timing": "wall clock around K proofs, barrier + cuda synchronize on both sides, max over ranks; "
                          "kernel times from CUDA events on the library's stream",
                "host_buffers": "e2e passes the witness table from PINNED host memory (torch pin_memory); `e2e_pageable` "
                                "passes a plain malloc'd table — what a Rust Vec<Fr> is unless the shim registers it "
                                "(cudaHostRegister)"},
        "steady_state": steady, "e2e_pageable": e2e_pageable,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "msm_accumulate_kernel (the 4 batched commitments of every timed proof)",
                     "peak_source": peak_src, "launches_timed": live_launches,
                     "avg_launch_ms": live_ms / max(live_launches, 1.0), "avg_pairs_per_launch": live_pairs / max(live_launches, 1.0),
                     "achieved_kernel_alone": achieved_alone,
                     "note": "integer-multiply-pipe bound: ~9.5 Fq product-equivalents per bucket addition, one addition per "
                             "window digit (16 per scalar); `achieved` is in situ (several proofs share the SMs), "
                             "`achieved_kernel_alone` the same kernel timed alone; see DESIGN.md for the INT-pipe roofline"},
        "e2e": {"value": world * args.steps / dt_e2e, "unit": "proofs/s", "h2d_bytes_per_step": 5 * n * 32 + circ.num_inputs * 32 + 17 * 32,
                "d2h_bytes_per_step": 1152, "ms_per_step": dt_e2e / args.steps * 1e3},
        # counted by the library (b200_kernel_launches) around the timed region of this rank; the ncu launch list
        # of the same command is under profiles/ (tools/kernel_shares.py gives launches per proof)
        "gpu_launches": gpu_launches * world, "gpu_launches_per_proof": gpu_launches / max(args.steps, 1),
        # host submissions: from the second proof of a key on a worker each prover round is one CUDA-graph launch
        "graph_launches_per_proof": graph_launches / max(args.steps, 1),
        "latency_ms_one_proof_in_flight": single_ms, "latency_phases_ms": single,
        "clocks": clocks, "setup_s": setup_s, "msm": msm, "ntt": ntt,
    })

    if not args.no_cpu_baseline and world == 1:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_c  # CPU baseline leg: the only place the product arm executes the oracle
        oracle_c.autotune_threads()
        h_srs = d_srs.cpu().numpy().view(np.uint64)
        opk = oracle_c.plonk_preprocess(LOG_N, circ.selectors, circ.perm, circ.k, h_srs)
        bl = blinders[args.warmup + args.steps - 1]
        t = time.perf_counter()
        rc, oproof, _, _ = oracle_c.plonk_prove(LOG_N, circ.num_inputs, circ.k, opk, circ.wires, circ.pub_inputs, bl, h_srs)
        cdt = time.perf_counter() - t
        gproof = prove_raw(ctx, pk, d_wires.data_ptr(), circ.pub_inputs, bl)
        out["cpu_baseline"] = {
            "value": 1.0 / cdt, "unit": "proofs/s", "cores": oracle_c.num_threads(), "kind": "port",
            "sample": "1 full proof of the same circuit, same SRS and blinders (%.2f s)" % cdt,
            "bit_exact_vs_gpu": bool(rc == 0 and bytes(oproof) == bytes(gproof)),
            "note": "restated CPU prover (C + OpenMP; arkworks msm_bigint / radix-2 FFT algorithms, jellyfish "
                    "TurboPlonk rounds) — not the Rust reference itself",
        }
    if world == 1 and not args.no_real_statements:
        # extras, in a process of their own: nothing in them — an exception, a crash, a hang — may cost the headline line
        try:
            # the real statements are 8-16x smaller than the headline circuit: latency-bound per proof, so more of them are
            # kept in flight (B200_BENCH_EXTRAS_CONCURRENCY)
            xconc = int(os.environ.get("B200_BENCH_EXTRAS_CONCURRENCY", str(max(conc, 16))))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--extras-only", "--concurrency", str(xconc)] +
                               (["--no-cpu-baseline"] if args.no_cpu_baseline else []),
                               capture_output=True, text=True, timeout=420)
            extras = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            extras = {"real_statements": {"error": repr(e)[:300]}}
        out.update(extras)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
