"""Collaborative-prover latency on one GPU: P = 2 parties on device 0 (one context and one thread each, the in-process
local group as transport, dealer preprocessing made before each timed proof) at 2^12, 2^13, 2^14 and 2^16 gates.

    python tools/mpc_bench.py [--proofs 20] [--warmup 3] [--sizes 12,13,14,16] [--authenticated] [--json out.json]

Per size: median, p10 and p90 of the joint-proof wall time (both parties started to both finished), the milliseconds
party 0 spent inside all_gather (waiting for the other party included), bytes each party sent, exchanges, and the
single-prover latency (`b200_plonk_prove`) of the same circuit.  Also the host-orchestrated Python path
(`MultiproverPlonkKzgSnark` on `DeviceBackend`) at 2^12, and the GPU name and power limit.  With --authenticated, the
same numbers for `b200_mpc_prove_auth` (MAC-authenticated shares, dealer key and inputs), its proofs alternating with
the plain ones in the same loop."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

TAU = 0xB200B200B200


def pct(xs, q):
    return float(np.percentile(np.asarray(xs), q))


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                                      text=True, timeout=30).strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sizes", default="12,13,14,16")
    ap.add_argument("--python-proofs", type=int, default=3)
    ap.add_argument("--json", default=None)
    ap.add_argument("--authenticated", action="store_true")
    args = ap.parse_args()

    import oracle_c
    import bn254_py as py
    import renegade_b200 as rb
    from renegade_b200 import collaborative as co
    from renegade_b200 import synth
    from renegade_b200.backend import PlonkKzgSnark

    sizes = [int(s) for s in args.sizes.split(",")]
    ctx = rb.Context(0)
    parties = [rb.Context(0) for _ in range(2)]
    tau = oracle_c.int_to_limbs(py.to_mont(TAU % py.R, py.R))
    srs = oracle_c.srs_from_tau(tau, (1 << max(sizes)) + 3)
    name, limit = gpu_info()
    report = {"gpu": name, "power_limit": limit, "parties": 2, "sizes": {}}
    print(f"{name}, power limit {limit}; 2 parties on device 0, local-group transport, dealer preprocessing")
    for log_n in sizes:
        n = 1 << log_n
        circ = synth.synth_circuit(log_n, num_inputs=5, seed=500 + log_n, check=False)
        bases = ctx.load_bases(srs[:n + 3])
        pk = PlonkKzgSnark.preprocess(ctx, bases, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
        bl = synth.splitmix_blinders(40 + log_n)
        single, _ = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, bl)
        ts = []
        for _ in range(args.warmup + args.proofs):
            t0 = time.perf_counter()
            PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, bl)
            ts.append((time.perf_counter() - t0) * 1e3)
        single_ms = float(np.median(ts[args.warmup:]))
        ws = co.share_table(np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), 2, seed=1)
        bs = co.share_table(np.asarray(bl, dtype=np.uint64).reshape(-1, 4), 2, seed=2)
        table = np.concatenate([np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), np.asarray(bl, dtype=np.uint64).reshape(-1, 4)])

        def joint(seed, auth):
            """One timed joint proof: (wall ms, party 0's stats)."""
            group = co.LocalGroup(2, 600000)
            trs = [group.transport(p) for p in range(2)]
            if auth:
                made = [co.MpcPrep.dealer_auth(parties[p], pk, seed, p, 2) for p in range(2)]
                preps = [m[0] for m in made]
                ins = [co.dealer_share_auth(parties[p], seed, p, 2, table) for p in range(2)]
                k = 5 * n
                fns = [lambda p=p: co.prove_party_auth(parties[p], pk, trs[p], preps[p], made[p][1], ins[p][0][:k], ins[p][1][:k],
                                                       circ.pub_inputs, ins[p][0][k:], ins[p][1][k:]) for p in range(2)]
            else:
                preps = [co.MpcPrep.dealer(parties[p], pk, seed, p, 2) for p in range(2)]
                fns = [lambda p=p: co.prove_party(parties[p], pk, trs[p], preps[p], ws[p], circ.pub_inputs, bs[p]) for p in range(2)]
            t0 = time.perf_counter()
            res = co._run_parties(fns)
            dt = (time.perf_counter() - t0) * 1e3
            for r in res:
                if isinstance(r, Exception):
                    raise r
                assert bytes(r.proof) == bytes(single), "joint proof differs from the single-prover proof"
            for pr in preps:
                pr.free()
            group.close()
            return dt, res[0].stats

        modes = [False, True] if args.authenticated else [False]
        lat = {m: [] for m in modes}
        gather = {m: [] for m in modes}
        stats = {}
        for i in range(args.warmup + args.proofs):
            for m in modes:  # alternating, so that both modes see the same host and device conditions
                dt, st = joint(77 + i, m)
                if i >= args.warmup:
                    lat[m].append(dt)
                    gather[m].append(st["all_gather_ms"])
                    stats[m] = st
        for m in modes:
            row = {"joint_ms_median": float(np.median(lat[m])), "joint_ms_p10": pct(lat[m], 10), "joint_ms_p90": pct(lat[m], 90),
                   "all_gather_ms_median": float(np.median(gather[m])), "bytes_sent": stats[m]["bytes_sent"],
                   "exchanges": stats[m]["exchanges"], "triples": stats[m]["triples"], "single_prover_ms": single_ms,
                   "proofs": args.proofs}
            report["sizes"][f"2^{log_n}" + (" authenticated" if m else "")] = row
            print(f"2^{log_n}{' authenticated' if m else ''}: joint {row['joint_ms_median']:.1f} ms (p10 {row['joint_ms_p10']:.1f}, "
                  f"p90 {row['joint_ms_p90']:.1f}), in all_gather {row['all_gather_ms_median']:.1f} ms, sent "
                  f"{row['bytes_sent'] / 1e6:.1f} MB in {row['exchanges']} exchanges; single prover {single_ms:.2f} ms", flush=True)
        pk.free()
    # the host-orchestrated Python protocol at 2^12, same run
    log_n = 12
    n = 1 << log_n
    circ = synth.synth_circuit(log_n, num_inputs=5, seed=500 + log_n, check=False)
    bases = ctx.load_bases(srs[:n + 3])
    be = co.DeviceBackend(ctx, bases)
    cpk = co.CollaborativeProvingKey.build(be, log_n, circ.num_inputs, circ.selectors, circ.perm, circ.k)
    bl = synth.splitmix_blinders(40 + log_n)
    ws = co.share_table(np.asarray(circ.wires, dtype=np.uint64).reshape(-1, 4), 2, seed=1)
    bs = co.share_table(np.asarray(bl, dtype=np.uint64).reshape(-1, 4), 2, seed=2)
    co.MultiproverPlonkKzgSnark.prove_with_link_hint(be, cpk, ws, circ.pub_inputs, bs)
    ts = []
    for _ in range(args.python_proofs):
        t0 = time.perf_counter()
        co.MultiproverPlonkKzgSnark.prove_with_link_hint(be, cpk, ws, circ.pub_inputs, bs)
        ts.append((time.perf_counter() - t0) * 1e3)
    report["python_path_2^12_ms_median"] = float(np.median(ts))
    print(f"Python path (collaborative.py) at 2^12: {np.median(ts):.1f} ms median of {args.python_proofs}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(report, f, indent=1)
    for c in parties:
        c.close()
    ctx.close()


if __name__ == "__main__":
    main()
