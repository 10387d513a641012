"""Batch verifier vs the serial host verifiers, on one GPU: items/s per batch size N.

A few distinct PlonK proofs (2^10 and 2^13, with the public-input counts of the example statements: 17 as the private
settlement, 13 as VALID BALANCE CREATE, 9 as the fee payments) and link proofs are made with the device prover on an
SRS of known tau, replicated into batches of N = 1, 16, 256, 1024 (proofs and links 3:1), and checked with
`b200_plonk_batch_verify` and with the `b200_plonk_verify` / `b200_plonk_verify_link` loop on the same items.  Then one
failing batch of 1024 with one bad item, with the pairing products its bisection used.  Prints one JSON line.

    python tools/verify_bench.py [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

import numpy as np  # noqa: E402

import renegade_b200 as rb  # noqa: E402
from renegade_b200 import synth  # noqa: E402
from renegade_b200.backend import (B200BatchLink, B200BatchProof, B200BatchVk, GroupLayout, PlonkKzgSnark,  # noqa: E402
                                   VerifyingKey, link_proofs, verify_link_proof, pairing_check)

TAU = 0xB200B200B200
LAYOUT = GroupLayout(alignment=9, offset=20, size=16)


def setup(ctx):
    import bn254_pairing_py as pr
    import bn254_py as py
    import oracle_c
    oracle_c.build()
    srs = oracle_c.srs_from_tau(oracle_c.int_to_limbs(py.to_mont(TAU % py.R, py.R)), (1 << 13) + 3)
    raw = np.frombuffer(open(os.path.join(ROOT, "tests", "golden", "srs_g2.bin"), "rb").read(), dtype=np.uint64)
    h = raw[:16].copy()
    tau_h = np.frombuffer(pr.encode_g2_mont(pr.g2_mul(pr.decode_g2_mont(h.tobytes(), 0), TAU)), dtype=np.uint64).copy()
    bases = ctx.load_bases(srs)
    vals = [(i * 0x9E3779B97F4A7C15 + 3) % py.R for i in range(LAYOUT.size)]
    proofs, hints = [], []
    for log_n, ni, seed in ((13, 13, 1), (10, 17, 2), (13, 9, 3), (10, 9, 4)):
        circ = synth.synth_circuit(log_n, num_inputs=ni, seed=seed, link=(LAYOUT.alignment, LAYOUT.offset, vals))
        pk = PlonkKzgSnark.preprocess(ctx, bases, log_n, ni, circ.selectors, circ.perm, circ.k)
        proof, hint = PlonkKzgSnark.prove_with_link_hint(ctx, pk, circ.wires, circ.pub_inputs, synth.splitmix_blinders(seed))
        proofs.append((VerifyingKey.from_proving_key(pk, h, tau_h), circ.pub_inputs, proof))
        hints.append(hint)
        pk.free()
    links = []
    for a, b in ((0, 1), (2, 3)):
        lp, _ = link_proofs(ctx, bases, hints[a], hints[b], LAYOUT)
        links.append((hints[a].linking_wire_comm, hints[b].linking_wire_comm, lp, LAYOUT))
    bases.free()
    return proofs, links, h, tau_h


class RawBatch:
    """The ctypes arrays of one batch, built once so that the timed region is the library call."""

    def __init__(self, proofs, links, h, tau_h):
        self.keep, vks, index = [], [], {}
        for vk, _, _ in proofs:
            if id(vk) not in index:
                index[id(vk)] = len(vks)
                arrs = [np.ascontiguousarray(x, dtype=np.uint64) for x in (vk.k, vk.selector_comms, vk.sigma_comms)]
                self.keep.append(arrs)
                vks.append(B200BatchVk(vk.log_n, vk.num_inputs, *(a.ctypes.data_as(C.c_void_p) for a in arrs)))
        self.vks = (B200BatchVk * len(vks))(*vks)
        self.proofs = (B200BatchProof * len(proofs))()
        for i, (vk, pi, proof) in enumerate(proofs):
            pia = np.ascontiguousarray(pi, dtype=np.uint64)
            self.keep.append(pia)
            self.proofs[i] = B200BatchProof(index[id(vk)], pia.ctypes.data_as(C.c_void_p), pia.shape[0], C.addressof(proof))
        self.links = (B200BatchLink * max(len(links), 1))()
        for i, (ca, cb, lp, lay) in enumerate(links):
            ca, cb = np.ascontiguousarray(ca, dtype=np.uint64), np.ascontiguousarray(cb, dtype=np.uint64)
            self.keep.append((ca, cb))
            self.links[i] = B200BatchLink(ca.ctypes.data_as(C.c_void_p), cb.ctypes.data_as(C.c_void_p), lay.alignment,
                                          lay.offset, lay.size, C.addressof(lp))
        self.n_vks, self.n_proofs, self.n_links = len(vks), len(proofs), len(links)
        self.h, self.tau_h = h, tau_h
        self.flags = np.zeros(len(proofs) + len(links), dtype=np.uint8)

    def run(self, ctx):
        ok, pairings = C.c_int(0), C.c_size_t(0)
        rb._lib.check(ctx._lib.b200_plonk_batch_verify(
            ctx._h, self.vks, self.n_vks, self.proofs, self.n_proofs, self.links, self.n_links,
            self.h.ctypes.data_as(C.c_void_p), self.tau_h.ctypes.data_as(C.c_void_p), C.byref(ok),
            self.flags.ctypes.data_as(C.c_void_p), None, C.byref(pairings)))
        return bool(ok.value), pairings.value


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    ctx = rb.Context(0)
    proofs, links, h, tau_h = setup(ctx)
    # one 2-pair pairing product on the host (what the batch call adds per pairing)
    g = np.zeros(8, dtype=np.uint64)
    import bn254_py as py
    g[:] = np.frombuffer(py.encode_g1_mont(py.G1_GEN), dtype=np.uint64)
    pairing_check([g, g], [tau_h, h])
    t = time.perf_counter()
    for _ in range(args.reps):
        pairing_check([g, g], [tau_h, h])
    pairing_ms = (time.perf_counter() - t) * 1e3 / args.reps
    result = {"gpu": gpu_info(), "cpu": cpu_model(), "pairing_product_ms": round(pairing_ms, 3), "sizes": {}}
    for n in (1, 16, 256, 1024):
        n_links = n // 4
        items_p = [proofs[i % len(proofs)] for i in range(n - n_links)]
        items_l = [links[i % len(links)] for i in range(n_links)]
        batch = RawBatch(items_p, items_l, h, tau_h)
        ok, _ = batch.run(ctx)  # warm-up
        assert ok, "honest batch rejected"
        t = time.perf_counter()
        for _ in range(args.reps):
            batch.run(ctx)
        batch_ms = (time.perf_counter() - t) * 1e3 / args.reps
        host_reps = 1 if n >= 256 else args.reps
        t = time.perf_counter()
        for _ in range(host_reps):
            for vk, pi, proof in items_p:
                assert PlonkKzgSnark.verify(vk, pi, proof)
            for ca, cb, lp, lay in items_l:
                assert verify_link_proof(ca, cb, lp, lay, h, tau_h)
        host_ms = (time.perf_counter() - t) * 1e3 / host_reps
        result["sizes"][str(n)] = {
            "batch_ms": round(batch_ms, 3), "batch_items_per_s": round(n / batch_ms * 1e3, 1),
            # the call's time less its one pairing product: the device stages, copies and the rho hash
            "batch_device_and_transfer_ms": round(batch_ms - pairing_ms, 3),
            "host_serial_ms": round(host_ms, 3), "host_items_per_s": round(n / host_ms * 1e3, 1)}
    # one bad item in 1024: the opening of link 777 moved by G
    n, n_links = 1024, 256
    items_p = [proofs[i % len(proofs)] for i in range(n - n_links)]
    items_l = [links[i % len(links)] for i in range(n_links)]
    ca, cb, lp, lay = items_l[777 - (n - n_links)]
    bad = type(lp).from_buffer_copy(bytes(lp))
    moved = py.g1_add(py.decode_g1_mont(np.asarray(lp.opening_proof, dtype=np.uint64).tobytes(), 0), py.G1_GEN)
    for j, v in enumerate(np.frombuffer(py.encode_g1_mont(moved), dtype=np.uint64)):
        bad.opening_proof[j] = int(v)
    items_l[777 - (n - n_links)] = (ca, cb, bad, lay)
    batch = RawBatch(items_p, items_l, h, tau_h)
    t = time.perf_counter()
    ok, pairings = batch.run(ctx)
    fail_ms = (time.perf_counter() - t) * 1e3
    assert not ok and np.flatnonzero(batch.flags == 0).tolist() == [777]
    result["failing_1024"] = {"ms": round(fail_ms, 3), "pairing_products": pairings, "bad_items_found": [777]}
    print(json.dumps(result))
    ctx.close()


if __name__ == "__main__":
    main()
