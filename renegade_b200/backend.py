"""Host-side mirror of the reference's interface for the proving hot path, over the C ABI.

Names follow the Rust surface the reference calls (SURVEY.md §8(a)/(b)):

  parse_ptau_file                      crates/circuits/circuit-types/src/primitives/srs.rs:63-71
  UnivariateUniversalParams            jf-primitives (built at srs.rs:70)
  VariableBaseMSM.msm_bigint           ark-ec 0.4.2 (under UnivariateKzgPCS::commit)
  UnivariateKzgPCS.commit              jf-primitives (reached from traits.rs:850,996)
  Radix2EvaluationDomain               ark-poly 0.4.2 (fft / ifft / coset_fft / coset_ifft)

Field elements are numpy uint64 arrays with a trailing dimension of 4 (little-endian limbs,
Montgomery form unless stated), G1 affine points have a trailing dimension of 8 (x || y).
All arithmetic runs in libb200prover.so on the GPU; nothing here computes on the host.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib

MAX_SRS_POWER = 17
MAX_SRS_DEGREE = (1 << MAX_SRS_POWER) + 2  # srs.rs:44-47


def _ptr(a: np.ndarray):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA device + stream + scratch (b200_ctx).  Calls on one context are serialised."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self._lib.b200_init(device, C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200_shutdown(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def use_graphs(self, on: bool = True):
        """Replay the prover's rounds as CUDA graphs from the second proof of a key on (default: on; B200_GRAPHS=0)."""
        _lib.check(self._lib.b200_ctx_use_graphs(self._h, int(on)))

    def kernel_launches(self) -> int:
        """Kernels the library has launched (or replayed inside graphs) in this process so far."""
        return int(self._lib.b200_kernel_launches())

    def graph_launches(self) -> int:
        return int(self._lib.b200_graph_launches())

    # ---- bases / SRS ------------------------------------------------------------------------
    def load_bases(self, points, window_bits: int = 0, check_on_curve: bool = False) -> "Bases":
        """points: (n, 8) uint64 array or bytes of 64-byte records."""
        if isinstance(points, (bytes, bytearray, memoryview)):
            buf = np.frombuffer(bytes(points), dtype=np.uint64).reshape(-1, 8)
        else:
            buf = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
        h = C.c_void_p()
        _lib.check(self._lib.b200_bases_load(self._h, _ptr(buf), buf.shape[0], window_bits,
                                             int(check_on_curve), C.byref(h)))
        return Bases(self, h)

    def load_bases_device(self, d_ptr: int, n: int, window_bits: int = 0) -> "Bases":
        h = C.c_void_p()
        _lib.check(self._lib.b200_bases_load_device(self._h, C.c_void_p(d_ptr), n, window_bits, C.byref(h)))
        return Bases(self, h)

    # ---- MSM --------------------------------------------------------------------------------
    def msm(self, bases: "Bases", scalars: np.ndarray, montgomery: bool = False, base_off: int = 0):
        s = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        out = np.zeros(8, dtype=np.uint64)
        inf = C.c_int(0)
        _lib.check(self._lib.b200_msm(self._h, bases._h, base_off, _ptr(s), s.shape[0], int(montgomery),
                                      _ptr(out), C.byref(inf)))
        return out, bool(inf.value)

    def msm_device(self, bases: "Bases", d_scalars: int, n: int, montgomery: bool = False, base_off: int = 0):
        out = np.zeros(8, dtype=np.uint64)
        inf = C.c_int(0)
        _lib.check(self._lib.b200_msm_device(self._h, bases._h, base_off, C.c_void_p(d_scalars), n,
                                             int(montgomery), _ptr(out), C.byref(inf)))
        return out, bool(inf.value)

    def msm_timing(self, enable: bool = True) -> dict:
        """Enable device-side phase timing; returns the last MSM's phases in ms."""
        arr = (C.c_float * 4)()
        _lib.check(self._lib.b200_msm_timing(self._h, int(enable), C.byref(arr)))
        return {"total": arr[0], "sort": arr[1], "accumulate": arr[2], "reduce": arr[3]}

    def msm_tuning(self, throughput_mode: bool) -> None:
        """False (default): latency-tuned MSM; True: throughput-tuned (longer per-thread chains in the bucket
        reduction, fewer operations) — same results, for when several MSMs are in flight on the GPU."""
        _lib.check(self._lib.b200_msm_tuning(self._h, int(throughput_mode)))

    def msm_timing_totals(self, reset: bool = False) -> dict:
        """Bucket-accumulation totals since the last reset (timing must be enabled): ms, pairs, launches."""
        arr = (C.c_double * 3)()
        _lib.check(self._lib.b200_msm_timing_totals(self._h, int(reset), C.byref(arr)))
        return {"accumulate_ms": arr[0], "pairs": arr[1], "launches": arr[2]}

    def ntt_last_ms(self) -> float:
        v = C.c_float(0)
        _lib.check(self._lib.b200_ntt_last_ms(self._h, C.byref(v)))
        return v.value

    def g1_sum_affine(self, points: np.ndarray, is_identity=None):
        p = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
        flags = None
        if is_identity is not None:
            flags = (C.c_int * p.shape[0])(*[int(bool(x)) for x in is_identity])
        out = np.zeros(8, dtype=np.uint64)
        inf = C.c_int(0)
        _lib.check(self._lib.b200_g1_sum_affine(_ptr(p), flags, p.shape[0], _ptr(out), C.byref(inf)))
        return out, bool(inf.value)

    # ---- NTT --------------------------------------------------------------------------------
    def ntt(self, data: np.ndarray, inverse: bool = False, coset: bool = False) -> np.ndarray:
        out = np.array(data, dtype=np.uint64, copy=True, order="C").reshape(-1, 4)
        n = out.shape[0]
        log_n = n.bit_length() - 1
        if n == 0 or (1 << log_n) != n:
            raise ValueError("domain size must be a power of two")
        _lib.check(self._lib.b200_ntt(self._h, _ptr(out), log_n, int(inverse), int(coset)))
        return out

    def ntt_device(self, d_ptr: int, log_n: int, inverse: bool = False, coset: bool = False,
                   batch: int = 1, stride: int | None = None) -> None:
        stride = (1 << log_n) if stride is None else stride
        _lib.check(self._lib.b200_ntt_device(self._h, C.c_void_p(d_ptr), log_n, int(inverse), int(coset),
                                             batch, stride))

    def domain_generator(self, log_n: int) -> np.ndarray:
        out = np.zeros(4, dtype=np.uint64)
        _lib.check(self._lib.b200_domain_generator(self._h, log_n, _ptr(out)))
        return out

    # ---- synthetic inputs (device) ------------------------------------------------------------
    def splitmix_fr_device(self, seed: int, n: int, d_out: int, montgomery: bool, first: int = 0) -> None:
        _lib.check(self._lib.b200_splitmix_fr_device(self._h, seed, first, n, int(montgomery), C.c_void_p(d_out)))

    def known_dlog_bases_device(self, seed: int, n: int, d_out: int, first: int = 0) -> None:
        _lib.check(self._lib.b200_known_dlog_bases_device(self._h, seed, first, n, C.c_void_p(d_out)))

    # ---- self tests -----------------------------------------------------------------------------
    def selftest_field(self, seed: int, iters: int) -> int:
        bad = C.c_uint64(0)
        _lib.check(self._lib.b200_selftest_field(self._h, seed, iters, C.byref(bad)))
        return bad.value

    def field_op(self, field: int, op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
        b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 4)
        out = np.zeros_like(a)
        _lib.check(self._lib.b200_field_op(self._h, field, op, _ptr(a), _ptr(b), a.shape[0], _ptr(out)))
        return out


class Bases:
    """Device-resident G1 bases with their precomputed window tables (b200_bases)."""

    def __init__(self, ctx: Context, handle):
        self._ctx = ctx
        self._h = handle

    def __len__(self) -> int:
        return int(self._ctx._lib.b200_bases_len(self._h))

    @property
    def plan(self) -> dict:
        arr = (C.c_int * 4)()
        self._ctx._lib.b200_bases_plan(self._h, C.byref(arr))
        return {"window_bits": arr[0], "digits": arr[1], "physical_windows": arr[2], "tables": arr[3]}

    def free(self):
        if self._h:  # a context that is already gone is passed as NULL (the library allows it)
            self._ctx._lib.b200_bases_free(self._ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# Reference-shaped interface
# ---------------------------------------------------------------------------------------------
@dataclass
class UnivariateUniversalParams:
    """jf-primitives `UnivariateUniversalParams<Bn254>` as built at srs.rs:70: the G1 powers
    live on the device; `powers_of_g_host` keeps the raw 64-byte records for inspection."""
    powers_of_g: Bases
    powers_of_g_host: np.ndarray


def parse_ptau_file(ctx: Context, data: bytes, window_bits: int = 0,
                    check_on_curve: bool = True, count: int | None = None) -> UnivariateUniversalParams:
    """srs.rs:63-71: header/section checks, MAX_SRS_DEGREE+1 G1 powers, on-curve assertion
    (srs.rs:178-179, run on the device).  `count` overrides the number of powers kept (the
    reference always keeps MAX_SRS_DEGREE + 1; smaller values serve truncated test files)."""
    lib = _lib.load()
    buf = (C.c_char * len(data)).from_buffer_copy(data)
    rec = C.c_void_p()
    n = C.c_size_t()
    _lib.check(lib.b200_srs_parse_ptau(C.cast(buf, C.c_void_p), len(data), C.byref(rec), C.byref(n)))
    need = MAX_SRS_DEGREE + 1 if count is None else count
    if n.value < need:
        raise _lib.B200Error(-4, f"ptau: only {n.value} G1 records available, need {need}")
    off = rec.value - C.addressof(buf)
    host = np.frombuffer(data, dtype=np.uint64, count=need * 8, offset=off).reshape(need, 8).copy()
    bases = ctx.load_bases(host, window_bits=window_bits, check_on_curve=check_on_curve)
    return UnivariateUniversalParams(powers_of_g=bases, powers_of_g_host=host)


class VariableBaseMSM:
    """ark-ec 0.4.2 `VariableBaseMSM`."""

    @staticmethod
    def msm_bigint(ctx: Context, bases: Bases, bigints: np.ndarray):
        """sum_i bigints[i] * bases[i]; bigints canonical (`BigInt<4>`).  Returns the affine
        result (x||y Montgomery, identity flag) — what `.into_affine()` yields."""
        return ctx.msm(bases, bigints, montgomery=False)


class UnivariateKzgPCS:
    """jf-primitives `UnivariateKzgPCS`."""

    @staticmethod
    def commit(ctx: Context, prover_param: Bases, poly_coeffs: np.ndarray):
        """Commitment to a dense polynomial given by Montgomery `Fr` coefficients: the
        Montgomery->canonical conversion jf-primitives does on the CPU
        (`convert_to_bigints`) is fused into the device digit extraction."""
        return ctx.msm(prover_param, poly_coeffs, montgomery=True)


class Radix2EvaluationDomain:
    """ark-poly 0.4.2 `Radix2EvaluationDomain<Fr>`: natural order in and out."""

    def __init__(self, ctx: Context, num_coeffs: int):
        size = 1
        while size < num_coeffs:
            size <<= 1
        self.ctx = ctx
        self.size = size
        self.log_size_of_group = size.bit_length() - 1
        self.group_gen = ctx.domain_generator(self.log_size_of_group)

    def _pad(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.uint64).reshape(-1, 4)
        if x.shape[0] > self.size:
            raise ValueError("more coefficients than the domain size")
        if x.shape[0] < self.size:  # ark-poly resizes with zeros
            x = np.concatenate([x, np.zeros((self.size - x.shape[0], 4), dtype=np.uint64)])
        return x

    def fft(self, coeffs: np.ndarray) -> np.ndarray:
        return self.ctx.ntt(self._pad(coeffs), inverse=False, coset=False)

    def ifft(self, evals: np.ndarray) -> np.ndarray:
        return self.ctx.ntt(self._pad(evals), inverse=True, coset=False)

    def coset_fft(self, coeffs: np.ndarray) -> np.ndarray:
        return self.ctx.ntt(self._pad(coeffs), inverse=False, coset=True)

    def coset_ifft(self, evals: np.ndarray) -> np.ndarray:
        return self.ctx.ntt(self._pad(evals), inverse=True, coset=True)


# ---------------------------------------------------------------------------------------------
# TurboPlonk prover (boundary B2)
# ---------------------------------------------------------------------------------------------
class B200Proof(C.Structure):
    """b200_proof: field order of the reference's `PlonkProof` (plonk_proof_def.rs:197-222)."""
    _fields_ = [
        ("wires_poly_comms", (C.c_uint64 * 8) * 5),
        ("prod_perm_poly_comm", C.c_uint64 * 8),
        ("split_quot_poly_comms", (C.c_uint64 * 8) * 5),
        ("opening_proof", C.c_uint64 * 8),
        ("shifted_opening_proof", C.c_uint64 * 8),
        ("wires_evals", (C.c_uint64 * 4) * 5),
        ("wire_sigma_evals", (C.c_uint64 * 4) * 4),
        ("perm_next_eval", C.c_uint64 * 4),
    ]

    def to_array(self) -> np.ndarray:
        return np.frombuffer(bytes(self), dtype=np.uint64).copy()


@dataclass
class LinkingHint:
    """mpc-plonk `LinkingHint` (plonk_proof_def.rs:143-150)."""
    linking_wire_poly: np.ndarray
    linking_wire_comm: np.ndarray


class ProvingKey:
    """Device-resident `ProvingKey` + the `VerifyingKey` commitments (b200_pk)."""

    def __init__(self, ctx: Context, handle, log_n: int, num_inputs: int, k: np.ndarray):
        self._ctx, self._h = ctx, handle
        self.log_n, self.num_inputs, self.k = log_n, num_inputs, k
        self.selector_comms = np.zeros((13, 8), dtype=np.uint64)
        self.sigma_comms = np.zeros((5, 8), dtype=np.uint64)
        _lib.check(ctx._lib.b200_pk_verifying_key(handle, _ptr(self.selector_comms), _ptr(self.sigma_comms)))

    @property
    def domain_size(self) -> int:
        return 1 << self.log_n

    def free(self):
        if self._h:
            self._ctx._lib.b200_pk_free(self._ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class VerifyingKey:
    """mpc-plonk `VerifyingKey<Bn254>` flattened: domain size, public-input count, coset representatives, the 13
    selector and 5 sigma commitments, and the two G2 elements of the `open_key` (`h`, `beta_h`: 128-byte ptau
    records x0 || x1 || y0 || y1, srs.rs:185-199).  Plain host data: verification needs no device."""
    log_n: int
    num_inputs: int
    k: np.ndarray
    selector_comms: np.ndarray
    sigma_comms: np.ndarray
    g2_h: np.ndarray
    g2_tau_h: np.ndarray

    @staticmethod
    def from_proving_key(pk: "ProvingKey", g2_h: np.ndarray, g2_tau_h: np.ndarray) -> "VerifyingKey":
        return VerifyingKey(pk.log_n, pk.num_inputs, pk.k, pk.selector_comms, pk.sigma_comms, g2_h, g2_tau_h)


def _u64(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.reshape(shape) if shape is not None else a


def pairing_check(g1_points, g2_points) -> bool:
    """prod e(P_i, Q_i) == 1 (`b200_pairing_check`; host only).  P_i: 8 x uint64, Q_i: 16 x uint64."""
    lib = _lib.load()
    p = _u64(np.stack([_u64(x) for x in g1_points]), (-1, 8))
    q = _u64(np.stack([_u64(x) for x in g2_points]), (-1, 16))
    if p.shape[0] != q.shape[0]:
        raise ValueError("one G2 point per G1 point")
    one = C.c_int(0)
    _lib.check(lib.b200_pairing_check(_ptr(p), _ptr(q), p.shape[0], C.byref(one)))
    return bool(one.value)


def verify_link_proof(comm_a: np.ndarray, comm_b: np.ndarray, proof: "B200LinkProof", layout: "GroupLayout",
                      g2_h: np.ndarray, g2_tau_h: np.ndarray) -> bool:
    """`PlonkKzgSnark::verify_link_proof::<SolidityTranscript>` (proof_linking/intent_only.rs:77-84)."""
    ok = C.c_int(0)
    _lib.check(_lib.load().b200_plonk_verify_link(_ptr(_u64(comm_a)), _ptr(_u64(comm_b)), layout.alignment, layout.offset,
                                                  layout.size, C.byref(proof), _ptr(_u64(g2_h)), _ptr(_u64(g2_tau_h)),
                                                  C.byref(ok)))
    return bool(ok.value)


class PlonkKzgSnark:
    """mpc-plonk `PlonkKzgSnark<Bn254>` as called at traits.rs:850, traits.rs:996 and traits.rs:1012."""

    @staticmethod
    def verify(vk: VerifyingKey, pub_inputs: np.ndarray, proof: "B200Proof") -> bool:
        """`PlonkKzgSnark::verify::<SolidityTranscript>(&vk, &public_inputs, &proof, None)` (traits.rs:1012-1018).
        Host only."""
        pi = _u64(pub_inputs, (-1, 4))
        if pi.shape[0] != vk.num_inputs:
            return False  # the reference's verifier errors on a wrong public-input count: not accepted
        ok = C.c_int(0)
        _lib.check(_lib.load().b200_plonk_verify(vk.log_n, vk.num_inputs, _ptr(_u64(vk.k, (5, 4))),
                                                 _ptr(_u64(vk.selector_comms, (13, 8))), _ptr(_u64(vk.sigma_comms, (5, 8))),
                                                 _ptr(pi) if pi.size else None, C.byref(proof), _ptr(_u64(vk.g2_h)),
                                                 _ptr(_u64(vk.g2_tau_h)), C.byref(ok)))
        return bool(ok.value)

    @staticmethod
    def batch_verify(ctx: Context, vks, public_inputs, proofs, links=(), want_operands: bool = False, g2=None):
        """Verifies many proofs and link proofs on the device with one pairing product (`b200_plonk_batch_verify`).

        vks[i], public_inputs[i], proofs[i] describe proof i; links are (comm_a, comm_b, B200LinkProof, GroupLayout).
        Returns a numpy bool array of per-item verdicts, proofs first, each what `verify` / `verify_link_proof` says
        for that item alone (a wrong public-input count is False).  With want_operands, also the (n, 2, 8) uint64 array
        of each item's unweighted pairing operands (A_j, B_j).  The G2 pair (h, beta_h) comes from the verifying keys,
        which must agree on it, or from `g2` for a batch of link proofs only.  `ctx` runs the device work: give the verifier a context of its own (not a prover pool worker's)."""
        vks, public_inputs, proofs, links = list(vks), list(public_inputs), list(proofs), list(links)
        if not (len(vks) == len(public_inputs) == len(proofs)):
            raise ValueError("vks, public_inputs and proofs must have the same length")
        if not vks and not links:
            raise ValueError("empty batch")
        if vks:
            g2_h, g2_tau_h = _u64(vks[0].g2_h, (16,)), _u64(vks[0].g2_tau_h, (16,))
        elif g2 is not None:
            g2_h, g2_tau_h = _u64(g2[0], (16,)), _u64(g2[1], (16,))
        else:
            raise ValueError("a batch of link proofs only needs the G2 pair: pass g2=(h, beta_h)")
        keep = []  # every array whose address goes into the call stays referenced here until it returns
        table, index = [], {}
        for vk in vks:
            if not (np.array_equal(_u64(vk.g2_h, (16,)), g2_h) and np.array_equal(_u64(vk.g2_tau_h, (16,)), g2_tau_h)):
                raise ValueError("verifying keys of one batch must share the G2 elements")
            if id(vk) not in index:
                index[id(vk)] = len(table)
                arrs = (_u64(vk.k, (5, 4)), _u64(vk.selector_comms, (13, 8)), _u64(vk.sigma_comms, (5, 8)))
                keep.append(arrs)
                table.append(B200BatchVk(vk.log_n, vk.num_inputs, *(_ptr(a) for a in arrs)))
        bp = (B200BatchProof * len(proofs))()
        for i, (vk, pi, proof) in enumerate(zip(vks, public_inputs, proofs)):
            pia = _u64(pi, (-1, 4))
            keep.append(pia)
            bp[i] = B200BatchProof(index[id(vk)], _ptr(pia) if pia.size else None, pia.shape[0], C.addressof(proof))
        bl = (B200BatchLink * len(links))()
        for i, (comm_a, comm_b, lp, layout) in enumerate(links):
            ca, cb = _u64(comm_a, (8,)), _u64(comm_b, (8,))
            keep.append((ca, cb))
            bl[i] = B200BatchLink(_ptr(ca), _ptr(cb), layout.alignment, layout.offset, layout.size, C.addressof(lp))
        vt = (B200BatchVk * len(table))(*table)
        n = len(proofs) + len(links)
        flags = np.zeros(n, dtype=np.uint8)
        ops = np.zeros((n, 2, 8), dtype=np.uint64) if want_operands else None
        ok = C.c_int(0)
        _lib.check(ctx._lib.b200_plonk_batch_verify(ctx._h, vt, len(table), bp, len(proofs), bl if links else None, len(links),
                                                    _ptr(g2_h), _ptr(g2_tau_h), C.byref(ok),
                                                    flags.ctypes.data_as(C.c_void_p),
                                                    _ptr(ops) if want_operands else None, None))
        verdicts = flags.astype(bool)
        return (verdicts, ops) if want_operands else verdicts

    @staticmethod
    def preprocess(ctx: Context, srs: Bases, log_n: int, num_inputs: int, selectors: np.ndarray,
                   perm: np.ndarray, k: np.ndarray) -> ProvingKey:
        sel = np.ascontiguousarray(selectors, dtype=np.uint64).reshape(13, 1 << log_n, 4)
        pm = np.ascontiguousarray(perm, dtype=np.uint64).reshape(5 << log_n)
        kk = np.ascontiguousarray(k, dtype=np.uint64).reshape(5, 4)
        h = C.c_void_p()
        _lib.check(ctx._lib.b200_plonk_preprocess(ctx._h, srs._h, log_n, num_inputs, _ptr(sel), _ptr(pm), _ptr(kk),
                                                  C.byref(h)))
        return ProvingKey(ctx, h, log_n, num_inputs, kk)

    @staticmethod
    def prove_with_link_hint(ctx: Context, pk: ProvingKey, wires: np.ndarray, pub_inputs: np.ndarray,
                             blinders: np.ndarray, want_challenges: bool = False):
        """Returns (proof, LinkingHint[, challenges]).  `blinders` are the 17 field elements the
        reference draws from `thread_rng()` (traits.rs:994), in draw order."""
        n = pk.domain_size
        w = np.ascontiguousarray(wires, dtype=np.uint64).reshape(5, n, 4)
        pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64).reshape(-1, 4)
        if pi.shape[0] != pk.num_inputs:
            raise ValueError("wrong number of public inputs")
        bl = np.ascontiguousarray(blinders, dtype=np.uint64).reshape(17, 4)
        proof = B200Proof()
        link = np.zeros((n + 2, 4), dtype=np.uint64)
        ch = np.zeros((6, 4), dtype=np.uint64)
        _lib.check(ctx._lib.b200_plonk_prove(ctx._h, pk._h, _ptr(w), _ptr(pi) if pi.size else None, _ptr(bl),
                                             C.byref(proof), _ptr(link), _ptr(ch) if want_challenges else None))
        hint = LinkingHint(linking_wire_poly=link, linking_wire_comm=np.array(proof.wires_poly_comms[0], dtype=np.uint64))
        return (proof, hint, ch) if want_challenges else (proof, hint)


def keccak256(data: bytes) -> bytes:
    out = (C.c_uint8 * 32)()
    _lib.load().b200_keccak256(data, len(data), out)
    return bytes(out)


def plonk_last_timings(ctx: Context) -> dict:
    arr = (C.c_float * 8)()
    _lib.check(ctx._lib.b200_plonk_last_timings(ctx._h, C.byref(arr)))
    names = ("round1", "round2", "round3_quotient", "round3_commit", "round4", "round5")
    return {k: arr[i] for i, k in enumerate(names)}


def prove_raw(ctx: Context, pk: ProvingKey, wires_ptr: int, pub_inputs: np.ndarray, blinders: np.ndarray) -> B200Proof:
    """prove with the wire table given by address (pinned host or device memory)."""
    proof = B200Proof()
    pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64)
    bl = np.ascontiguousarray(blinders, dtype=np.uint64)
    _lib.check(ctx._lib.b200_plonk_prove(ctx._h, pk._h, C.c_void_p(wires_ptr), _ptr(pi) if pi.size else None, _ptr(bl),
                                         C.byref(proof), None, None))
    return proof


class B200LinkProof(C.Structure):
    """b200_link_proof: mpc-plonk `LinkingProof { quotient_commitment, opening_proof }`."""
    _fields_ = [("quotient_commitment", C.c_uint64 * 8), ("opening_proof", C.c_uint64 * 8)]

    def to_array(self) -> np.ndarray:
        return np.frombuffer(bytes(self), dtype=np.uint64).copy()


class B200BatchVk(C.Structure):
    """b200_batch_vk: one verifying key of a batch (the flat key of b200_plonk_verify)."""
    _fields_ = [("log_n", C.c_uint), ("num_inputs", C.c_size_t), ("k", C.c_void_p), ("selector_comms", C.c_void_p),
                ("sigma_comms", C.c_void_p)]


class B200BatchProof(C.Structure):
    """b200_batch_proof: one PlonK proof of a batch against key `vk` of the batch's key table."""
    _fields_ = [("vk", C.c_uint), ("pub_inputs", C.c_void_p), ("num_inputs", C.c_size_t), ("proof", C.c_void_p)]


class B200BatchLink(C.Structure):
    """b200_batch_link: one link proof of a batch (the arguments of b200_plonk_verify_link)."""
    _fields_ = [("comm1", C.c_void_p), ("comm2", C.c_void_p), ("alignment", C.c_uint), ("offset", C.c_size_t),
                ("size", C.c_size_t), ("proof", C.c_void_p)]


@dataclass
class GroupLayout:
    """mpc-relation `GroupLayout`: the link group occupies the roots g^(offset + i), i < size,
    of the 2^alignment-th roots of unity."""
    alignment: int
    offset: int
    size: int


def link_proofs(ctx: Context, srs: Bases, hint_a: LinkingHint, hint_b: LinkingHint, layout: GroupLayout):
    """`PlonkKzgSnark::link_proofs::<SolidityTranscript>` (proof_linking/intent_only.rs:42-47).
    Returns (B200LinkProof, eta)."""
    a1 = np.ascontiguousarray(hint_a.linking_wire_poly, dtype=np.uint64).reshape(-1, 4)
    a2 = np.ascontiguousarray(hint_b.linking_wire_poly, dtype=np.uint64).reshape(-1, 4)
    c1 = np.ascontiguousarray(hint_a.linking_wire_comm, dtype=np.uint64)
    c2 = np.ascontiguousarray(hint_b.linking_wire_comm, dtype=np.uint64)
    proof = B200LinkProof()
    eta = np.zeros(4, dtype=np.uint64)
    _lib.check(ctx._lib.b200_plonk_link(ctx._h, srs._h, _ptr(a1), a1.shape[0], _ptr(a2), a2.shape[0], _ptr(c1), _ptr(c2),
                                        layout.alignment, layout.offset, layout.size, C.byref(proof), _ptr(eta)))
    return proof, eta


def compute_poseidon_hash_batch(ctx: Context, values: np.ndarray) -> np.ndarray:
    """`batch` x `crypto::hash::compute_poseidon_hash(&values[i])` (crates/crypto/src/hash/mod.rs:12-18):
    values has shape (batch, len, 4) Montgomery; returns (batch, 4)."""
    v = np.ascontiguousarray(values, dtype=np.uint64)
    batch, ln = v.shape[0], v.shape[1]
    out = np.zeros((batch, 4), dtype=np.uint64)
    _lib.check(ctx._lib.b200_poseidon2_hash_batch(ctx._h, _ptr(v) if v.size else None, batch, ln, _ptr(out)))
    return out


def merkle_root_batch(ctx: Context, leaf_hashes: np.ndarray, sisters: np.ndarray, is_right: np.ndarray) -> np.ndarray:
    """Roots of a batch of Merkle openings (`b200_poseidon2_merkle_root_batch`): leaf_hashes (batch, 4), sisters
    (batch, height, 4) Montgomery limbs, is_right (batch, height) booleans -> (batch, 4)."""
    leaf = np.ascontiguousarray(leaf_hashes, dtype=np.uint64).reshape(-1, 4)
    batch = leaf.shape[0]
    sis = np.ascontiguousarray(sisters, dtype=np.uint64).reshape(batch, -1, 4)
    height = sis.shape[1]
    bits = np.ascontiguousarray(is_right, dtype=np.uint8).reshape(batch, height)
    out = np.zeros((batch, 4), dtype=np.uint64)
    _lib.check(ctx._lib.b200_poseidon2_merkle_root_batch(ctx._h, _ptr(leaf), _ptr(sis) if sis.size else None,
                                                         bits.ctypes.data_as(C.c_void_p) if bits.size else None, batch, height,
                                                         _ptr(out)))
    return out


def csprng_batch(ctx: Context, seeds: np.ndarray, first_index, count: int) -> np.ndarray:
    """`count` consecutive values of each Poseidon CSPRNG stream (`b200_poseidon2_csprng_batch`): seeds (batch, 4)
    Montgomery limbs, first_index (batch,) integers -> (batch, count, 4)."""
    sd = np.ascontiguousarray(seeds, dtype=np.uint64).reshape(-1, 4)
    idx = np.ascontiguousarray(first_index, dtype=np.uint64).reshape(-1)
    out = np.zeros((sd.shape[0], count, 4), dtype=np.uint64)
    _lib.check(ctx._lib.b200_poseidon2_csprng_batch(ctx._h, _ptr(sd), _ptr(idx), sd.shape[0], count, _ptr(out)))
    return out


def poseidon2_permute_batch(ctx: Context, states: np.ndarray) -> np.ndarray:
    """`Poseidon2Sponge::permute` (poseidon2.rs:90-110) on (batch, 3, 4) states; returns the permuted copy."""
    s = np.array(states, dtype=np.uint64, copy=True, order="C")
    _lib.check(ctx._lib.b200_poseidon2_permute_batch(ctx._h, _ptr(s), s.shape[0]))
    return s


# ---- names the reference gives these objects (circuit-types/src/lib.rs:72-101; SURVEY.md §8 row a11) ------------
PlonkProof = B200Proof                 # `pub type PlonkProof = Proof<SystemCurve>`
PlonkLinkProof = B200LinkProof         # `pub type PlonkLinkProof = LinkingProof<SystemCurve>`
ProofLinkingHint = LinkingHint         # `pub type ProofLinkingHint = LinkingHint<SystemCurve>`
ProverError = _lib.B200Error           # circuit-types/src/errors.rs:33-58: a failing prove surfaces as an error value


class BundleProof(C.Structure):
    """b200_bundle_proof"""
    _fields_ = [("pk", C.c_void_p), ("wires", C.c_void_p), ("pub_inputs", C.c_void_p), ("num_inputs", C.c_size_t),
                ("blinders", C.c_void_p), ("proof", C.c_void_p), ("link_poly", C.c_void_p)]


class BundleLink(C.Structure):
    """b200_bundle_link"""
    _fields_ = [("a", C.c_uint), ("b", C.c_uint), ("alignment", C.c_uint), ("offset", C.c_size_t), ("size", C.c_size_t),
                ("proof", C.c_void_p)]


class ProverPool:
    """b200_pool: the device-side counterpart of the reference's `NativeProofManager` thread pool
    (crates/workers/proof-manager/src/implementations/native_proof_manager.rs:138-201, `spawn_fifo`
    per job).  `workers` proofs are in flight on one GPU; keys and SRS tables are shared.

    Buffers passed to `submit_*` are kept alive by the pool object until the ticket is waited for."""

    def __init__(self, device: int = 0, workers: int = 6):
        self._lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self._lib.b200_pool_create(device, workers, C.byref(h)))
        self._h = h
        self.device = device
        self._keep = {}  # ticket -> objects the job reads or writes
        self._borrowed = []

    @property
    def workers(self) -> int:
        return int(self._lib.b200_pool_workers(self._h))

    def context(self, worker: int = 0) -> Context:
        """Worker `worker`'s context (borrowed: the pool frees it), for set-up calls."""
        raw = self._lib.b200_pool_ctx(self._h, worker)
        if not raw:
            raise IndexError("worker index out of range")
        ctx = Context.__new__(Context)
        ctx._lib, ctx._h, ctx.device, ctx._borrowed = self._lib, C.c_void_p(raw), self.device, True
        ctx.close = lambda: None  # the pool owns it
        self._borrowed.append(ctx)
        return ctx

    def submit_prove(self, pk: "ProvingKey", wires_ptr: int, pub_inputs: np.ndarray, blinders: np.ndarray,
                     with_link_poly: bool = False, keep=None) -> int:
        """Queue one proof; returns the ticket.  `wires_ptr`: address of the 5 x n wire table (pinned host
        or device memory), which the caller keeps valid until `wait(ticket)` returns (pass the owning
        object as `keep` to let the pool hold a reference)."""
        proof = B200Proof()
        pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64)
        bl = np.ascontiguousarray(blinders, dtype=np.uint64)
        if pi.size != 4 * pk.num_inputs:
            raise ProverError(-1, f"submit_prove: {pi.size // 4} public inputs for a key with {pk.num_inputs}")
        if bl.size != 4 * 17:
            raise ProverError(-1, "submit_prove: blinders must be 17 Fr elements")
        link = np.zeros((pk.domain_size + 2, 4), dtype=np.uint64) if with_link_poly else None
        ticket = C.c_uint64()
        _lib.check(self._lib.b200_pool_submit_prove(self._h, pk._h, C.c_void_p(wires_ptr), _ptr(pi) if pi.size else None,
                                                    pi.size // 4, _ptr(bl), C.byref(proof),
                                                    _ptr(link) if link is not None else None, C.byref(ticket)))
        self._keep[ticket.value] = (proof, link, keep, pk)
        return ticket.value

    def submit_link(self, srs: "Bases", hint_a: "LinkingHint", hint_b: "LinkingHint", layout: "GroupLayout") -> int:
        a1 = np.ascontiguousarray(hint_a.linking_wire_poly, dtype=np.uint64).reshape(-1, 4)
        a2 = np.ascontiguousarray(hint_b.linking_wire_poly, dtype=np.uint64).reshape(-1, 4)
        c1 = np.ascontiguousarray(hint_a.linking_wire_comm, dtype=np.uint64)
        c2 = np.ascontiguousarray(hint_b.linking_wire_comm, dtype=np.uint64)
        proof = B200LinkProof()
        ticket = C.c_uint64()
        _lib.check(self._lib.b200_pool_submit_link(self._h, srs._h, _ptr(a1), a1.shape[0], _ptr(a2), a2.shape[0],
                                                   _ptr(c1), _ptr(c2), layout.alignment, layout.offset, layout.size,
                                                   C.byref(proof), C.byref(ticket)))
        self._keep[ticket.value] = (proof, None, (a1, a2, c1, c2), srs)
        return ticket.value

    def submit_bundle(self, srs: "Bases", proofs, links) -> int:
        """One ticket for a whole proof bundle (`b200_pool_submit_bundle`): `proofs` = [(pk, wires_ptr, pub_inputs,
        blinders)], `links` = [(a, b, GroupLayout)] — link proof between the hints of proofs a and b, forked inside the
        pool once every proof is in (native_proof_manager.rs:526-584, 726-782).  `wait(ticket)` returns
        ([B200Proof], [link polys], [B200LinkProof])."""
        n_p, n_l = len(proofs), len(links)
        arr_p = (BundleProof * n_p)()
        arr_l = (BundleLink * max(n_l, 1))()
        keep, out_proofs, out_polys, out_links = [], [], [], []
        for i, (pk, wires_ptr, pub_inputs, blinders) in enumerate(proofs):
            pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64)
            bl = np.ascontiguousarray(blinders, dtype=np.uint64)
            if pi.size != 4 * pk.num_inputs or bl.size != 4 * 17:
                raise ProverError(-1, "submit_bundle: public inputs / blinders do not match the key")
            proof = B200Proof()
            poly = np.zeros((pk.domain_size + 2, 4), dtype=np.uint64)
            arr_p[i].pk, arr_p[i].wires = pk._h, C.c_void_p(wires_ptr)
            arr_p[i].pub_inputs = pi.ctypes.data_as(C.c_void_p) if pi.size else None
            arr_p[i].num_inputs, arr_p[i].blinders = pi.size // 4, bl.ctypes.data_as(C.c_void_p)
            arr_p[i].proof, arr_p[i].link_poly = C.cast(C.pointer(proof), C.c_void_p), poly.ctypes.data_as(C.c_void_p)
            keep += [pi, bl, pk]
            out_proofs.append(proof)
            out_polys.append(poly)
        for i, (a, b, lay) in enumerate(links):
            lp = B200LinkProof()
            arr_l[i].a, arr_l[i].b, arr_l[i].alignment, arr_l[i].offset, arr_l[i].size = a, b, lay.alignment, lay.offset, lay.size
            arr_l[i].proof = C.cast(C.pointer(lp), C.c_void_p)
            out_links.append(lp)
        ticket = C.c_uint64()
        _lib.check(self._lib.b200_pool_submit_bundle(self._h, srs._h, arr_p, n_p, arr_l, n_l, C.byref(ticket)))
        self._keep[ticket.value] = ((out_proofs, out_polys, out_links), None, keep, srs)
        return ticket.value

    def wait(self, ticket: int):
        """Blocks until the job is done; returns its B200Proof (or (B200Proof, link_poly) when the job was
        submitted with `with_link_poly`, or the B200LinkProof of a link job); raises B200Error with the
        job's own status and message if it failed."""
        rc = self._lib.b200_pool_wait(self._h, ticket)
        proof, link, _, _ = self._keep.pop(ticket, (None, None, None, None))
        _lib.check(rc)
        return (proof, link) if link is not None else proof

    def wait_all(self) -> None:
        rc = self._lib.b200_pool_wait_all(self._h)
        self._keep.clear()
        _lib.check(rc)

    def stats(self) -> dict:
        out = (C.c_uint64 * 4)()
        _lib.check(self._lib.b200_pool_stats(self._h, C.byref(out)))
        return dict(zip(("submitted", "completed", "failed", "queued"), (int(v) for v in out)))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200_pool_destroy(self._h)
            self._h = None
            self._keep.clear()
            for ctx in self._borrowed:  # their handles died with the pool
                ctx._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ProverBox:
    """`b200_box`: every GPU of the box behind one object — one prover pool per device, the SRS tables and the proving
    keys replicated on each, jobs routed to the least-loaded device.  The single-process counterpart of running one
    `ProverPool` per rank under torchrun."""

    def __init__(self, devices, workers_per_device: int = 6):
        self._lib = _lib.load()
        arr = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        _lib.check(self._lib.b200_box_create(arr, len(devices), workers_per_device, C.byref(h)))
        self._h, self._keep, self.devices = h, {}, list(devices)

    def load_srs(self, points: np.ndarray, window_bits: int = 0, check_on_curve: bool = False):
        pts = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
        h = C.c_void_p()
        _lib.check(self._lib.b200_box_srs_load(self._h, _ptr(pts), pts.shape[0], window_bits, int(check_on_curve), C.byref(h)))
        return h

    def preprocess(self, srs, log_n: int, num_inputs: int, selectors: np.ndarray, perm: np.ndarray, k: np.ndarray):
        sel = np.ascontiguousarray(selectors, dtype=np.uint64).reshape(13, 1 << log_n, 4)
        pm = np.ascontiguousarray(perm, dtype=np.uint64).reshape(5 << log_n)
        kk = np.ascontiguousarray(k, dtype=np.uint64).reshape(5, 4)
        h = C.c_void_p()
        _lib.check(self._lib.b200_box_preprocess(self._h, srs, log_n, num_inputs, _ptr(sel), _ptr(pm), _ptr(kk), C.byref(h)))
        return h

    def verifying_key(self, pk):
        sel, sig = np.zeros((13, 8), dtype=np.uint64), np.zeros((5, 8), dtype=np.uint64)
        _lib.check(self._lib.b200_box_pk_verifying_key(pk, _ptr(sel), _ptr(sig)))
        return sel, sig

    def submit_prove(self, pk, wires_ptr: int, pub_inputs: np.ndarray, blinders: np.ndarray, log_n: int = 0, keep=None) -> int:
        proof = B200Proof()
        pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64)
        bl = np.ascontiguousarray(blinders, dtype=np.uint64)
        link = np.zeros(((1 << log_n) + 2, 4), dtype=np.uint64) if log_n else None
        ticket = C.c_uint64()
        _lib.check(self._lib.b200_box_submit_prove(self._h, pk, C.c_void_p(wires_ptr), _ptr(pi) if pi.size else None, pi.size // 4,
                                                   _ptr(bl), C.byref(proof), _ptr(link) if link is not None else None,
                                                   C.byref(ticket)))
        self._keep[ticket.value] = (proof, link, keep, pi, bl)
        return ticket.value

    def wait(self, ticket: int):
        rc = self._lib.b200_box_wait(self._h, ticket)
        proof, link, *_ = self._keep.pop(ticket, (None, None))
        _lib.check(rc)
        return (proof, link) if link is not None else proof

    def ticket_device(self, ticket: int) -> int:
        return self._lib.b200_box_ticket_device(self._h, ticket)

    def free_pk(self, pk):
        self._lib.b200_box_pk_free(self._h, pk)

    def free_srs(self, srs):
        self._lib.b200_box_srs_free(self._h, srs)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200_box_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
