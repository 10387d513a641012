"""Collaborative (multi-party) TurboPlonk prover over additive shares — the compute side of the reference's
`MultiProverCircuit::{prove, prove_with_link_hint}` -> `MultiproverPlonkKzgSnark::prove_with_link_hint(&circuit, &pk,
fabric)` (/root/reference/crates/circuits/circuit-types/src/traits.rs:1103-1154, circuits-core/src/lib.rs:145-177).

In the reference the witness of VALID MATCH MPC never exists in one place: each party holds a share of every wire value
and the proof is produced jointly; only the proof is opened.  The upstream prover (mpc-jellyfish `multiprover/`, on the
ark-mpc fabric) is not vendored; what is restated here is the standard construction it follows:

  * the witness table, the 17 blinding scalars and every polynomial derived from them are ADDITIVE shares over Fr;
  * everything linear in the witness is computed share-wise with the single-prover primitives — inverse / coset NTTs,
    KZG commitments (MSM is linear: the opened commitment is the sum of the parties' commitments), polynomial
    evaluation and division by X - z;
  * the non-linear steps — the 5-factor numerators / denominators and the running product of round 2, the gate and
    permutation products of the quotient in round 3 — are Beaver multiplications: with a preprocessed triple
    ([a], [b], [ab]) the parties open d = x - a and e = y - b and set [xy] = [ab] + d[b] + e[a] + de;  inverses use
    a shared random mask ([r]: open B r, invert in public, scale [r]);
  * what is opened: the 13 commitments, the 10 evaluations, the masked values of the multiplications — never a wire value.

Because every step is the single prover's arithmetic on shares, the opened proof is BIT-IDENTICAL to the single-prover
proof of the summed witness with the summed blinders; the tests check exactly that (CPU: against the oracle prover, with
a host backend; GPU: against `b200_plonk_prove`).

Scope.  This module is the arithmetic of the protocol, party by party, with the transport collapsed to in-process sums
(`Fabric.open`): the network layer (ark-mpc's fabric, authenticated SPDZ shares with MACs, the offline triple
generation) stays where the north star leaves it — untouched, outside the proving path.  `Dealer` stands for the
preprocessing phase (a seeded PRG instead of an offline protocol).  Shares here are semi-honest additive shares; the MAC
half of an authenticated share is a second additive share and would ride through the same linear operations.

The arithmetic goes through a backend: `DeviceBackend` (the product: `libb200prover` on a B200 through the C ABI —
`b200_fr_vec_op`, `b200_ntt_device`, `b200_msm_device`, `b200_fr_batch_inverse_device`, `b200_fr_poly_eval_device`,
`b200_fr_poly_div_linear_device`) or any object with the same methods (the CPU tests inject one built on the oracle).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .backend import B200Proof, Bases, Context, LinkingHint, keccak256
from .fields import BASE_FIELD_MODULUS, SCALAR_FIELD_MODULUS as R, limbs_to_scalars, scalars_to_limbs

NW, NS = 5, 13


# ---------------------------------------------------------------------------------------------------------------
# Fiat–Shamir transcript (the library's SolidityTranscript, csrc/transcript.h, on the host side of the protocol)
# ---------------------------------------------------------------------------------------------------------------
class SolidityTranscript:
    def __init__(self):
        self.state, self.buf = bytes(64), bytearray()

    def append_fr(self, v: int):
        self.buf += int(v % R).to_bytes(32, "big")

    def append_g1(self, xy: np.ndarray):
        x, y = limbs_to_scalars(np.asarray(xy, dtype=np.uint64).reshape(2, 4), BASE_FIELD_MODULUS)
        self.buf += x.to_bytes(32, "big") + y.to_bytes(32, "big")

    def challenge(self) -> int:
        msg = self.state + bytes(self.buf)
        h0, h1 = keccak256(msg + b"\x00"), keccak256(msg + b"\x01")
        self.state = h0 + h1
        return int.from_bytes(self.state[:48], "big") % R


# ---------------------------------------------------------------------------------------------------------------
# backends
# ---------------------------------------------------------------------------------------------------------------
class DeviceBackend:
    """Fr vectors are int64 CUDA tensors of shape (len, 4) (Montgomery limbs); arithmetic through the C ABI."""

    def __init__(self, ctx: Context, srs: Bases):
        import torch
        self.torch, self.ctx, self.srs, self.lib = torch, ctx, srs, ctx._lib
        self.dev = torch.device("cuda", getattr(ctx, "device", 0) or 0)

    def _sync(self):
        """torch builds / moves the vectors on ITS stream (zeros, cat, roll, clone, H2D); the library runs on its own
        non-blocking stream: everything torch has queued must be complete before a pointer is handed over.  The library's
        calls synchronise their stream before returning, so the other direction needs nothing."""
        self.torch.cuda.current_stream(self.dev).synchronize()

    # construction / conversion
    def from_limbs(self, arr: np.ndarray):
        a = np.ascontiguousarray(arr, dtype=np.uint64).reshape(-1, 4)
        return self.torch.from_numpy(a.view(np.int64).copy()).to(self.dev)

    def to_limbs(self, v) -> np.ndarray:
        return v.cpu().numpy().view(np.uint64).reshape(-1, 4)

    def zeros(self, n: int):
        return self.torch.zeros((n, 4), dtype=self.torch.int64, device=self.dev)

    def concat(self, parts):
        return self.torch.cat(list(parts), dim=0)

    def clone(self, v):
        return v.clone()

    def roll(self, v, shift: int):
        return self.torch.roll(v, shifts=-shift, dims=0)  # out[i] = v[i + shift]

    def random(self, seed: int, n: int):
        out = self.zeros(n)
        self._sync()
        self.ctx.splitmix_fr_device(seed, n, out.data_ptr(), montgomery=True)
        return out

    # arithmetic
    def _op(self, op: int, a, b):
        scalar = b.shape[0] == 1 and a.shape[0] != 1
        out = self.torch.empty_like(a)
        self._sync()
        _lib.check(self.lib.b200_fr_vec_op(self.ctx._h, op, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), int(scalar),
                                           a.shape[0], C.c_void_p(out.data_ptr())))
        return out

    def add(self, a, b):
        return self._op(0, a, b)

    def sub(self, a, b):
        return self._op(1, a, b)

    def mul(self, a, b):
        return self._op(2, a, b)

    def scalar(self, v: int):
        return self.from_limbs(scalars_to_limbs([v]))

    def batch_inverse(self, a):
        out = a.clone()
        self._sync()
        _lib.check(self.lib.b200_fr_batch_inverse_device(self.ctx._h, C.c_void_p(out.data_ptr()), out.shape[0]))
        return out

    def ntt(self, a, inverse: bool, coset: bool):
        out = a.clone()
        log_n = out.shape[0].bit_length() - 1
        self._sync()
        self.ctx.ntt_device(out.data_ptr(), log_n, inverse=inverse, coset=coset)
        return out

    def commit(self, coeffs):
        self._sync()
        xy, inf = self.ctx.msm_device(self.srs, coeffs.data_ptr(), coeffs.shape[0], montgomery=True)
        return xy, inf

    def poly_eval(self, coeffs, z: int) -> int:
        zz = scalars_to_limbs([z])
        out = np.zeros(4, dtype=np.uint64)
        self._sync()
        _lib.check(self.lib.b200_fr_poly_eval_device(self.ctx._h, C.c_void_p(coeffs.data_ptr()), coeffs.shape[0],
                                                     zz.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        return limbs_to_scalars(out.reshape(1, 4))[0]

    def div_linear(self, coeffs, z: int):
        zz = scalars_to_limbs([z])
        out = self.zeros(coeffs.shape[0] - 1)
        self._sync()
        _lib.check(self.lib.b200_fr_poly_div_linear_device(self.ctx._h, C.c_void_p(coeffs.data_ptr()), coeffs.shape[0],
                                                           zz.ctypes.data_as(C.c_void_p), C.c_void_p(out.data_ptr())))
        return out

    def g1_sum(self, points: Sequence) -> np.ndarray:
        xy, _ = self.ctx.g1_sum_affine(np.stack([p[0] for p in points]), [p[1] for p in points])
        return xy


# ---------------------------------------------------------------------------------------------------------------
# the protocol
# ---------------------------------------------------------------------------------------------------------------
Shared = List  # one backend vector per party


@dataclass
class Fabric:
    """In-process stand-in for the MPC fabric: `open` is "every party broadcasts its share, everyone adds"."""
    be: object
    parties: int
    opened_elements: int = 0
    multiplications: int = 0

    def open(self, x: Shared):
        acc = x[0]
        for s in x[1:]:
            acc = self.be.add(acc, s)
        self.opened_elements += x[0].shape[0]
        return acc

    def open_scalar(self, vals: Sequence[int]) -> int:
        self.opened_elements += 1
        return sum(vals) % R


@dataclass
class Dealer:
    """Preprocessing phase (SPDZ offline): Beaver triples and inversion masks, here from a seeded PRG."""
    be: object
    parties: int
    seed: int = 0xBEA7E5
    counter: int = 0

    def _rand(self, n: int):
        self.counter += 1
        return self.be.random(self.seed + 0x9E37 * self.counter, n)

    def _share(self, value) -> Shared:
        shares = [self._rand(value.shape[0]) for _ in range(self.parties - 1)]
        last = value
        for s in shares:
            last = self.be.sub(last, s)
        return shares + [last]

    def triple(self, n: int):
        a, b = self._rand(n), self._rand(n)
        return self._share(a), self._share(b), self._share(self.be.mul(a, b))

    def mask(self, n: int) -> Shared:
        return self._share(self._rand(n))  # non-zero with overwhelming probability


def sh_add_public(be, x: Shared, pub) -> Shared:
    """[x] + public: party 0 adds it."""
    return [be.add(x[0], pub)] + list(x[1:])


def sh_mul_public(be, x: Shared, pub) -> Shared:
    return [be.mul(s, pub) for s in x]


def sh_add(be, x: Shared, y: Shared) -> Shared:
    return [be.add(a, b) for a, b in zip(x, y)]


def sh_sub(be, x: Shared, y: Shared) -> Shared:
    return [be.sub(a, b) for a, b in zip(x, y)]


def beaver_mul(fab: Fabric, dealer: Dealer, x: Shared, y: Shared) -> Shared:
    """[x][y] element-wise with one preprocessed triple per element: two openings, then local operations."""
    be = fab.be
    a, b, c = dealer.triple(x[0].shape[0])
    d = fab.open(sh_sub(be, x, a))
    e = fab.open(sh_sub(be, y, b))
    out = [be.add(be.add(c[p], be.mul(b[p], d)), be.mul(a[p], e)) for p in range(fab.parties)]
    out[0] = be.add(out[0], be.mul(d, e))
    fab.multiplications += x[0].shape[0]
    return out


def beaver_mul_many(fab: Fabric, dealer: Dealer, pairs: Sequence) -> List[Shared]:
    """One round for several independent products of equal length (concatenated: one pair of openings)."""
    be = fab.be
    n = pairs[0][0][0].shape[0]
    X = [be.concat([pr[0][p] for pr in pairs]) for p in range(fab.parties)]
    Y = [be.concat([pr[1][p] for pr in pairs]) for p in range(fab.parties)]
    Z = beaver_mul(fab, dealer, X, Y)
    return [[Z[p][i * n:(i + 1) * n] for p in range(fab.parties)] for i in range(len(pairs))]


@dataclass
class CollaborativeProvingKey:
    """The public part every party holds: circuit polynomials and the verifying-key commitments."""
    log_n: int
    num_inputs: int
    k: List[int]
    selector_coeffs: list      # 13 backend vectors (n)
    sigma_coeffs: list         # 5
    sigma_evals: list          # 5 (over H)
    selector_comms: np.ndarray  # (13, 8)
    sigma_comms: np.ndarray     # (5, 8)

    @staticmethod
    def build(be, log_n: int, num_inputs: int, selectors: np.ndarray, perm: np.ndarray, k: np.ndarray) -> "CollaborativeProvingKey":
        n = 1 << log_n
        kk = limbs_to_scalars(np.asarray(k, dtype=np.uint64).reshape(5, 4))
        sel = np.ascontiguousarray(selectors, dtype=np.uint64).reshape(NS, n, 4)
        w = domain_generator(log_n)
        dom = [1] * n
        for j in range(1, n):
            dom[j] = dom[j - 1] * w % R
        pm = np.asarray(perm, dtype=np.uint64).reshape(NW * n)
        sig_ev = [be.from_limbs(scalars_to_limbs([kk[int(t) // n] * dom[int(t) % n] % R for t in pm[i * n:(i + 1) * n]]))
                  for i in range(NW)]
        sel_c = [be.ntt(be.from_limbs(sel[s]), True, False) for s in range(NS)]
        sig_c = [be.ntt(v, True, False) for v in sig_ev]
        comm = lambda v: (lambda xy, inf: np.zeros(8, dtype=np.uint64) if inf else xy)(*be.commit(v))
        return CollaborativeProvingKey(log_n, num_inputs, kk, sel_c, sig_c, sig_ev,
                                       np.stack([comm(v) for v in sel_c]), np.stack([comm(v) for v in sig_c]))


def domain_generator(log_n: int) -> int:
    """Radix2EvaluationDomain::group_gen: TWO_ADIC_ROOT_OF_UNITY^(2^(28 - log_n)) (SURVEY.md §8(a5))."""
    root = 19103219067921713944291392827692070036145651957329286315305642004821462161904
    return pow(root, 1 << (28 - log_n), R)


def share_table(values: np.ndarray, parties: int, seed: int) -> List[np.ndarray]:
    """Split a (rows, 4)-limb Montgomery table into `parties` additive shares (test / example helper: in the reference
    the parties arrive with their shares)."""
    import random
    rnd = random.Random(seed)
    ints = limbs_to_scalars(np.asarray(values, dtype=np.uint64).reshape(-1, 4))
    shares = [[rnd.randrange(R) for _ in ints] for _ in range(parties - 1)]
    last = [(v - sum(col)) % R for v, col in zip(ints, zip(*shares))] if parties > 1 else list(ints)
    return [scalars_to_limbs(s) for s in shares] + [scalars_to_limbs(last)]


class MultiproverPlonkKzgSnark:
    """`MultiproverPlonkKzgSnark::prove_with_link_hint` on additive shares (see the module docstring)."""

    @staticmethod
    def prove_with_link_hint(be, pk: CollaborativeProvingKey, wire_shares: Sequence[np.ndarray], pub_inputs: np.ndarray,
                             blinder_shares: Sequence[np.ndarray], dealer_seed: int = 0xBEA7E5):
        """wire_shares[p]: party p's share of the 5 x n wire table (Montgomery limbs); blinder_shares[p]: its share of
        the 17 blinders.  Returns (opened B200Proof, opened LinkingHint, Fabric with the communication counters)."""
        P = len(wire_shares)
        n, log_n = 1 << pk.log_n, pk.log_n
        m, log_m = 8 * n, pk.log_n + 3
        fab, dealer = Fabric(be, P), Dealer(be, P, dealer_seed)
        pi_ints = limbs_to_scalars(np.asarray(pub_inputs, dtype=np.uint64).reshape(-1, 4)) if pk.num_inputs else []
        bl = [limbs_to_scalars(np.asarray(b, dtype=np.uint64).reshape(17, 4)) for b in blinder_shares]
        W = [[be.from_limbs(np.asarray(ws, dtype=np.uint64).reshape(NW, n, 4)[i]) for i in range(NW)] for ws in wire_shares]
        w_gen = domain_generator(log_n)
        proof = B200Proof()

        def opened_commitment(per_party) -> np.ndarray:
            return be.g1_sum([be.commit(v) for v in per_party])  # MSM is linear: the parties' commitments add up

        def set_g1(dst, xy):
            dst[:] = [int(v) for v in xy]

        def set_fr(dst, v):
            dst[:] = [int(x) for x in scalars_to_limbs([v])[0]]

        tr = SolidityTranscript()
        tr.buf += (254).to_bytes(4, "big") + n.to_bytes(8, "big") + pk.num_inputs.to_bytes(8, "big")
        for v in pk.k:
            tr.append_fr(v)
        for c in list(pk.selector_comms) + list(pk.sigma_comms):
            tr.append_g1(c)
        for v in pi_ints:
            tr.append_fr(v)

        def blind(poly_p, p: int, idx: Sequence[int], length: int):
            """poly + (b0 + b1 X + ...) Z_H on party p's share: coefficient j loses b_j, coefficient n + j gains it.
            Only the 2 x len(idx) touched coefficients are built on the host."""
            k = len(idx)
            head = be.from_limbs(scalars_to_limbs([(R - bl[p][bi]) % R for bi in idx]))
            tail = be.from_limbs(scalars_to_limbs([bl[p][bi] for bi in idx] + [0] * (length - n - k)))
            delta = be.concat([head, be.zeros(n - k), tail])
            return be.add(be.concat([poly_p, be.zeros(length - n)]), delta)

        # ---- round 1: wire polynomials (linear) ------------------------------------------------------------------
        wire_polys = [[blind(be.ntt(W[p][i], True, False), p, (2 * i, 2 * i + 1), n + 2) for i in range(NW)] for p in range(P)]
        for i in range(NW):
            xy = opened_commitment([wire_polys[p][i] for p in range(P)])
            set_g1(proof.wires_poly_comms[i], xy)
            tr.append_g1(xy)
        pi_poly = be.ntt(be.from_limbs(scalars_to_limbs(list(pi_ints) + [0] * (n - len(pi_ints)))), True, False)
        link_poly = fab.open([wire_polys[p][0] for p in range(P)])  # opened here for the hint; an MPC keeps it shared

        # ---- round 2: permutation product ----------------------------------------------------------------------------
        beta, gamma = tr.challenge(), tr.challenge()
        dom = [1] * n
        for j in range(1, n):
            dom[j] = dom[j - 1] * w_gen % R
        dom_v = be.from_limbs(scalars_to_limbs(dom))
        s_beta, s_gamma = be.scalar(beta), be.scalar(gamma)
        nf, df = [], []
        for i in range(NW):
            pub_n = be.add(be.mul(dom_v, be.scalar(beta * pk.k[i] % R)), s_gamma)       # beta k_i w^j + gamma
            pub_d = be.add(be.mul(pk.sigma_evals[i], s_beta), s_gamma)                  # beta sigma_i(w^j) + gamma
            wi = [W[p][i] for p in range(P)]
            nf.append(sh_add_public(be, wi, pub_n))
            df.append(sh_add_public(be, wi, pub_d))
        n01, n23, d01, d23 = beaver_mul_many(fab, dealer, [(nf[0], nf[1]), (nf[2], nf[3]), (df[0], df[1]), (df[2], df[3])])
        n0123, d0123 = beaver_mul_many(fab, dealer, [(n01, n23), (d01, d23)])
        num, den = beaver_mul_many(fab, dealer, [(n0123, nf[4]), (d0123, df[4])])
        mask = dealer.mask(n)
        m_open = fab.open(beaver_mul(fab, dealer, den, mask))            # den * r, safe to open
        den_inv = sh_mul_public(be, mask, be.batch_inverse(m_open))     # [1/den] = (den r)^-1 [r]
        ratio = beaver_mul(fab, dealer, num, den_inv)
        # z(w^0) = 1, z(w^(j+1)) = z(w^j) * ratio_j: inclusive prefix products by doubling, each level one multiplication
        x = ratio
        d = 1
        while d < n:
            prod = beaver_mul(fab, dealer, [s[d:] for s in x], [s[:n - d] for s in x])
            x = [be.concat([x[p][:d], prod[p]]) for p in range(P)]
            d <<= 1
        one_v = be.from_limbs(scalars_to_limbs([1]))
        z_evals = [be.concat([one_v if p == 0 else be.zeros(1), x[p][:n - 1]]) for p in range(P)]
        z_polys = [blind(be.ntt(z_evals[p], True, False), p, (10, 11, 12), n + 3) for p in range(P)]
        xy = opened_commitment(z_polys)
        set_g1(proof.prod_perm_poly_comm, xy)
        tr.append_g1(xy)

        # ---- round 3: quotient on the coset g H_8n -------------------------------------------------------------------------
        alpha = tr.challenge()
        pad = lambda v: be.concat([v, be.zeros(m - v.shape[0])])
        cfft = lambda v: be.ntt(pad(v), False, True)
        ce_sel = [cfft(v) for v in pk.selector_coeffs]
        ce_sig = [cfft(v) for v in pk.sigma_coeffs]
        ce_pi = cfft(pi_poly)
        ce_w = [[cfft(wire_polys[p][i]) for p in range(P)] for i in range(NW)]  # [wire][party]
        ce_z = [cfft(z_polys[p]) for p in range(P)]
        ce_zw = [be.roll(v, 8) for v in ce_z]                                     # z(w x): 8 steps of the 8n-th root
        wm = domain_generator(log_m)
        pts = [5] * m
        for i in range(1, m):
            pts[i] = pts[i - 1] * wm % R
        pts_v = be.from_limbs(scalars_to_limbs(pts))
        zh_inv8 = [pow((pow(5 * pow(wm, i, R) % R, n, R) - 1) % R, -1, R) for i in range(8)]
        zh_inv_v = be.from_limbs(scalars_to_limbs([zh_inv8[i % 8] for i in range(m)]))
        l1_inv_v = be.batch_inverse(be.mul(be.sub(pts_v, be.scalar(1)), be.scalar(n)))   # 1 / (n (x - 1))
        nfq, dfq = [], []
        for j in range(NW):
            pub_n = be.add(be.mul(pts_v, be.scalar(beta * pk.k[j] % R)), s_gamma)
            pub_d = be.add(be.mul(ce_sig[j], s_beta), s_gamma)
            nfq.append(sh_add_public(be, ce_w[j], pub_n))
            dfq.append(sh_add_public(be, ce_w[j], pub_d))
        # multiplication depth 1 .. 4, independent products of a depth in one round
        r1 = beaver_mul_many(fab, dealer, [(ce_w[0], ce_w[1]), (ce_w[2], ce_w[3])] + [(ce_w[j], ce_w[j]) for j in range(4)] +
                             [(nfq[0], nfq[1]), (nfq[2], nfq[3]), (dfq[0], dfq[1]), (dfq[2], dfq[3])])
        w01, w23, sq, (qn01, qn23, qd01, qd23) = r1[0], r1[1], r1[2:6], r1[6:10]
        r2 = beaver_mul_many(fab, dealer, [(w01, w23)] + [(sq[j], sq[j]) for j in range(4)] + [(qn01, qn23), (qd01, qd23)])
        w0123, p4, (qn0123, qd0123) = r2[0], r2[1:5], r2[5:7]
        r3 = beaver_mul_many(fab, dealer, [(w0123, ce_w[4])] + [(p4[j], ce_w[j]) for j in range(4)] +
                             [(qn0123, nfq[4]), (qd0123, dfq[4])])
        w01234, p5, (qnum, qden) = r3[0], r3[1:5], r3[5:7]
        zn, zd = beaver_mul_many(fab, dealer, [(ce_z, qnum), (ce_zw, qden)])
        # gate: q_c + pi + sum q_lc w + q_mul0 w0w1 + q_mul1 w2w3 + q_ecc w0..w4 + sum q_hash w^5 - q_o w4
        t_circ = [be.zeros(m) for _ in range(P)]
        for j in range(4):
            t_circ = sh_add(be, t_circ, sh_mul_public(be, ce_w[j], ce_sel[j]))
            t_circ = sh_add(be, t_circ, sh_mul_public(be, p5[j], ce_sel[6 + j]))
        t_circ = sh_add(be, t_circ, sh_mul_public(be, w01, ce_sel[4]))
        t_circ = sh_add(be, t_circ, sh_mul_public(be, w23, ce_sel[5]))
        t_circ = sh_add(be, t_circ, sh_mul_public(be, w01234, ce_sel[12]))
        t_circ = sh_sub(be, t_circ, sh_mul_public(be, ce_w[4], ce_sel[10]))
        t_circ = sh_add_public(be, t_circ, be.add(ce_sel[11], ce_pi))
        perm = sh_mul_public(be, sh_sub(be, zn, zd), be.scalar(alpha))
        zm1 = sh_add_public(be, ce_z, be.scalar(R - 1))
        r2term = sh_mul_public(be, sh_mul_public(be, zm1, be.scalar(alpha * alpha % R)), l1_inv_v)
        quot = sh_add(be, sh_mul_public(be, sh_add(be, t_circ, perm), zh_inv_v), r2term)
        quot_c = [be.ntt(q, True, True) for q in quot]                    # coset iFFT, share-wise
        deg = NW * (n + 1) + 2
        tail = limbs_to_scalars(be.to_limbs(fab.open([q[deg:] for q in quot_c])))  # zero for a satisfied circuit: opening leaks nothing
        if tail[0] == 0 or any(tail[1:]):
            raise _lib.B200Error(-7, "WrongQuotientPolyDegree: the shared witness does not satisfy the circuit")
        total = NW * (n + 1) + 3
        split = [[None] * NW for _ in range(P)]
        for p in range(P):
            last = 0
            for i in range(NW):
                beg = i * (n + 2)
                end = beg + n + 2 if i < NW - 1 else total
                part = quot_c[p][beg:end]                                  # stays on the backend
                if last:
                    part = be.sub(part, be.concat([be.scalar(last), be.zeros(end - beg - 1)]))
                if i < NW - 1:
                    last = bl[p][13 + i]
                    part = be.concat([part, be.scalar(last)])
                split[p][i] = part
        for i in range(NW):
            xy = opened_commitment([split[p][i] for p in range(P)])
            set_g1(proof.split_quot_poly_comms[i], xy)
            tr.append_g1(xy)

        # ---- round 4: evaluations (linear: each party evaluates its share, the values are opened) ---------------------------------
        zeta = tr.challenge()
        zeta_w = zeta * w_gen % R
        we = [fab.open_scalar([be.poly_eval(wire_polys[p][i], zeta) for p in range(P)]) for i in range(NW)]
        se = [be.poly_eval(pk.sigma_coeffs[i], zeta) for i in range(NW - 1)]    # public polynomials
        zw_eval = fab.open_scalar([be.poly_eval(z_polys[p], zeta_w) for p in range(P)])
        for i in range(NW):
            set_fr(proof.wires_evals[i], we[i])
            tr.append_fr(we[i])
        for i in range(NW - 1):
            set_fr(proof.wire_sigma_evals[i], se[i])
            tr.append_fr(se[i])
        set_fr(proof.perm_next_eval, zw_eval)
        tr.append_fr(zw_eval)

        # ---- round 5: linearisation + batched opening (linear) ------------------------------------------------------------------------
        v = tr.challenge()
        vanish = (pow(zeta, n, R) - 1) % R
        l1 = vanish * pow(n * (zeta - 1) % R, -1, R) % R
        coeff_z = alpha
        for j in range(NW):
            coeff_z = coeff_z * ((pk.k[j] * zeta % R * beta + we[j] + gamma) % R) % R
        coeff_z = (coeff_z + alpha * alpha % R * l1) % R
        coeff_s = alpha * beta % R * zw_eval % R
        for j in range(NW - 1):
            coeff_s = coeff_s * ((se[j] * beta + we[j] + gamma) % R) % R
        LL = n + 3
        padto = lambda vec, ln: be.concat([vec, be.zeros(ln - vec.shape[0])]) if vec.shape[0] < ln else vec
        pow5 = lambda a: pow(a, 5, R)
        pub = be.zeros(LL)                                           # the public part of the linearisation: party 0's
        sel_scal = [we[0], we[1], we[2], we[3], we[0] * we[1] % R, we[2] * we[3] % R, pow5(we[0]), pow5(we[1]), pow5(we[2]),
                    pow5(we[3]), (R - we[4]) % R, 1, we[0] * we[1] % R * we[2] % R * we[3] % R * we[4] % R]
        for s_idx, sc in enumerate(sel_scal):
            pub = be.add(pub, padto(be.mul(pk.selector_coeffs[s_idx], be.scalar(sc)), LL))
        pub = be.add(pub, padto(be.mul(pk.sigma_coeffs[NW - 1], be.scalar((R - coeff_s) % R)), LL))
        zn2 = (vanish + 1) * zeta % R * zeta % R
        vp = [pow(v, i + 1, R) for i in range(2 * NW - 1)]
        for i in range(NW - 1):                                       # + v^(6+i) sigma_i
            pub = be.add(pub, padto(be.mul(pk.sigma_coeffs[i], be.scalar(vp[NW + i])), LL))
        batch = []
        for p in range(P):
            acc = be.mul(z_polys[p], be.scalar(coeff_z))             # z(X) term, n + 3 coefficients
            c = (R - vanish) % R
            for i in range(NW):
                acc = be.add(acc, padto(be.mul(split[p][i], be.scalar(c)), LL))
                c = c * zn2 % R
            for i in range(NW):
                acc = be.add(acc, padto(be.mul(wire_polys[p][i], be.scalar(vp[i])), LL))
            batch.append(be.add(acc, pub) if p == 0 else acc)
        xy = opened_commitment([be.div_linear(batch[p], zeta) for p in range(P)])
        set_g1(proof.opening_proof, xy)
        xy = opened_commitment([be.div_linear(z_polys[p], zeta_w) for p in range(P)])
        set_g1(proof.shifted_opening_proof, xy)
        hint = LinkingHint(linking_wire_poly=be.to_limbs(link_poly), linking_wire_comm=np.array(proof.wires_poly_comms[0], dtype=np.uint64))
        return proof, hint, fab


# ---------------------------------------------------------------------------------------------------------------
# the protocol on the device: one party per call (b200_mpc_prove / b200_mpc_link)
# ---------------------------------------------------------------------------------------------------------------
ALL_GATHER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)
ABORT = C.CFUNCTYPE(None, C.c_void_p)


class MpcTransport(C.Structure):
    """b200_mpc_transport: all_gather(user, mine, bytes, all) and abort(user) of one party."""
    _fields_ = [("all_gather", ALL_GATHER), ("abort", ABORT), ("user", C.c_void_p), ("party", C.c_int), ("parties", C.c_int)]


def callback_transport(party: int, parties: int, all_gather, abort=None) -> MpcTransport:
    """A transport written in Python: `all_gather(mine: bytes) -> bytes` returns every party's message in party order
    (or None / raises to fail the exchange); `abort()` is called when this party gives up."""
    def _gather(_user, mine, nbytes, out):
        try:
            got = all_gather(C.string_at(mine, nbytes))
        except Exception:
            return -1
        if got is None or len(got) != parties * nbytes:
            return -1
        C.memmove(out, got, len(got))
        return 0

    def _abort(_user):
        if abort is not None:
            abort()

    t = MpcTransport(ALL_GATHER(_gather), ABORT(_abort), None, party, parties)
    t._keep = (t.all_gather, t.abort)  # the C callbacks live as long as the structure
    return t


class LocalGroup:
    """b200_mpc_local_group: an in-process all-gather between the threads of `parties` parties."""

    def __init__(self, parties: int, timeout_ms: int = 120000):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        _lib.check(self._lib.b200_mpc_local_group_create(parties, timeout_ms, C.byref(self._h)))
        self.parties = parties

    def transport(self, party: int) -> MpcTransport:
        t = MpcTransport()
        _lib.check(self._lib.b200_mpc_local_group_transport(self._h, party, C.byref(t)))
        return t

    def close(self):
        if self._h:
            self._lib.b200_mpc_local_group_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MpcPrep:
    """b200_mpc_prep: one party's Beaver triples and masks for ONE proof (device-resident, single-use)."""

    def __init__(self, ctx: Context, handle):
        self._ctx, self._h = ctx, handle

    @staticmethod
    def size(pk) -> tuple:
        t, m = C.c_size_t(), C.c_size_t()
        _lib.check(_lib.load().b200_mpc_prep_size(pk._h, C.byref(t), C.byref(m)))
        return t.value, m.value

    @staticmethod
    def dealer(ctx: Context, pk, seed: int, party: int, parties: int) -> "MpcPrep":
        """INSECURE stand-in for an offline phase (tests, benchmarks): shares derived from (seed, party, parties)."""
        h = C.c_void_p()
        _lib.check(ctx._lib.b200_mpc_prep_dealer(ctx._h, pk._h, seed & (2**64 - 1), party, parties, C.byref(h)))
        return MpcPrep(ctx, h)

    @staticmethod
    def dealer_auth(ctx: Context, pk, seed: int, party: int, parties: int) -> tuple:
        """INSECURE, as `dealer`, with MACs: (MpcPrep for `prove_party_auth`, this party's MAC-key share as (4,) limbs)."""
        h = C.c_void_p()
        key = np.zeros(4, dtype=np.uint64)
        _lib.check(ctx._lib.b200_mpc_prep_dealer_auth(ctx._h, pk._h, seed & (2**64 - 1), party, parties,
                                                      key.ctypes.data_as(C.c_void_p), C.byref(h)))
        return MpcPrep(ctx, h), key

    def free(self):
        if self._h:
            self._ctx._lib.b200_mpc_prep_free(self._ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class MpcResult:
    proof: B200Proof
    link_poly_share: np.ndarray   # (n + 2, 4): this party's share of the linking polynomial
    challenges: np.ndarray        # (6, 4): beta, gamma, alpha, zeta, v, u
    stats: dict


def mpc_last_stats(ctx: Context) -> dict:
    arr = (C.c_double * 4)()
    _lib.check(ctx._lib.b200_mpc_last_stats(ctx._h, C.byref(arr)))
    return {"exchanges": int(arr[0]), "bytes_sent": int(arr[1]), "triples": int(arr[2]), "all_gather_ms": arr[3]}


def prove_party(ctx: Context, pk, transport: MpcTransport, prep: MpcPrep, wire_share: np.ndarray, pub_inputs: np.ndarray,
                blinder_share: np.ndarray) -> MpcResult:
    """`b200_mpc_prove` for one party over any transport (a caller's, or a LocalGroup's)."""
    n = pk.domain_size
    w = np.ascontiguousarray(wire_share, dtype=np.uint64).reshape(5 * n, 4)
    pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64).reshape(-1, 4)
    bl = np.ascontiguousarray(blinder_share, dtype=np.uint64).reshape(17, 4)
    proof = B200Proof()
    link = np.zeros((n + 2, 4), dtype=np.uint64)
    ch = np.zeros((6, 4), dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(ctx._lib.b200_mpc_prove(ctx._h, pk._h, C.byref(transport), prep._h, vp(w), vp(pi) if pi.size else None, vp(bl),
                                       C.byref(proof), vp(link), vp(ch)))
    return MpcResult(proof, link, ch, mpc_last_stats(ctx))


def _run_parties(fns):
    """Runs fns[p]() on one thread per party; returns each party's result or the exception it raised."""
    import threading
    out = [None] * len(fns)

    def run(p):
        try:
            out[p] = fns[p]()
        except Exception as e:  # noqa: BLE001 - handed back to the caller per party
            out[p] = e

    ts = [threading.Thread(target=run, args=(p,)) for p in range(len(fns))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return out


def prove_jointly(ctxs, pks, wire_shares, pub_inputs, blinder_shares, seed: int = 0xBEA7E5, timeout_ms: int = 120000,
                  transports=None):
    """All parties of one collaborative proof in this process: one thread per party over a LocalGroup (or over
    `transports`), dealer preprocessing from `seed`.  Returns every party's MpcResult, or the B200Error it failed with."""
    P = len(ctxs)
    group = LocalGroup(P, timeout_ms) if transports is None else None
    trs = transports if transports is not None else [group.transport(p) for p in range(P)]
    preps = [MpcPrep.dealer(ctxs[p], pks[p], seed, p, P) for p in range(P)]
    try:
        return _run_parties([lambda p=p: prove_party(ctxs[p], pks[p], trs[p], preps[p], wire_shares[p], pub_inputs,
                                                     blinder_shares[p]) for p in range(P)])
    finally:
        for pr in preps:
            pr.free()
        if group is not None:
            group.close()


def link_party(ctx: Context, srs: Bases, transport: MpcTransport, a1_share: np.ndarray, a2_share: np.ndarray,
               comm1: np.ndarray, comm2: np.ndarray, layout):
    """`b200_mpc_link` for one party: (B200LinkProof, eta)."""
    from .backend import B200LinkProof
    a1 = np.ascontiguousarray(a1_share, dtype=np.uint64).reshape(-1, 4)
    a2 = np.ascontiguousarray(a2_share, dtype=np.uint64).reshape(-1, 4)
    c1 = np.ascontiguousarray(comm1, dtype=np.uint64).reshape(8)
    c2 = np.ascontiguousarray(comm2, dtype=np.uint64).reshape(8)
    proof = B200LinkProof()
    eta = np.zeros(4, dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(ctx._lib.b200_mpc_link(ctx._h, srs._h, C.byref(transport), vp(a1), a1.shape[0], vp(a2), a2.shape[0], vp(c1),
                                      vp(c2), layout.alignment, layout.offset, layout.size, C.byref(proof), vp(eta)))
    return proof, eta


def link_jointly(ctxs, srss, a1_shares, a2_shares, comm1, comm2, layout, timeout_ms: int = 120000):
    """All parties of one collaborative link proof over a LocalGroup; per party (B200LinkProof, eta) or its B200Error."""
    P = len(ctxs)
    group = LocalGroup(P, timeout_ms)
    trs = [group.transport(p) for p in range(P)]
    try:
        return _run_parties([lambda p=p: link_party(ctxs[p], srss[p], trs[p], a1_shares[p], a2_shares[p], comm1, comm2, layout)
                             for p in range(P)])
    finally:
        group.close()


# ---------------------------------------------------------------------------------------------------------------
# authenticated shares (b200_mpc_prove_auth / b200_mpc_link_auth): every share x comes with its MAC share [alpha x]
# ---------------------------------------------------------------------------------------------------------------
def auth_share_table(values: np.ndarray, parties: int, mac_key_shares, seed: int = 0) -> tuple:
    """Authenticated additive shares of a (k, 4) table of Montgomery limbs under the MAC key alpha = sum(mac_key_shares)
    (each a (4,) limb array), in Python integers: (shares, macs), each a list of `parties` (k, 4) tables whose sums are
    the values and alpha times the values.  For small tables; `dealer_share_auth` does the same on the device."""
    import random
    rnd = random.Random(seed)
    alpha = sum(limbs_to_scalars(np.asarray(k, dtype=np.uint64).reshape(1, 4))[0] for k in mac_key_shares) % R
    vals = limbs_to_scalars(np.asarray(values, dtype=np.uint64).reshape(-1, 4))
    shares = [[rnd.randrange(R) for _ in vals] for _ in range(parties - 1)]
    macs = [[rnd.randrange(R) for _ in vals] for _ in range(parties - 1)]
    shares.append([(v - sum(col)) % R for v, col in zip(vals, zip(*shares))])
    macs.append([(alpha * v - sum(col)) % R for v, col in zip(vals, zip(*macs))])
    return [scalars_to_limbs(s) for s in shares], [scalars_to_limbs(m) for m in macs]


def dealer_share_auth(ctx: Context, seed: int, party: int, parties: int, values: np.ndarray) -> tuple:
    """INSECURE input stand-in (tests, benchmarks): this party's (shares, macs) of a table the caller knows in full,
    under the MAC key `MpcPrep.dealer_auth` derives from the same seed."""
    v = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
    sh, mac = np.zeros_like(v), np.zeros_like(v)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(ctx._lib.b200_mpc_dealer_share_auth(ctx._h, seed & (2**64 - 1), party, parties, vp(v), v.shape[0], vp(sh), vp(mac)))
    return sh, mac


@dataclass
class MpcAuthResult:
    proof: B200Proof
    link_poly_share: np.ndarray   # (n + 2, 4): this party's share of the linking polynomial
    link_poly_mac: np.ndarray     # (n + 2, 4): its MAC shares
    challenges: np.ndarray        # (6, 4): beta, gamma, alpha, zeta, v, u
    stats: dict


def prove_party_auth(ctx: Context, pk, transport: MpcTransport, prep: MpcPrep, mac_key_share: np.ndarray, wire_share: np.ndarray,
                     wire_mac: np.ndarray, pub_inputs: np.ndarray, blinder_share: np.ndarray, blinder_mac: np.ndarray,
                     proof: B200Proof = None) -> MpcAuthResult:
    """`b200_mpc_prove_auth` for one party.  `proof` (optional) is the buffer the opened proof is written to; it is
    left untouched when the call fails."""
    n = pk.domain_size
    arr = lambda a, k: np.ascontiguousarray(a, dtype=np.uint64).reshape(k, 4)
    w, wm = arr(wire_share, 5 * n), arr(wire_mac, 5 * n)
    bl, blm = arr(blinder_share, 17), arr(blinder_mac, 17)
    key = arr(mac_key_share, 1)
    pi = np.ascontiguousarray(pub_inputs, dtype=np.uint64).reshape(-1, 4)
    proof = B200Proof() if proof is None else proof
    link, link_mac = np.zeros((n + 2, 4), dtype=np.uint64), np.zeros((n + 2, 4), dtype=np.uint64)
    ch = np.zeros((6, 4), dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(ctx._lib.b200_mpc_prove_auth(ctx._h, pk._h, C.byref(transport), prep._h, vp(key), vp(w), vp(wm), vp(pi) if pi.size else None,
                                            vp(bl), vp(blm), C.byref(proof), vp(link), vp(link_mac), vp(ch)))
    return MpcAuthResult(proof, link, link_mac, ch, mpc_last_stats(ctx))


def prove_jointly_auth(ctxs, pks, wire_values, pub_inputs, blinder_values, seed: int = 0xBEA7E5, timeout_ms: int = 120000,
                       transports=None, inputs=None, keys=None):
    """All parties of one authenticated collaborative proof in this process, with dealer preprocessing from `seed`.
    The wire table and blinders are input with the dealer's MAC key (`dealer_share_auth`), unless `inputs` gives every
    party's (wire_share, wire_mac, blinder_share, blinder_mac); `keys` may replace the parties' MAC-key shares.  Returns
    every party's MpcAuthResult, or the B200Error it failed with."""
    P = len(ctxs)
    group = LocalGroup(P, timeout_ms) if transports is None else None
    trs = transports if transports is not None else [group.transport(p) for p in range(P)]
    made = [MpcPrep.dealer_auth(ctxs[p], pks[p], seed, p, P) for p in range(P)]
    preps = [m[0] for m in made]
    keys = keys if keys is not None else [m[1] for m in made]
    if inputs is None:  # wires and blinders as one table, so that no two values share a mask
        table = np.concatenate([np.asarray(wire_values, dtype=np.uint64).reshape(-1, 4), np.asarray(blinder_values, dtype=np.uint64).reshape(-1, 4)])
        k = table.shape[0] - 17
        inputs = []
        for p in range(P):
            sh, mac = dealer_share_auth(ctxs[p], seed, p, P, table)
            inputs.append((sh[:k], mac[:k], sh[k:], mac[k:]))
    try:
        return _run_parties([lambda p=p: prove_party_auth(ctxs[p], pks[p], trs[p], preps[p], keys[p], inputs[p][0], inputs[p][1],
                                                          pub_inputs, inputs[p][2], inputs[p][3]) for p in range(P)])
    finally:
        for pr in preps:
            pr.free()
        if group is not None:
            group.close()


def link_party_auth(ctx: Context, srs: Bases, transport: MpcTransport, mac_key_share: np.ndarray, a1_share: np.ndarray,
                    a1_mac: np.ndarray, a2_share: np.ndarray, a2_mac: np.ndarray, comm1: np.ndarray, comm2: np.ndarray, layout):
    """`b200_mpc_link_auth` for one party: (B200LinkProof, eta)."""
    from .backend import B200LinkProof
    arr = lambda a: np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
    a1, a1m, a2, a2m, key = arr(a1_share), arr(a1_mac), arr(a2_share), arr(a2_mac), arr(mac_key_share)
    c1 = np.ascontiguousarray(comm1, dtype=np.uint64).reshape(8)
    c2 = np.ascontiguousarray(comm2, dtype=np.uint64).reshape(8)
    proof = B200LinkProof()
    eta = np.zeros(4, dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(ctx._lib.b200_mpc_link_auth(ctx._h, srs._h, C.byref(transport), vp(key), vp(a1), vp(a1m), a1.shape[0], vp(a2), vp(a2m),
                                           a2.shape[0], vp(c1), vp(c2), layout.alignment, layout.offset, layout.size, C.byref(proof),
                                           vp(eta)))
    return proof, eta


def link_jointly_auth(ctxs, srss, keys, a1, a2, comm1, comm2, layout, timeout_ms: int = 120000, transports=None):
    """All parties of one authenticated collaborative link proof; `a1` / `a2` are per-party (share, mac) pairs.  Per
    party (B200LinkProof, eta) or its B200Error."""
    P = len(ctxs)
    group = LocalGroup(P, timeout_ms) if transports is None else None
    trs = transports if transports is not None else [group.transport(p) for p in range(P)]
    try:
        return _run_parties([lambda p=p: link_party_auth(ctxs[p], srss[p], trs[p], keys[p], a1[p][0], a1[p][1], a2[p][0], a2[p][1],
                                                         comm1, comm2, layout) for p in range(P)])
    finally:
        if group is not None:
            group.close()
