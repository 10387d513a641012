// Verifier algebra shared by the host verifiers (verify.cu) and the batch verifier's device threads
// (batch_verify.cu): the transcript replay and the scalar assembly that turn one PlonK proof or one link proof into
// the two G1 operands of its KZG check
//     e(A, [tau]_2) == e(B, [1]_2),
// each given as a fixed-size list of (point, scalar) terms.  What the terms are summed with, and where, is the
// caller's business; the append order and the scalar formulas live only here.
#pragma once
#include "b200prover.h"
#include "ec.cuh"
#include "ff.cuh"
#include "transcript.h"

namespace b200 {

constexpr int kNW = 5, kNS = 13;

struct ProofIn {  // layout of b200_proof
    g1_affine wires_poly_comms[kNW];
    g1_affine prod_perm_poly_comm;
    g1_affine split_quot_poly_comms[kNW];
    g1_affine opening_proof;
    g1_affine shifted_opening_proof;
    fe wires_evals[kNW];
    fe wire_sigma_evals[kNW - 1];
    fe perm_next_eval;
};
static_assert(sizeof(ProofIn) == sizeof(b200_proof), "proof layout");

struct VkIn {  // the flat verifying key of b200_plonk_verify
    const fe* k;            // 5 coset representatives
    const g1_affine* sel;   // 13 selector commitments
    const g1_affine* sig;   // 5 sigma commitments
};

// s * P, s a Montgomery Fr element; a term with s == 0 or P the identity contributes nothing
struct G1Term {
    g1_affine p;
    fe s;
};
constexpr int kTermsA = 2, kTermsB = 34;  // the PlonK check's counts; a link check uses 1 and 4 of them
struct OperandTerms {
    G1Term a[kTermsA];
    G1Term b[kTermsB];
    int na, nb;
};

// Transcript bytes the PlonK verifier appends for `num_inputs` public inputs (size of its ByteSpan)
TR_HD constexpr size_t plonk_transcript_bytes(size_t num_inputs) {
    return 4 + 8 + 8 + 32 * kNW + 64 * kNS + 64 * kNW + 32 * num_inputs + 64 * kNW + 64 + 64 * kNW + 32 * (2 * kNW) + 128;
}
constexpr size_t kLinkTranscriptBytes = 3 * 64;

FF_HD fe fr_pow_u64(fe a, uint64_t e) {
    fe r = fe_one<FrCfg>();
    while (e) {
        if (e & 1) r = fe_mul<FrCfg>(r, a);
        a = fe_sqr<FrCfg>(a);
        e >>= 1;
    }
    return r;
}

FF_HD void term_put(G1Term* t, int* n, const g1_affine& p, const fe& s) {
    t[*n].p = p;
    t[*n].s = s;
    ++*n;
}

// PlonkKzgSnark::verify's challenges and operands.  Returns false, with no terms, when a proof or key element is off
// the curve (a rejection).  w: the generator of the 2^log_n-th roots of unity; tr: a fresh transcript with room for
// plonk_transcript_bytes(num_inputs).
template <class Bytes>
TR_HD bool plonk_verify_terms(unsigned log_n, size_t num_inputs, const VkIn& vk, const fe* pi, const ProofIn& proof,
                              const fe& w, TranscriptT<Bytes>& tr, OperandTerms* out) {
    using Fr = FrCfg;
    out->na = out->nb = 0;
    // every group element the verifier multiplies must be on the curve (the identity is allowed)
    bool ok = true;
    for (int i = 0; i < kNS; ++i) ok = ok && g1_affine_on_curve(vk.sel[i]);
    for (int i = 0; i < kNW; ++i)
        ok = ok && g1_affine_on_curve(vk.sig[i]) && g1_affine_on_curve(proof.wires_poly_comms[i]) &&
             g1_affine_on_curve(proof.split_quot_poly_comms[i]);
    ok = ok && g1_affine_on_curve(proof.prod_perm_poly_comm) && g1_affine_on_curve(proof.opening_proof) &&
         g1_affine_on_curve(proof.shifted_opening_proof);
    if (!ok) return false;
    const uint64_t n = (uint64_t)1 << log_n;
    // ---- challenges (same transcript as the prover, plonk.cu) ------------------------------------------------
    tr.append_u32_be(254);
    tr.append_u64_be(n);
    tr.append_u64_be((uint64_t)num_inputs);
    for (int i = 0; i < kNW; ++i) tr.append_field_elem(vk.k[i]);
    for (int s = 0; s < kNS; ++s) tr.append_commitment(vk.sel[s]);
    for (int i = 0; i < kNW; ++i) tr.append_commitment(vk.sig[i]);
    for (size_t i = 0; i < num_inputs; ++i) tr.append_field_elem(pi[i]);
    for (int i = 0; i < kNW; ++i) tr.append_commitment(proof.wires_poly_comms[i]);
    const fe beta = tr.get_and_append_challenge();
    const fe gamma = tr.get_and_append_challenge();
    tr.append_commitment(proof.prod_perm_poly_comm);
    const fe alpha = tr.get_and_append_challenge();
    for (int i = 0; i < kNW; ++i) tr.append_commitment(proof.split_quot_poly_comms[i]);
    const fe zeta = tr.get_and_append_challenge();
    for (int i = 0; i < kNW; ++i) tr.append_field_elem(proof.wires_evals[i]);
    for (int i = 0; i < kNW - 1; ++i) tr.append_field_elem(proof.wire_sigma_evals[i]);
    tr.append_field_elem(proof.perm_next_eval);
    const fe v = tr.get_and_append_challenge();
    tr.append_commitment(proof.opening_proof);
    tr.append_commitment(proof.shifted_opening_proof);
    const fe u = tr.get_and_append_challenge();

    // ---- scalars ---------------------------------------------------------------------------------------------
    const fe one = fe_one<Fr>();
    const fe vanish = fe_sub<Fr>(fr_pow_u64(zeta, n), one);
    fe nfr = fe_zero();
    nfr.l[0] = (uint32_t)n;
    nfr.l[1] = (uint32_t)(n >> 32);
    nfr = fe_to_mont<Fr>(nfr);
    // PI(zeta) = sum_j pi_j w^j Z_H(zeta) / (n (zeta - w^j)) and L_1(zeta) = Z_H(zeta) / (n (zeta - 1)) with ONE
    // inversion: the fractions are summed over a common denominator.  zeta on the domain makes a denominator vanish;
    // such a term takes the inverse 0 (fe_inv(0) == 0 on the host and the device alike), and the proof is rejected
    // by the pairing, as the reference rejects it (probability ~ n / r).
    fe num = fe_zero(), den = one, wj = one;
    for (size_t j = 0; j < num_inputs; ++j) {
        const fe d = fe_mul<Fr>(fe_sub<Fr>(zeta, wj), nfr);
        if (!fe_is_zero(d)) {
            const fe c = fe_mul<Fr>(fe_mul<Fr>(vanish, wj), pi[j]);
            num = fe_add<Fr>(fe_mul<Fr>(num, d), fe_mul<Fr>(c, den));
            den = fe_mul<Fr>(den, d);
        }
        wj = fe_mul<Fr>(wj, w);
    }
    const fe d0 = fe_mul<Fr>(fe_sub<Fr>(zeta, one), nfr);
    const bool d0_zero = fe_is_zero(d0);
    const fe d0x = d0_zero ? one : d0;
    const fe inv = fe_inv<Fr>(fe_mul<Fr>(den, d0x));
    const fe pi_eval = fe_mul<Fr>(fe_mul<Fr>(num, inv), d0x);
    const fe l1 = d0_zero ? fe_zero() : fe_mul<Fr>(vanish, fe_mul<Fr>(inv, den));
    const fe alpha2 = fe_sqr<Fr>(alpha);
    const fe* we = proof.wires_evals;
    const fe* se = proof.wire_sigma_evals;
    // r0 = PI - alpha^2 L1 - alpha z_w prod_{i<4} (w_i + beta s_i + gamma) (w_4 + gamma)
    fe prod = fe_mul<Fr>(alpha, proof.perm_next_eval);
    for (int j = 0; j < kNW - 1; ++j) prod = fe_mul<Fr>(prod, fe_add<Fr>(fe_add<Fr>(fe_mul<Fr>(se[j], beta), we[j]), gamma));
    const fe prod4 = fe_mul<Fr>(prod, fe_add<Fr>(we[4], gamma));
    const fe r0 = fe_sub<Fr>(fe_sub<Fr>(pi_eval, fe_mul<Fr>(alpha2, l1)), prod4);

    // ---- D: linearisation commitment (B collects D, then F, then the opening terms) -------------------------------
    G1Term* B = out->b;
    int* nb = &out->nb;
    for (int j = 0; j < 4; ++j) term_put(B, nb, vk.sel[j], we[j]);
    term_put(B, nb, vk.sel[4], fe_mul<Fr>(we[0], we[1]));
    term_put(B, nb, vk.sel[5], fe_mul<Fr>(we[2], we[3]));
    for (int j = 0; j < 4; ++j) term_put(B, nb, vk.sel[6 + j], fe_mul<Fr>(fe_sqr<Fr>(fe_sqr<Fr>(we[j])), we[j]));
    term_put(B, nb, vk.sel[10], fe_neg<Fr>(we[4]));
    term_put(B, nb, vk.sel[11], one);
    term_put(B, nb, vk.sel[12], fe_mul<Fr>(fe_mul<Fr>(fe_mul<Fr>(we[0], we[1]), fe_mul<Fr>(we[2], we[3])), we[4]));
    fe coeff = alpha;
    for (int j = 0; j < kNW; ++j)
        coeff = fe_mul<Fr>(coeff, fe_add<Fr>(fe_add<Fr>(fe_mul<Fr>(fe_mul<Fr>(vk.k[j], zeta), beta), we[j]), gamma));
    coeff = fe_add<Fr>(coeff, fe_mul<Fr>(alpha2, l1));
    term_put(B, nb, proof.prod_perm_poly_comm, coeff);
    term_put(B, nb, vk.sig[kNW - 1], fe_neg<Fr>(fe_mul<Fr>(prod, beta)));
    const fe zn2 = fe_mul<Fr>(fe_mul<Fr>(fe_add<Fr>(vanish, one), zeta), zeta);
    fe c = fe_neg<Fr>(vanish);
    for (int i = 0; i < kNW; ++i) {
        term_put(B, nb, proof.split_quot_poly_comms[i], c);
        c = fe_mul<Fr>(c, zn2);
    }
    // ---- F, E: batched opening at zeta -------------------------------------------------------------------------
    fe E = fe_neg<Fr>(r0), vp = one;
    for (int i = 0; i < kNW; ++i) {
        vp = fe_mul<Fr>(vp, v);
        term_put(B, nb, proof.wires_poly_comms[i], vp);
        E = fe_add<Fr>(E, fe_mul<Fr>(vp, we[i]));
    }
    for (int i = 0; i < kNW - 1; ++i) {
        vp = fe_mul<Fr>(vp, v);
        term_put(B, nb, vk.sig[i], vp);
        E = fe_add<Fr>(E, fe_mul<Fr>(vp, se[i]));
    }
    // ---- pairing operands: A = W_z + u W_zw,  B = zeta W_z + u zeta w W_zw + F - E G + u ([z] - z_w G) -------------
    g1_affine G;
    G.x = fe_one<FqCfg>();
    G.y = fe_from_u32<FqCfg>(2);
    term_put(out->a, &out->na, proof.opening_proof, one);
    term_put(out->a, &out->na, proof.shifted_opening_proof, u);
    term_put(B, nb, G, fe_neg<Fr>(E));
    term_put(B, nb, proof.opening_proof, zeta);
    term_put(B, nb, proof.shifted_opening_proof, fe_mul<Fr>(u, fe_mul<Fr>(zeta, w)));
    term_put(B, nb, proof.prod_perm_poly_comm, u);
    term_put(B, nb, G, fe_neg<Fr>(fe_mul<Fr>(u, proof.perm_next_eval)));
    return true;
}

// PlonkKzgSnark::verify_link_proof's challenge and operands: (tau - eta) pi == C1 - C2 - Z_D(eta) Cq, i.e.
// A = pi, B = C1 - C2 - Z_D(eta) Cq + eta pi, with Z_D the vanishing polynomial of the group g^(offset + i), i < size.
// Returns false, with no terms, when a point is off the curve.  g: the generator of the 2^alignment-th roots of unity;
// tr: a fresh transcript with room for kLinkTranscriptBytes.
template <class Bytes>
TR_HD bool link_verify_terms(const g1_affine& c1, const g1_affine& c2, const g1_affine& cq, const g1_affine& op,
                             const fe& g, uint64_t offset, uint64_t size, TranscriptT<Bytes>& tr, OperandTerms* out) {
    using Fr = FrCfg;
    out->na = out->nb = 0;
    if (!g1_affine_on_curve(c1) || !g1_affine_on_curve(c2) || !g1_affine_on_curve(cq) || !g1_affine_on_curve(op))
        return false;
    tr.append_commitment(c1);
    tr.append_commitment(c2);
    tr.append_commitment(cq);
    const fe eta = tr.get_and_append_challenge();
    fe root = fr_pow_u64(g, offset), zd = fe_one<Fr>();
    for (uint64_t i = 0; i < size; ++i) {
        zd = fe_mul<Fr>(zd, fe_sub<Fr>(eta, root));
        root = fe_mul<Fr>(root, g);
    }
    term_put(out->a, &out->na, op, fe_one<Fr>());
    term_put(out->b, &out->nb, c1, fe_one<Fr>());
    term_put(out->b, &out->nb, g1_affine_neg(c2), fe_one<Fr>());
    term_put(out->b, &out->nb, cq, fe_neg<Fr>(zd));
    term_put(out->b, &out->nb, op, eta);
    return true;
}

}  // namespace b200
