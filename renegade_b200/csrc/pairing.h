// Host BN254 pairing of verify.cu, exposed within the library for the batch verifier's final check.
#pragma once
#include <cstddef>
#include <cstdint>

#include "ec.cuh"

namespace b200 {

struct fq2 {
    fe a, b;  // a + b u
};
struct g2_affine {
    fq2 x, y;
    bool inf;
};

// 128-byte record x0 || x1 || y0 || y1 (Montgomery), the ptau layout read by srs.rs:185-199
g2_affine g2_load(const uint64_t rec[16]);
bool g2_on_curve(const g2_affine& p);
// prod_i e(ps[i], qs[i]) == 1: one shared Miller loop (miller_loop_product) and one final_exponentiation
bool pairing_product_is_one(const g1_affine* ps, const g2_affine* qs, size_t k);

}  // namespace b200
