// Fiat–Shamir transcript of the prover: Keccak-256 "SolidityTranscript".
//
// Replaces the `SolidityTranscript` type parameter of
// `PlonkKzgSnark::prove_with_link_hint::<_, _, SolidityTranscript>`
// (/root/reference/crates/circuits/circuit-types/src/traits.rs:996) and of `link_proofs`
// (circuits-core/src/zk_circuits/proof_linking/intent_only.rs:42-47).  The type itself lives in
// the un-vendored mpc-jellyfish fork (plonk/src/transcript/solidity.rs @311568a4); the byte layout
// below is the published jellyfish 0.4 layout as recalled (SURVEY.md App. A) and is kept in this
// one header so it can be aligned with the fork's source when that is available:
//   * append-only byte buffer + 64-byte state;
//   * field elements / curve coordinates appended as 32-byte big-endian canonical integers;
//   * challenge = from_be_bytes_mod_order(state'[..48]),
//     state' = keccak256(state || transcript || 0x00) || keccak256(state || transcript || 0x01).
// Serial, a few KB per proof: runs on the host between device rounds of the prover.  Everything here is also
// __host__ __device__: the batch verifier (batch_verify.cu) replays one transcript per item in a device thread, so
// the layout stays defined once.
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#include "ec.cuh"
#include "ff.cuh"

namespace b200 {

#if defined(__CUDACC__)
#define TR_HD __host__ __device__
#define TR_HD_NOINLINE __host__ __device__ __noinline__
// TranscriptT<ByteVec> is instantiated by host code only: no device body is made for its calls into std::vector
#define TR_HOST_STORAGE_OK _Pragma("nv_exec_check_disable")
#else
#define TR_HD inline
#define TR_HD_NOINLINE
#define TR_HOST_STORAGE_OK
#endif

// Keccak-256 (pre-FIPS padding, as Ethereum's keccak256) as a streaming sponge, so a caller can absorb a common
// prefix once and finish two copies with different suffixes.
class Keccak256 {
  public:
    static constexpr size_t kRate = 136;
    TR_HD Keccak256() : fill_(0) {
        for (int i = 0; i < 25; ++i) st_[i] = 0;
    }
    TR_HD void absorb(const uint8_t* p, size_t n) {
#if !defined(__CUDA_ARCH__)
        while (fill_ == 0 && n >= kRate) {  // whole blocks straight from the input (host: the prover's transcript)
            absorb_block(st_, p);
            p += kRate;
            n -= kRate;
        }
#endif
        for (size_t i = 0; i < n; ++i) {
            blk_[fill_++] = p[i];
            if (fill_ == kRate) {
                absorb_block(st_, blk_);
                fill_ = 0;
            }
        }
    }
    TR_HD void finish(uint8_t out[32]) {
        for (unsigned i = fill_; i < kRate; ++i) blk_[i] = 0;
        blk_[fill_] ^= 0x01;
        blk_[kRate - 1] ^= 0x80;
        absorb_block(st_, blk_);
        for (int i = 0; i < 32; ++i) out[i] = (uint8_t)(st_[i >> 3] >> (8 * (i & 7)));
    }
    static TR_HD void hash(const uint8_t* data, size_t len, uint8_t out[32]) {
        Keccak256 k;
        k.absorb(data, len);
        k.finish(out);
    }

  private:
    static TR_HD uint64_t rotl(uint64_t x, int s) { return s ? (x << s) | (x >> (64 - s)) : x; }
    static TR_HD void absorb_block(uint64_t st[25], const uint8_t* block) {
        for (int i = 0; i < 17; ++i) {
            uint64_t lane = 0;
            for (int b = 0; b < 8; ++b) lane |= (uint64_t)block[8 * i + b] << (8 * b);
            st[i] ^= lane;
        }
        permute(st);
    }
    static TR_HD constexpr uint64_t round_constant(int r) {
        constexpr uint64_t v[24] = {
            0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,
            0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,
            0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,
            0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,
            0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
            0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
        return v[r];
    }
    static TR_HD constexpr int pi_lane(int i) {
        constexpr int v[24] = {10, 7, 11, 17, 18, 3, 5, 16, 8, 21, 24, 4, 15, 23, 19, 13, 12, 2, 20, 14, 22, 9, 6, 1};
        return v[i];
    }
    static TR_HD constexpr int rho_off(int i) {
        constexpr int v[24] = {1, 3, 6, 10, 15, 21, 28, 36, 45, 55, 2, 14, 27, 41, 56, 8, 25, 43, 62, 18, 39, 61, 20, 44};
        return v[i];
    }
    // Fully unrolled so that on the device the 25 lanes stay in registers and every table entry is an immediate
    static TR_HD void permute(uint64_t st[25]) {
        uint64_t a[25];
#pragma unroll
        for (int i = 0; i < 25; ++i) a[i] = st[i];
#pragma unroll
        for (int r = 0; r < 24; ++r) {
            uint64_t col[5];
#pragma unroll
            for (int x = 0; x < 5; ++x) col[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
#pragma unroll
            for (int x = 0; x < 5; ++x) {
                const uint64_t d = col[(x + 4) % 5] ^ rotl(col[(x + 1) % 5], 1);
#pragma unroll
                for (int y = 0; y < 25; y += 5) a[x + y] ^= d;
            }
            // lane (x, y) lives at a[x + 5y]; walk the pi permutation in place with the rho offsets
            uint64_t carry = a[1];
#pragma unroll
            for (int i = 0; i < 24; ++i) {
                const int j = pi_lane(i);
                const uint64_t tmp = a[j];
                a[j] = rotl(carry, rho_off(i));
                carry = tmp;
            }
#pragma unroll
            for (int y = 0; y < 25; y += 5) {
                uint64_t row[5];
#pragma unroll
                for (int x = 0; x < 5; ++x) row[x] = a[y + x];
#pragma unroll
                for (int x = 0; x < 5; ++x) a[y + x] = row[x] ^ (~row[(x + 1) % 5] & row[(x + 2) % 5]);
            }
            a[0] ^= round_constant(r);
        }
#pragma unroll
        for (int i = 0; i < 25; ++i) st[i] = a[i];
    }

    uint64_t st_[25];
    uint8_t blk_[kRate];
    unsigned fill_;
};

// Append-only byte storage of a transcript.  The prover's grows on the host; the verifier's is a span the caller sizes
// (plonk_transcript_bytes in verify_algebra.cuh), which works the same on the host and in a device thread.
struct ByteVec {
    std::vector<uint8_t> v;
    ByteVec() {}
    void append(const uint8_t* p, size_t n) { v.insert(v.end(), p, p + n); }
    const uint8_t* data() const { return v.data(); }
    size_t size() const { return v.size(); }
};
struct ByteSpan {
    uint8_t* p;
    size_t len, cap;
    TR_HD void append(const uint8_t* q, size_t n) {  // bytes past `cap` are dropped: callers size the span exactly
        for (size_t i = 0; i < n && len < cap; ++i) p[len++] = q[i];
    }
    TR_HD const uint8_t* data() const { return p; }
    TR_HD size_t size() const { return len; }
};

template <class Bytes>
class TranscriptT {
  public:
    TR_HOST_STORAGE_OK
    TR_HD TranscriptT() : buf_() {
        for (int i = 0; i < 64; ++i) state_[i] = 0;
    }
    TR_HD explicit TranscriptT(const Bytes& b) : buf_(b) {
        for (int i = 0; i < 64; ++i) state_[i] = 0;
    }

    TR_HOST_STORAGE_OK
    TR_HD void append_message(const uint8_t* p, size_t n) { buf_.append(p, n); }
    TR_HD void append_u32_be(uint32_t v) {
        const uint8_t b[4] = {(uint8_t)(v >> 24), (uint8_t)(v >> 16), (uint8_t)(v >> 8), (uint8_t)v};
        append_message(b, 4);
    }
    TR_HD void append_u64_be(uint64_t v) {
        uint8_t b[8];
        for (int i = 0; i < 8; ++i) b[i] = (uint8_t)(v >> (56 - 8 * i));
        append_message(b, 8);
    }
    // Montgomery Fr element -> 32 bytes big-endian canonical
    TR_HD void append_field_elem(const fe& a_mont) {
        uint8_t b[32];
        to_be(fe_from_mont<FrCfg>(a_mont), b);
        append_message(b, 32);
    }
    // affine commitment (Montgomery Fq coordinates); the identity is 64 zero bytes
    TR_HD void append_commitment(const g1_affine& c) {
        uint8_t b[32];
        to_be(fe_from_mont<FqCfg>(c.x), b);
        append_message(b, 32);
        to_be(fe_from_mont<FqCfg>(c.y), b);
        append_message(b, 32);
    }
    // get_and_append_challenge: returns the challenge in Montgomery form.  The two hashes share the prefix
    // state || transcript, which is absorbed once.  Out of line: a verifier calls it from six places, and the
    // unrolled permutation is large.
    TR_HOST_STORAGE_OK
    TR_HD_NOINLINE fe get_and_append_challenge() {
        Keccak256 k0;
        k0.absorb(state_, 64);
        k0.absorb(buf_.data(), buf_.size());
        Keccak256 k1 = k0;
        const uint8_t zero = 0, one = 1;
        k0.absorb(&zero, 1);
        k1.absorb(&one, 1);
        k0.finish(state_);
        k1.finish(state_ + 32);
        // big-endian 48-byte integer mod r, by Horner in Montgomery form
        fe acc = fe_zero();
        const fe c256 = fe_from_u32<FrCfg>(256);
        for (int i = 0; i < 48; ++i) acc = fe_add<FrCfg>(fe_mul<FrCfg>(acc, c256), fe_from_u32<FrCfg>(state_[i]));
        return acc;
    }
    // the 64-byte state after the last challenge: binds everything appended so far
    TR_HD const uint8_t* state() const { return state_; }

  private:
    static TR_HD void to_be(const fe& canon, uint8_t out[32]) {
        for (int i = 0; i < 8; ++i)
            for (int j = 0; j < 4; ++j) out[31 - (4 * i + j)] = (uint8_t)(canon.l[i] >> (8 * j));
    }
    Bytes buf_;
    uint8_t state_[64];
};

using SolidityTranscript = TranscriptT<ByteVec>;

}  // namespace b200
