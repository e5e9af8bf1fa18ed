// SHA3-256 on the device (FIPS 202: Keccak-f[1600], rate 136 bytes, suffix 0x06), shared by the polynomial commitment's
// leaf and tree hashes (pc_commit.cu) and the device Fiat-Shamir transcript (fs_device.cuh). One thread runs the whole
// permutation; messages are whole 64-bit little-endian words.
#pragma once
#include <stdint.h>

#include "field.cuh"

namespace vp {

static __constant__ uint64_t VP_KECCAK_RC[24] = {
    0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL, 0x000000000000808bULL,
    0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL, 0x000000000000008aULL, 0x0000000000000088ULL,
    0x0000000080008009ULL, 0x000000008000000aULL, 0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL,
    0x8000000000008003ULL, 0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
    0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
VP_D uint64_t keccak_rotl(uint64_t x, int n) { return (x << n) | (x >> (64 - n)); }

VP_D void keccak_f1600(uint64_t (&a)[25]) {
#pragma unroll 1
    for (int round = 0; round < 24; ++round) {
        uint64_t c0 = a[0] ^ a[5] ^ a[10] ^ a[15] ^ a[20], c1 = a[1] ^ a[6] ^ a[11] ^ a[16] ^ a[21],
                 c2 = a[2] ^ a[7] ^ a[12] ^ a[17] ^ a[22], c3 = a[3] ^ a[8] ^ a[13] ^ a[18] ^ a[23],
                 c4 = a[4] ^ a[9] ^ a[14] ^ a[19] ^ a[24];
        const uint64_t d0 = c4 ^ keccak_rotl(c1, 1), d1 = c0 ^ keccak_rotl(c2, 1), d2 = c1 ^ keccak_rotl(c3, 1),
                       d3 = c2 ^ keccak_rotl(c4, 1), d4 = c3 ^ keccak_rotl(c0, 1);
#pragma unroll
        for (int j = 0; j < 25; j += 5) { a[j] ^= d0; a[j + 1] ^= d1; a[j + 2] ^= d2; a[j + 3] ^= d3; a[j + 4] ^= d4; }
        // rho + pi
        uint64_t b[25];
        b[0] = a[0];
        b[10] = keccak_rotl(a[1], 1);   b[7] = keccak_rotl(a[10], 3);   b[11] = keccak_rotl(a[7], 6);   b[17] = keccak_rotl(a[11], 10);
        b[18] = keccak_rotl(a[17], 15); b[3] = keccak_rotl(a[18], 21);  b[5] = keccak_rotl(a[3], 28);   b[16] = keccak_rotl(a[5], 36);
        b[8] = keccak_rotl(a[16], 45);  b[21] = keccak_rotl(a[8], 55);  b[24] = keccak_rotl(a[21], 2);  b[4] = keccak_rotl(a[24], 14);
        b[15] = keccak_rotl(a[4], 27);  b[23] = keccak_rotl(a[15], 41); b[19] = keccak_rotl(a[23], 56); b[13] = keccak_rotl(a[19], 8);
        b[12] = keccak_rotl(a[13], 25); b[2] = keccak_rotl(a[12], 43);  b[20] = keccak_rotl(a[2], 62);  b[14] = keccak_rotl(a[20], 18);
        b[22] = keccak_rotl(a[14], 39); b[9] = keccak_rotl(a[22], 61);  b[6] = keccak_rotl(a[9], 20);   b[1] = keccak_rotl(a[6], 44);
        // chi
#pragma unroll
        for (int j = 0; j < 25; j += 5) {
            a[j] = b[j] ^ (~b[j + 1] & b[j + 2]);
            a[j + 1] = b[j + 1] ^ (~b[j + 2] & b[j + 3]);
            a[j + 2] = b[j + 2] ^ (~b[j + 3] & b[j + 4]);
            a[j + 3] = b[j + 3] ^ (~b[j + 4] & b[j]);
            a[j + 4] = b[j + 4] ^ (~b[j] & b[j + 1]);
        }
        a[0] ^= VP_KECCAK_RC[round];
    }
}

// SHA3-256 of one 64-byte block: a single permutation. msg: 8 words in, digest: words 0..3 out
VP_D void sha3_256_64(const uint64_t (&msg)[8], uint64_t (&dig)[4]) {
    uint64_t a[25];
#pragma unroll
    for (int i = 0; i < 25; ++i) a[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = msg[i];
    a[8] = 0x06ULL;                      // domain suffix + first pad bit right after the 64 message bytes
    a[16] = 0x8000000000000000ULL;       // last pad bit in the last byte of the 136-byte rate
    keccak_f1600(a);
#pragma unroll
    for (int i = 0; i < 4; ++i) dig[i] = a[i];
}

// SHA3-256 of n_words words (any length: multi-block absorb, 17 words per block)
VP_D void sha3_256_words(const uint64_t* w, uint32_t n_words, uint64_t (&dig)[4]) {
    uint64_t a[25];
#pragma unroll
    for (int i = 0; i < 25; ++i) a[i] = 0;
    uint32_t k = 0;
    for (; k + 17 <= n_words; k += 17) {
#pragma unroll
        for (int i = 0; i < 17; ++i) a[i] ^= w[k + i];
        keccak_f1600(a);
    }
    // the last, partial block and the padding: 0x06 in the byte right after the message, 0x80 in the last byte of the
    // rate (the state is only indexed by constants, so that it stays in registers)
    const uint32_t rest = n_words - k;
#pragma unroll
    for (int i = 0; i < 17; ++i) {
        if ((uint32_t)i < rest) a[i] ^= w[k + i];
        if ((uint32_t)i == rest) a[i] ^= 0x06ULL;
    }
    a[16] ^= 0x8000000000000000ULL;
    keccak_f1600(a);
#pragma unroll
    for (int i = 0; i < 4; ++i) dig[i] = a[i];
}

}  // namespace vp
