// Bases stored as fixed-width codes (host only), the one description the reader and the rows writer share: BITS bits per
// base, most significant first, record r's base i in byte rec_byte[r] + i / (8 / BITS).
//   BITS = 2: a .2bit file's packed bases, T=0 C=1 A=2 G=3.
//   BITS = 4: a BAM file's codes =ACMGRSVTWYHKDBN; the complement of a code is its 4-bit bit-reversal.
#pragma once
#include <stdint.h>
#include <string.h>

template <int BITS>
struct PackedCodes {
    static_assert(BITS == 2 || BITS == 4, "2 or 4 bits per base");
    static constexpr uint32_t PER_BYTE = 8 / BITS;
    static constexpr const char *LETTERS = BITS == 2 ? "TCAG" : "=ACMGRSVTWYHKDBN";
};

// The letter of base i of the record whose codes start at rec.
template <int BITS>
static inline uint8_t code_letter(const uint8_t *rec, uint64_t i) {
    using C = PackedCodes<BITS>;
    return (uint8_t)C::LETTERS[(rec[i / C::PER_BYTE] >> (8 - BITS - BITS * (i % C::PER_BYTE))) & ((1u << BITS) - 1)];
}

// Bases [i, e) of the record whose codes start at rec, as letters into out[i, e): whole bytes through a table.
template <int BITS>
static void code_letters(const uint8_t *rec, uint64_t i, uint64_t e, uint8_t *out) {
    constexpr uint32_t PER_BYTE = PackedCodes<BITS>::PER_BYTE;
    static const struct Table {                           // a byte -> its PER_BYTE letters
        uint8_t v[256][PER_BYTE];
        Table() {
            for (uint32_t b = 0; b < 256; ++b) {
                const uint8_t byte = (uint8_t)b;
                for (uint32_t j = 0; j < PER_BYTE; ++j) v[b][j] = code_letter<BITS>(&byte, j);
            }
        }
    } table;
    for (; i < e && i % PER_BYTE; ++i) out[i] = code_letter<BITS>(rec, i);
    for (; i + PER_BYTE <= e; i += PER_BYTE) memcpy(out + i, table.v[rec[i / PER_BYTE]], PER_BYTE);
    for (; i < e; ++i) out[i] = code_letter<BITS>(rec, i);
}
