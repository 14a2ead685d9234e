// Packed wire format of the _host_packed entry points (include/amplisolve_b200.h): encoder / decoder of one
// (sample, strand, slot) word, shared by the C ABI (as_capi.cu), the ASEQ loader of the programs (as_host.cpp) and the
// pileup encoder on the device (as_pileup.cu), so that the packing rule lives in one place.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define AS_WIRE_HD __host__ __device__
#else
#define AS_WIRE_HD
#endif

// packed wire word -> four counts
AS_WIRE_HD static inline void as_unpack_word(uint32_t w, uint32_t* o) {
    const uint32_t m = w & 0xFFFFu, j = (w >> 16) & 3u;
    const uint32_t minor[3] = {(w >> 18) & 15u, (w >> 22) & 15u, (w >> 26) & 15u};
    for (uint32_t b = 0, k = 0; b < 4; ++b) o[b] = b == j ? m : minor[k++];
}

// four counts -> packed wire word; false when they do not fit (major > 65535 or another count > 15; *out is then
// unspecified).  The major base is the first largest count, the other three follow in base order.  Which base is the major
// one changes from row to row and the ASEQ loader calls this twice per row, so nothing here branches on it: a count beyond
// a nibble IS the major one (two of them do not fit), and only a word of four small counts needs the arg-max.
AS_WIRE_HD static inline bool as_pack_word(const uint32_t* v, uint32_t* out) {
    const uint32_t big = (uint32_t)(v[0] > 15u) | (uint32_t)(v[1] > 15u) << 1 | (uint32_t)(v[2] > 15u) << 2 | (uint32_t)(v[3] > 15u) << 3;
    if (big & (big - 1u)) return false;
    uint32_t j;
    if (big) {
#ifdef __CUDA_ARCH__
        j = (uint32_t)(__ffs((int)big) - 1);
#else
        j = (uint32_t)__builtin_ctz(big);
#endif
    } else {
        uint32_t m = v[1] > v[0] ? v[1] : v[0];
        j = v[1] > v[0] ? 1u : 0u;
        j = v[2] > m ? 2u : j;
        m = v[2] > m ? v[2] : m;
        j = v[3] > m ? 3u : j;
    }
    const uint32_t m = v[j];
    // nibbles of the four counts with the major one's taken out: the nibbles above it move down by one
    const uint32_t all = (v[0] & 15u) | (v[1] & 15u) << 4 | (v[2] & 15u) << 8 | (v[3] & 15u) << 12;
    const uint32_t below = (1u << (4 * j)) - 1u;
    *out = m | (j << 16) | (((all & below) | ((all >> 4) & ~below)) << 18);
    return m <= 0xFFFFu;
}

// The 16-bit wire format keeps four counts as they are unless one of them is >= AS_WIRE_ESCAPE (0xFFFE): then the record
// is escaped.  The rule of the ASEQ loader (as_host.cpp) and of the pileup encoder.
AS_WIRE_HD static inline bool as_wire16_fits(const uint32_t* v) {
    return v[0] < 0xFFFEu && v[1] < 0xFFFEu && v[2] < 0xFFFEu && v[3] < 0xFFFEu;
}
