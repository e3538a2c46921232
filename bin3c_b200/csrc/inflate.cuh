// Raw-deflate (RFC 1951) decoder and CRC-32 for one BGZF block, written once for the device decoder (bamdec.cu) and
// for a plain C++ build on the host (tests/native/inflate_check.cpp compares that build with zlib).
//
// Decoding follows the canonical-Huffman scheme of Mark Adler's puff.c: a code is described by the number of codes of
// each length and the symbols in canonical order, and a symbol is decoded one bit at a time against those counts.
// Tables of that form are small (about 700 bytes for the literal/length and distance codes), so each decoding thread
// keeps its own in local memory.  What is accepted and what is rejected is what zlib's inflate accepts and rejects:
// stored length check, at most 286 literal/length and 30 distance codes, complete code-length code, over-subscribed
// codes, incomplete codes only for a single code of length one, a missing end-of-block code, repeats without a
// previous length or past the end, invalid fixed-code symbols, and distances reaching before the start of the output.
// Every read of the input and every write of the output is bounds-checked.
#pragma once

#include <stdint.h>

#ifdef __CUDACC__
#define B3C_HD __host__ __device__ __forceinline__
#else
#define B3C_HD inline
#endif

namespace b3c_inflate {

enum {
    OK = 0,
    ERR_INPUT = -1,          // input ended before the last block did
    ERR_OUTPUT = -2,         // output would exceed its capacity
    ERR_BLOCK_TYPE = -3,     // block type 3
    ERR_STORED_LEN = -4,     // stored block length does not match its complement
    ERR_COUNTS = -5,         // too many literal/length or distance codes
    ERR_CODELEN_CODE = -6,   // code-length code over-subscribed or incomplete
    ERR_REPEAT = -7,         // repeat without a previous length, or past the end of the lengths
    ERR_LITLEN_CODE = -8,    // literal/length code over-subscribed or incomplete, or no end-of-block code
    ERR_DIST_CODE = -9,      // distance code over-subscribed or incomplete
    ERR_SYMBOL = -10,        // a bit pattern that is no code of the table, or a fixed-code symbol outside the alphabet
    ERR_DISTANCE = -11,      // distance before the start of the output
};

constexpr int MAXBITS = 15;
constexpr int MAXLCODES = 286;
constexpr int MAXDCODES = 30;
constexpr int FIXLCODES = 288;

struct Huffman {
    uint16_t count[MAXBITS + 1];
    uint16_t symbol[FIXLCODES];
};

struct State {
    const uint8_t *in;
    int64_t in_len, in_pos;
    uint8_t *out;
    int64_t out_cap, out_pos;
    uint64_t bitbuf;
    int bitcnt;
    bool overrun;            // a read past the end of the input was attempted
};

// the next `need` bits (0 <= need <= 32), least significant first; past the end of the input, zeros and `overrun`
B3C_HD uint32_t bits(State &s, int need) {
    while (s.bitcnt < need) {
        uint64_t b = 0;
        if (s.in_pos < s.in_len) b = s.in[s.in_pos];
        else s.overrun = true;
        s.in_pos += 1;
        s.bitbuf |= b << s.bitcnt;
        s.bitcnt += 8;
    }
    const uint32_t v = (uint32_t)(s.bitbuf & ((need == 32) ? 0xffffffffull : ((1ull << need) - 1)));
    s.bitbuf >>= need;
    s.bitcnt -= need;
    return v;
}

// one symbol, read bit by bit against the canonical code; < 0 on an unused bit pattern
B3C_HD int decode(State &s, const Huffman &h) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= MAXBITS; ++len) {
        code |= (int)bits(s, 1);
        const int count = h.count[len];
        if (code - count < first) return h.symbol[index + (code - first)];
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
        if (s.overrun) return ERR_INPUT;
    }
    return ERR_SYMBOL;
}

// canonical tables from code lengths; returns 0 for a complete code, > 0 for an incomplete one, < 0 over-subscribed
B3C_HD int construct(Huffman &h, const uint8_t *length, int n) {
    for (int len = 0; len <= MAXBITS; ++len) h.count[len] = 0;
    for (int sym = 0; sym < n; ++sym) h.count[length[sym]]++;
    if (h.count[0] == n) return 0;          // no codes: complete, but decoding any symbol fails
    int left = 1;
    for (int len = 1; len <= MAXBITS; ++len) {
        left <<= 1;
        left -= h.count[len];
        if (left < 0) return left;
    }
    uint16_t offs[MAXBITS + 1];
    offs[1] = 0;
    for (int len = 1; len < MAXBITS; ++len) offs[len + 1] = offs[len] + h.count[len];
    for (int sym = 0; sym < n; ++sym)
        if (length[sym] != 0) h.symbol[offs[length[sym]]++] = (uint16_t)sym;
    return left;
}

B3C_HD int stored(State &s) {
    s.bitbuf = 0;                            // drop the rest of the current byte
    s.bitcnt = 0;
    if (s.in_pos + 4 > s.in_len) return ERR_INPUT;
    const uint32_t len = s.in[s.in_pos] | (s.in[s.in_pos + 1] << 8);
    const uint32_t nlen = s.in[s.in_pos + 2] | (s.in[s.in_pos + 3] << 8);
    s.in_pos += 4;
    if (len != (~nlen & 0xffffu)) return ERR_STORED_LEN;
    if (s.in_pos + len > s.in_len) return ERR_INPUT;
    if (s.out_pos + len > s.out_cap) return ERR_OUTPUT;
    for (uint32_t k = 0; k < len; ++k) s.out[s.out_pos + k] = s.in[s.in_pos + k];
    s.in_pos += len;
    s.out_pos += len;
    return OK;
}

B3C_HD int codes(State &s, const Huffman &lencode, const Huffman &distcode) {
    const uint16_t LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31,
                                35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    const uint8_t LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    const uint16_t DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129,
                                193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    const uint8_t DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    for (;;) {
        int symbol = decode(s, lencode);
        if (s.overrun) return ERR_INPUT;
        if (symbol < 0) return symbol;
        if (symbol < 256) {
            if (s.out_pos >= s.out_cap) return ERR_OUTPUT;
            s.out[s.out_pos++] = (uint8_t)symbol;
        } else if (symbol == 256) {
            return OK;
        } else {
            symbol -= 257;
            if (symbol >= 29) return ERR_SYMBOL;                 // 286, 287 of the fixed code
            const int len = LBASE[symbol] + (int)bits(s, LEXT[symbol]);
            symbol = decode(s, distcode);
            if (s.overrun) return ERR_INPUT;
            if (symbol < 0) return symbol;
            if (symbol >= 30) return ERR_SYMBOL;                 // 30, 31 of the fixed code
            const int64_t dist = DBASE[symbol] + (int64_t)bits(s, DEXT[symbol]);
            if (s.overrun) return ERR_INPUT;
            if (dist > s.out_pos) return ERR_DISTANCE;
            if (s.out_pos + len > s.out_cap) return ERR_OUTPUT;
            uint8_t *o = s.out + s.out_pos;
            for (int k = 0; k < len; ++k) o[k] = o[k - dist];   // byte by byte: overlapping copies repeat
            s.out_pos += len;
        }
    }
}

B3C_HD int fixed(State &s) {
    Huffman lencode, distcode;
    uint8_t lengths[FIXLCODES];
    int sym = 0;
    for (; sym < 144; ++sym) lengths[sym] = 8;
    for (; sym < 256; ++sym) lengths[sym] = 9;
    for (; sym < 280; ++sym) lengths[sym] = 7;
    for (; sym < FIXLCODES; ++sym) lengths[sym] = 8;
    construct(lencode, lengths, FIXLCODES);
    for (sym = 0; sym < MAXDCODES; ++sym) lengths[sym] = 5;
    construct(distcode, lengths, MAXDCODES);
    return codes(s, lencode, distcode);
}

B3C_HD int dynamic(State &s) {
    const uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint8_t lengths[MAXLCODES + MAXDCODES];
    Huffman lencode, distcode;
    const int nlen = (int)bits(s, 5) + 257;
    const int ndist = (int)bits(s, 5) + 1;
    const int ncode = (int)bits(s, 4) + 4;
    if (s.overrun) return ERR_INPUT;
    if (nlen > MAXLCODES || ndist > MAXDCODES) return ERR_COUNTS;
    int index = 0;
    for (; index < ncode; ++index) lengths[ORDER[index]] = (uint8_t)bits(s, 3);
    for (; index < 19; ++index) lengths[ORDER[index]] = 0;
    if (s.overrun) return ERR_INPUT;
    if (construct(lencode, lengths, 19) != 0) return ERR_CODELEN_CODE;
    index = 0;
    while (index < nlen + ndist) {
        int symbol = decode(s, lencode);
        if (s.overrun) return ERR_INPUT;
        if (symbol < 0) return symbol;
        if (symbol < 16) {
            lengths[index++] = (uint8_t)symbol;
        } else {
            uint8_t len = 0;
            if (symbol == 16) {
                if (index == 0) return ERR_REPEAT;
                len = lengths[index - 1];
                symbol = 3 + (int)bits(s, 2);
            } else if (symbol == 17) {
                symbol = 3 + (int)bits(s, 3);
            } else {
                symbol = 11 + (int)bits(s, 7);
            }
            if (s.overrun) return ERR_INPUT;
            if (index + symbol > nlen + ndist) return ERR_REPEAT;
            while (symbol--) lengths[index++] = len;
        }
    }
    if (lengths[256] == 0) return ERR_LITLEN_CODE;
    int err = construct(lencode, lengths, nlen);
    if (err && (err < 0 || nlen != lencode.count[0] + lencode.count[1])) return ERR_LITLEN_CODE;
    err = construct(distcode, lengths + nlen, ndist);
    if (err && (err < 0 || ndist != distcode.count[0] + distcode.count[1])) return ERR_DIST_CODE;
    return codes(s, lencode, distcode);
}

// Inflate the raw-deflate stream in[0, in_len) into out[0, out_cap).  Returns OK or a negative error; *out_len gets
// the bytes written.  Input after the last block is ignored (as zlib leaves it unused).
B3C_HD int inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_cap, int64_t *out_len) {
    State s;
    s.in = in;
    s.in_len = in_len;
    s.in_pos = 0;
    s.out = out;
    s.out_cap = out_cap;
    s.out_pos = 0;
    s.bitbuf = 0;
    s.bitcnt = 0;
    s.overrun = false;
    int last, err;
    do {
        last = (int)bits(s, 1);
        const int type = (int)bits(s, 2);
        if (s.overrun) {
            err = ERR_INPUT;
            break;
        }
        err = type == 0 ? stored(s) : type == 1 ? fixed(s) : type == 2 ? dynamic(s) : ERR_BLOCK_TYPE;
        if (err == OK && s.overrun) err = ERR_INPUT;
    } while (err == OK && !last);
    *out_len = s.out_pos;
    return err;
}

// ---- CRC-32 (the gzip polynomial, reflected) ------------------------------------------------------------------------
constexpr uint32_t CRC_POLY = 0xedb88320u;

B3C_HD void crc32_table(uint32_t *table) {
    for (uint32_t n = 0; n < 256; ++n) {
        uint32_t c = n;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
        table[n] = c;
    }
}

// crc of p[0, n) continuing from `crc` (0 for a fresh start), as zlib's crc32(crc, p, n)
B3C_HD uint32_t crc32_update(const uint32_t *table, uint32_t crc, const uint8_t *p, int64_t n) {
    uint32_t c = ~crc;
    for (int64_t k = 0; k < n; ++k) c = table[(c ^ p[k]) & 0xff] ^ (c >> 8);
    return ~c;
}

// a * b modulo the CRC polynomial, both reflected (zlib's multmodp)
B3C_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m; m >>= 1) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        b = (b & 1) ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}

// x^(8 n) modulo the polynomial: the operator that advances a CRC over n zero bytes
B3C_HD uint32_t x8nmodp(int64_t n) {
    uint32_t p = 1u << 31;                   // x^0
    uint32_t sq = 1u << 30;                  // x^1
    for (int k = 0; k < 3; ++k) sq = multmodp(sq, sq);   // x^8
    while (n) {
        if (n & 1) p = multmodp(sq, p);
        n >>= 1;
        if (n) sq = multmodp(sq, sq);
    }
    return p;
}

// crc(A || B) from crc(A), crc(B) and len(B) (zlib's crc32_combine)
B3C_HD uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, int64_t len2) {
    return multmodp(x8nmodp(len2), crc1) ^ crc2;
}

}  // namespace b3c_inflate
