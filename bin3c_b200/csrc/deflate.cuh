// Raw-deflate (RFC 1951) encoder for one BGZF member, written once for the device encoder (bgzf.cu) and for a plain
// C++ build on the host (tests/native/deflate_check.cpp compares that build with zlib and with the device output).
//
// A member is a function of its input bytes only (at most MEMBER_INPUT of them), so the output does not depend on how
// the stream is cut into slabs, nor on which build ran it.  The steps, each a function the device runs in parallel
// and deflate_member() below runs serially:
//   chains       prev[i]: the last position j < i with the same hash of 3 bytes (NONE if there is none)
//   find_match   the longest match at i over at most MAX_CHAIN chain entries within 32 KiB (nearest on ties; a search
//                stops at NICE bytes; a 3-byte match further than TOO_FAR away is dropped, as zlib drops it)
//   parse        greedy with one step of lazy evaluation (a match shorter than LAZY is given up for a literal when
//                the next position has a longer one): token starts are marked TOKEN | length (0 for a literal)
//   plan_dynamic Huffman code lengths from the token histograms (Moffat-Katajainen on the symbols sorted by
//                (frequency, symbol); longer than 15 bits, or 7 for the code-length code, folded back by the Kraft
//                count fix-up of miniz), canonical codes, the run-length coded header and the block's size in bits
//   emission     one final dynamic block, or one stored block when that is not longer
// The window never reaches into another member.
#pragma once

#include <stdint.h>

#include "inflate.cuh"

namespace b3c_deflate {

constexpr int MEMBER_INPUT = 65280;          // input bytes per member (what BGZF writers use)
constexpr int MEMBER_MAX = 65536;            // BSIZE is 16 bits: no member is longer
constexpr int HEADER_BYTES = 18, TRAILER_BYTES = 8;
constexpr int HASH_BITS = 13, HASH_SIZE = 1 << HASH_BITS;
constexpr uint16_t NONE = 0xffff;
constexpr int MIN_MATCH = 3, MAX_MATCH = 258, WINDOW = 32768;
constexpr int MAX_CHAIN = 48, NICE = 128, LAZY = 16, TOO_FAR = 4096;
constexpr uint16_t TOKEN = 0x8000;
constexpr int LCODES = 286, DCODES = 30, BLCODES = 19;
constexpr int MAX_RLE = LCODES + DCODES;

// the largest member payload: a stored block of MEMBER_INPUT bytes
constexpr int STORED_OVERHEAD = 5;
static_assert(HEADER_BYTES + MEMBER_INPUT + STORED_OVERHEAD + TRAILER_BYTES <= MEMBER_MAX, "member bound");

B3C_HD uint32_t hash3(const uint8_t *p) {
    return ((uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16)) * 2654435761u >> (32 - HASH_BITS);
}

B3C_HD int match_len(const uint8_t *a, const uint8_t *b, int maxlen) {
    int k = 0;
    while (k < maxlen && a[k] == b[k]) ++k;
    return k;
}

// the match at position i of in[0, n) over the hash chain prev; returns its length (0: none) and *dist
B3C_HD int find_match(const uint8_t *in, int n, const uint16_t *prev, int i, int *dist) {
    *dist = 0;
    if (i + MIN_MATCH > n) return 0;
    const int maxlen = n - i < MAX_MATCH ? n - i : MAX_MATCH;
    int best = MIN_MATCH - 1, bdist = 0;
    int j = prev[i];
    for (int c = 0; c < MAX_CHAIN && j != NONE && i - j <= WINDOW; ++c) {
        if (in[j + best] == in[i + best]) {           // cannot be longer otherwise
            const int l = match_len(in + j, in + i, maxlen);
            if (l > best) {
                best = l;
                bdist = i - j;
                if (l >= NICE || l == maxlen) break;
            }
        }
        j = prev[j];
    }
    if (best < MIN_MATCH || (best == MIN_MATCH && bdist > TOO_FAR)) return 0;
    *dist = bdist;
    return best;
}

// lens[i]: the match length at i (0: none); on return the token starts carry TOKEN | length (0 for a literal)
B3C_HD void parse(uint16_t *lens, int n) {
    int i = 0;
    while (i < n) {
        const int l = lens[i];
        if (l >= MIN_MATCH && (l >= LAZY || i + 1 >= n || lens[i + 1] <= l)) {
            lens[i] = (uint16_t)(TOKEN | l);
            i += l;
        } else {
            lens[i] = TOKEN;
            i += 1;
        }
    }
}

// the length and distance code tables of RFC 1951 3.2.5, as formulas (no table in device memory)
B3C_HD int lext(int c) { return (c < 8 || c == 28) ? 0 : (c >> 2) - 1; }
B3C_HD int lbase(int c) { return c < 8 ? c + 3 : c == 28 ? MAX_MATCH : ((4 + (c & 3)) << ((c >> 2) - 1)) + 3; }
B3C_HD int dext(int c) { return c < 4 ? 0 : (c >> 1) - 1; }
B3C_HD int dbase(int c) { return c < 4 ? c + 1 : ((2 + (c & 1)) << ((c >> 1) - 1)) + 1; }

B3C_HD int floor_log2(uint32_t v) {
    int r = 0;
    while (v >>= 1) ++r;
    return r;
}

// length 3..258 -> index of its length code (symbol 257 + index)
B3C_HD int len_code(int len) {
    if (len == MAX_MATCH) return 28;
    const int l = len - 3;
    if (l < 8) return l;
    const int nb = floor_log2((uint32_t)l);
    return 4 * (nb - 1) + ((l >> (nb - 2)) & 3);
}

// distance 1..32768 -> distance code
B3C_HD int dist_code(int dist) {
    if (dist <= 4) return dist - 1;
    const int d = dist - 1, nb = floor_log2((uint32_t)d);
    return 2 * nb + ((d >> (nb - 1)) & 1);
}

// Code lengths of at most `limit` bits for freq[0, n) (n <= LCODES); a symbol of zero frequency gets no code.  When
// fewer than two symbols occur, the lowest unused ones are added with weight one, so every code is complete (zlib's
// deflate does the same: inflaters refuse an empty distance code, and a one-code tree needs a second leaf).
B3C_HD void huff_lengths(const uint32_t *freq, int n, int limit, uint8_t *len) {
    uint16_t sym[LCODES];
    int32_t A[LCODES];
    int m = 0;
    for (int s = 0; s < n; ++s) {
        len[s] = 0;
        if (freq[s]) sym[m++] = (uint16_t)s;
    }
    for (int s = 0; m < 2 && s < n; ++s)
        if (!freq[s]) {
            int k = m++;                                  // keep sym[] in symbol order
            while (k > 0 && sym[k - 1] > s) {
                sym[k] = sym[k - 1];
                --k;
            }
            sym[k] = (uint16_t)s;
        }
    // sort by (weight, symbol): insertion sort, stable on the symbol order
    for (int k = 0; k < m; ++k) A[k] = freq[sym[k]] ? (int32_t)freq[sym[k]] : 1;
    for (int k = 1; k < m; ++k) {
        const int32_t w = A[k];
        const uint16_t s = sym[k];
        int j = k;
        while (j > 0 && A[j - 1] > w) {
            A[j] = A[j - 1];
            sym[j] = sym[j - 1];
            --j;
        }
        A[j] = w;
        sym[j] = s;
    }
    // Moffat and Katajainen, "In-place calculation of minimum-redundancy codes" (1995): A[k] becomes the depth of
    // the k-th lightest leaf
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < m - 1; ++next) {
        if (leaf >= m || A[root] < A[leaf]) {
            A[next] = A[root];
            A[root++] = next;
        } else {
            A[next] = A[leaf++];
        }
        if (leaf >= m || (root < next && A[root] < A[leaf])) {
            A[next] += A[root];
            A[root++] = next;
        } else {
            A[next] += A[leaf++];
        }
    }
    A[m - 2] = 0;
    for (int next = m - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
    int avbl = 1, used = 0, dpth = 0;
    root = m - 2;
    int next = m - 1;
    while (avbl > 0) {
        while (root >= 0 && A[root] == dpth) {
            ++used;
            --root;
        }
        while (avbl > used) {
            A[next--] = dpth;
            --avbl;
        }
        avbl = 2 * used;
        ++dpth;
        used = 0;
    }
    // depths past the limit: clamp, then restore the Kraft sum one leaf at a time (miniz)
    int cnt[b3c_inflate::MAXBITS + 1];
    for (int d = 0; d <= limit; ++d) cnt[d] = 0;
    for (int k = 0; k < m; ++k) cnt[A[k] > limit ? limit : A[k]]++;
    uint32_t total = 0;
    for (int d = 1; d <= limit; ++d) total += (uint32_t)cnt[d] << (limit - d);
    while (total > (1u << limit)) {
        cnt[limit]--;
        for (int d = limit - 1; d > 0; --d)
            if (cnt[d]) {
                cnt[d]--;
                cnt[d + 1] += 2;
                break;
            }
        total--;
    }
    // the heaviest symbols take the shortest codes
    int k = m - 1;
    for (int d = 1; d <= limit; ++d)
        for (int c = 0; c < cnt[d]; ++c) len[sym[k--]] = (uint8_t)d;
}

// canonical codes of the lengths, bit-reversed for the LSB-first bit order of deflate
B3C_HD void canonical(const uint8_t *len, int n, uint16_t *code) {
    uint16_t cnt[16], next[16];
    for (int b = 0; b < 16; ++b) cnt[b] = 0;
    for (int s = 0; s < n; ++s) cnt[len[s]]++;
    cnt[0] = 0;
    uint32_t c = 0;
    for (int b = 1; b < 16; ++b) {
        c = (c + cnt[b - 1]) << 1;
        next[b] = (uint16_t)c;
    }
    for (int s = 0; s < n; ++s) {
        code[s] = 0;
        if (!len[s]) continue;
        uint32_t v = next[len[s]]++, r = 0;
        for (int b = 0; b < len[s]; ++b) {
            r = (r << 1) | (v & 1);
            v >>= 1;
        }
        code[s] = (uint16_t)r;
    }
}

// a dynamic block: codes, the run-length coded lengths and the header's size
struct Dyn {
    uint8_t llen[LCODES], dlen[DCODES], cllen[BLCODES];
    uint16_t lcode[LCODES], dcode[DCODES], clcode[BLCODES];
    uint8_t rle[MAX_RLE], rle_x[MAX_RLE];
    int32_t hlit, hdist, hclen, nrle;
    int64_t header_bits;
};

B3C_HD int rle_extra_bits(int sym) { return sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0; }

// Plans the dynamic block for the histograms (lfreq[256], the end-of-block code, must be 1); returns its size in bits.
B3C_HD int64_t plan_dynamic(const uint32_t *lfreq, const uint32_t *dfreq, Dyn &D) {
    huff_lengths(lfreq, LCODES, b3c_inflate::MAXBITS, D.llen);
    huff_lengths(dfreq, DCODES, b3c_inflate::MAXBITS, D.dlen);
    canonical(D.llen, LCODES, D.lcode);
    canonical(D.dlen, DCODES, D.dcode);
    D.hlit = LCODES;
    while (D.hlit > 257 && D.llen[D.hlit - 1] == 0) --D.hlit;
    D.hdist = DCODES;
    while (D.hdist > 1 && D.dlen[D.hdist - 1] == 0) --D.hdist;
    // run-length code the lengths (one sequence: a run may cross from the literal/length into the distance lengths)
    const int total = D.hlit + D.hdist;
    uint32_t clfreq[BLCODES];
    for (int s = 0; s < BLCODES; ++s) clfreq[s] = 0;
    D.nrle = 0;
    auto push = [&](int sym, int x) {
        D.rle[D.nrle] = (uint8_t)sym;
        D.rle_x[D.nrle] = (uint8_t)x;
        D.nrle++;
        clfreq[sym]++;
    };
    for (int k = 0; k < total;) {
        const int v = k < D.hlit ? D.llen[k] : D.dlen[k - D.hlit];
        int r = 1;
        while (k + r < total && (k + r < D.hlit ? D.llen[k + r] : D.dlen[k + r - D.hlit]) == v) ++r;
        k += r;
        if (v == 0) {
            while (r >= 11) {
                const int t = r < 138 ? r : 138;
                push(18, t - 11);
                r -= t;
            }
            if (r >= 3) {
                push(17, r - 3);
                r = 0;
            }
            while (r-- > 0) push(0, 0);
        } else {
            push(v, 0);
            --r;
            while (r >= 3) {
                const int t = r < 6 ? r : 6;
                push(16, t - 3);
                r -= t;
            }
            while (r-- > 0) push(v, 0);
        }
    }
    huff_lengths(clfreq, BLCODES, 7, D.cllen);
    canonical(D.cllen, BLCODES, D.clcode);
    const uint8_t ORDER[BLCODES] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    D.hclen = BLCODES;
    while (D.hclen > 4 && D.cllen[ORDER[D.hclen - 1]] == 0) --D.hclen;
    int64_t bits = 3 + 5 + 5 + 4 + 3 * D.hclen;
    for (int k = 0; k < D.nrle; ++k) bits += D.cllen[D.rle[k]] + rle_extra_bits(D.rle[k]);
    D.header_bits = bits;
    for (int s = 0; s < LCODES; ++s) bits += (int64_t)lfreq[s] * D.llen[s];
    for (int c = 0; c < 29; ++c) bits += (int64_t)lfreq[257 + c] * lext(c);
    for (int c = 0; c < DCODES; ++c) bits += (int64_t)dfreq[c] * (D.dlen[c] + dext(c));
    return bits;
}

// the histogram entries of the token at i (tok[i] & TOKEN set); dist[i] is its match distance
B3C_HD int token_lsym(const uint8_t *in, const uint16_t *tok, int i) {
    const int l = tok[i] & 0x7fff;
    return l ? 257 + len_code(l) : in[i];
}

// bits of the token at i under the planned codes
B3C_HD int token_bits(const Dyn &D, const uint8_t *in, const uint16_t *tok, const uint16_t *dist, int i) {
    const int l = tok[i] & 0x7fff;
    if (!l) return D.llen[in[i]];
    const int lc = len_code(l), dc = dist_code(dist[i]);
    return D.llen[257 + lc] + lext(lc) + D.dlen[dc] + dext(dc);
}

// LSB-first bits into zeroed 32-bit little-endian words; on the device the words are OR-ed atomically, so that
// threads whose bit ranges share a word can write concurrently
struct BitWriter {
    uint32_t *words;
    int64_t w;
    uint64_t acc;
    int nacc;
    B3C_HD void begin(uint32_t *out, int64_t bit) {
        words = out;
        w = bit >> 5;
        nacc = (int)(bit & 31);
        acc = 0;
    }
    B3C_HD void store(int64_t idx, uint32_t v) {
#ifdef __CUDA_ARCH__
        if (v) atomicOr(words + idx, v);
#else
        words[idx] |= v;
#endif
    }
    B3C_HD void put(uint32_t v, int nb) {             // nb <= 16
        acc |= (uint64_t)v << nacc;
        nacc += nb;
        if (nacc >= 32) {
            store(w++, (uint32_t)acc);
            acc >>= 32;
            nacc -= 32;
        }
    }
    B3C_HD void end() {
        if (nacc > 0) store(w, (uint32_t)acc);
    }
};

B3C_HD void put_header(BitWriter &bw, const Dyn &D) {
    bw.put(1, 1);                                     // BFINAL
    bw.put(2, 2);                                     // BTYPE 10: dynamic codes
    bw.put((uint32_t)(D.hlit - 257), 5);
    bw.put((uint32_t)(D.hdist - 1), 5);
    bw.put((uint32_t)(D.hclen - 4), 4);
    const uint8_t ORDER[BLCODES] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (int k = 0; k < D.hclen; ++k) bw.put(D.cllen[ORDER[k]], 3);
    for (int k = 0; k < D.nrle; ++k) {
        const int s = D.rle[k];
        bw.put(D.clcode[s], D.cllen[s]);
        if (s >= 16) bw.put(D.rle_x[k], rle_extra_bits(s));
    }
}

B3C_HD void put_token(BitWriter &bw, const Dyn &D, const uint8_t *in, const uint16_t *tok, const uint16_t *dist, int i) {
    const int l = tok[i] & 0x7fff;
    if (!l) {
        bw.put(D.lcode[in[i]], D.llen[in[i]]);
        return;
    }
    const int lc = len_code(l), dc = dist_code(dist[i]);
    bw.put(D.lcode[257 + lc], D.llen[257 + lc]);
    if (lext(lc)) bw.put((uint32_t)(l - lbase(lc)), lext(lc));
    bw.put(D.dcode[dc], D.dlen[dc]);
    if (dext(dc)) bw.put((uint32_t)(dist[i] - dbase(dc)), dext(dc));
}

// a dynamic block is used when it is shorter than the stored block
B3C_HD bool use_stored(int64_t dyn_bits, int n) { return (dyn_bits + 7) / 8 >= (int64_t)n + STORED_OVERHEAD; }

B3C_HD void put_stored_head(uint8_t *p, int n) {
    p[0] = 1;                                         // BFINAL, BTYPE 00, padding to the byte
    p[1] = (uint8_t)n;
    p[2] = (uint8_t)(n >> 8);
    p[3] = (uint8_t)~n;
    p[4] = (uint8_t)(~n >> 8);
}

// the BGZF header (member_bytes = the whole member) and the trailer
B3C_HD void put_member_header(uint8_t *m, int member_bytes) {
    const uint8_t h[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    for (int k = 0; k < 16; ++k) m[k] = h[k];
    m[16] = (uint8_t)(member_bytes - 1);
    m[17] = (uint8_t)((member_bytes - 1) >> 8);
}

B3C_HD void put_u32(uint8_t *p, uint32_t v) {
    p[0] = (uint8_t)v;
    p[1] = (uint8_t)(v >> 8);
    p[2] = (uint8_t)(v >> 16);
    p[3] = (uint8_t)(v >> 24);
}

#ifndef __CUDA_ARCH__
// serial scratch of deflate_member
struct Scratch {
    uint16_t head[HASH_SIZE];
    uint16_t prev[MEMBER_INPUT], tok[MEMBER_INPUT], dist[MEMBER_INPUT];
    uint32_t words[MEMBER_MAX / 4];
    uint32_t crc_table[256];
    Dyn D;
};

// One member of in[0, n) (n <= MEMBER_INPUT) into out[0, MEMBER_MAX); returns its length.  The reference the device
// encoder is compared with, byte for byte.
inline int deflate_member(const uint8_t *in, int n, uint8_t *out, Scratch &S) {
    for (int h = 0; h < HASH_SIZE; ++h) S.head[h] = NONE;
    for (int i = 0; i < n; ++i) {
        if (i + MIN_MATCH <= n) {
            const uint32_t h = hash3(in + i);
            S.prev[i] = S.head[h];
            S.head[h] = (uint16_t)i;
        } else {
            S.prev[i] = NONE;
        }
    }
    for (int i = 0; i < n; ++i) {
        int d;
        S.tok[i] = (uint16_t)find_match(in, n, S.prev, i, &d);
        S.dist[i] = (uint16_t)d;
    }
    parse(S.tok, n);
    uint32_t lfreq[LCODES] = {0}, dfreq[DCODES] = {0};
    for (int i = 0; i < n; ++i)
        if (S.tok[i] & TOKEN) {
            lfreq[token_lsym(in, S.tok, i)]++;
            if (S.tok[i] & 0x7fff) dfreq[dist_code(S.dist[i])]++;
        }
    lfreq[256] = 1;
    const int64_t bits = plan_dynamic(lfreq, dfreq, S.D);
    uint8_t *payload = out + HEADER_BYTES;
    int plen;
    if (use_stored(bits, n)) {
        put_stored_head(payload, n);
        for (int i = 0; i < n; ++i) payload[STORED_OVERHEAD + i] = in[i];
        plen = n + STORED_OVERHEAD;
    } else {
        plen = (int)((bits + 7) / 8);
        for (int k = 0; k < (plen + 3) / 4; ++k) S.words[k] = 0;
        BitWriter bw;
        bw.begin(S.words, 0);
        put_header(bw, S.D);
        for (int i = 0; i < n; ++i)
            if (S.tok[i] & TOKEN) put_token(bw, S.D, in, S.tok, S.dist, i);
        bw.put(S.D.lcode[256], S.D.llen[256]);
        bw.end();
        for (int k = 0; k < plen; ++k) payload[k] = (uint8_t)(S.words[k >> 2] >> (8 * (k & 3)));
    }
    const int total = HEADER_BYTES + plen + TRAILER_BYTES;
    put_member_header(out, total);
    b3c_inflate::crc32_table(S.crc_table);
    put_u32(out + HEADER_BYTES + plen, b3c_inflate::crc32_update(S.crc_table, 0, in, n));
    put_u32(out + HEADER_BYTES + plen + 4, (uint32_t)n);
    return total;
}
#endif

}  // namespace b3c_deflate
