// bin3c_io, part 1: name-sorted BAM -> reference table + packed pair records (include/bin3c_io.h).
//
// The step BEFORE the contact-map hot path (SURVEY.md 8f-1).  Replaces what the reference does with
// pysam: AlignmentFile + header checks (contact_map.py:534-545), next_informative (:624-629), the
// pairing loop (:720-731), the matchers (:612-622) and the min_insert filter (:761-766).
//
// Shape: a reader thread walks the BGZF container (block headers carry the compressed size, the trailer
// the uncompressed size, so every block's place in the output is known before it is inflated), cuts it
// into batches of BATCH_BLOCKS blocks and hands the blocks of a batch to a pool of inflate threads (raw
// zlib inflate + CRC check).  Batches live in a ring of RING slots, so inflation runs up to two batches
// ahead of the parser.  The parser is the reference's sequential state machine, run by the caller's
// thread inside b3c_bam_read_pairs: it needs only a few fixed fields of each alignment, so it never
// decodes sequence, qualities or tags.
#include <zlib.h>

#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/bin3c_io.h"
#include "io_common.h"

namespace b3cio {
thread_local char t_err[512] = "";

void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}
}  // namespace b3cio

namespace {
using b3cio::set_err;

constexpr int BATCH_BLOCKS = 256;          // <= 16 MiB of alignments per batch
constexpr int RING = 3;
constexpr uint32_t BAD_TID = 0x7fffffffu;

inline uint16_t rd16(const uint8_t *p) { return (uint16_t)(p[0] | (p[1] << 8)); }
inline uint32_t rd32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

struct Block {
    size_t c_off, c_len;                   // deflate payload inside Batch::comp
    size_t u_off;                          // where the block's bytes go inside Batch::out
    uint32_t isize, crc;
};

struct Batch {
    std::vector<uint8_t> comp, out;
    std::vector<Block> blocks;
    std::atomic<int> next{0};              // next block to inflate
    int done = 0;                          // blocks inflated                          (under mu)
    int active = 0;                        // workers currently drawing from it        (under mu)
    int state = 0;                         // 0 free, 1 being inflated, 2 ready        (under mu)
    bool last = false;                     // end of file follows this batch
    int err = 0;
    std::string err_msg;
};

}  // namespace

struct b3c_bam {
    FILE *fp = nullptr;
    std::string path;
    // pipeline
    Batch ring[RING];
    std::mutex mu;
    std::condition_variable cv_work, cv_ready, cv_free;
    std::vector<std::thread> workers;
    std::thread reader;
    bool stop = false;
    int inflating = -1;                    // ring slot the workers draw blocks from, -1 none
    std::atomic<int64_t> n_blocks{0}, c_bytes{0}, u_bytes{0};     // written by the reader thread, read by b3c_bam_stats
    // stream cursor of the parser
    int cur = 0;                           // ring slot being parsed
    bool cur_held = false;
    size_t pos = 0;
    bool eof = false;
    std::vector<uint8_t> carry;            // a record that straddles two batches is assembled here
    // header
    std::string text;
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    int64_t data_off = 0;                  // uncompressed stream offset of the first alignment record
    // filter
    int32_t min_mapq = 0, strong = 0, min_insert = 0;
    std::vector<int32_t> tid2idx;
    // extent map (contact_map.py:779-788): bins per sequence
    bool extent = false;
    std::vector<int64_t> ext_first, ext_ptr, ext_edges;
    // tip-based map (contact_map.py:631-670): size of the sequence ends that count, 0 = whole sequences
    int64_t tip_size = 0;
    int64_t n_not_tip = 0;
    // pairing state (contact_map.py:720-731): the pending first mate
    bool have_r1 = false;
    std::string r1_name;
    int32_t r1_tid = 0, r1_pos = 0;
    int64_t r1_pos5 = 0;
    uint16_t r1_flag = 0;
    bool r1_match = false;
    bool started = false;
    int64_t n_aln = 0, n_inf = 0, n_pairs = 0, n_short = 0, n_orphan = 0;
    int status = 0;
};

namespace {

// ---- inflate pool ----------------------------------------------------------------------------------
// one z_stream per inflate thread, reset for every block (inflateInit2 allocates the window each time otherwise)
struct Inflater {
    z_stream zs;
    bool ok;
    Inflater() {
        memset(&zs, 0, sizeof(zs));
        ok = inflateInit2(&zs, -15) == Z_OK;
    }
    ~Inflater() {
        if (ok) inflateEnd(&zs);
    }
};

int inflate_block(Inflater &inf, const Batch &b, const Block &k, uint8_t *out, std::string *msg) {
    if (!inf.ok || inflateReset(&inf.zs) != Z_OK) {
        *msg = "inflateInit2 failed";
        return B3C_IO_ERR_FORMAT;
    }
    z_stream &zs = inf.zs;
    zs.next_in = const_cast<Bytef *>(b.comp.data() + k.c_off);
    zs.avail_in = (uInt)k.c_len;
    zs.next_out = out;
    zs.avail_out = k.isize;
    const int rc = inflate(&zs, Z_FINISH);
    const bool ok = (rc == Z_STREAM_END) && zs.total_out == k.isize;
    if (!ok) {
        *msg = "corrupt BGZF block (inflate)";
        return B3C_IO_ERR_FORMAT;
    }
    if (k.isize && (uint32_t)crc32(crc32(0L, Z_NULL, 0), out, k.isize) != k.crc) {
        *msg = "corrupt BGZF block (CRC mismatch)";
        return B3C_IO_ERR_FORMAT;
    }
    return 0;
}

void worker_main(b3c_bam *h) {
    Inflater inf;
    std::unique_lock<std::mutex> lk(h->mu);
    for (;;) {
        h->cv_work.wait(lk, [&] { return h->stop || h->inflating >= 0; });
        if (h->stop) return;
        const int slot = h->inflating;
        Batch &b = h->ring[slot];
        b.active += 1;                                 // the reader does not recycle a slot a worker still looks at
        lk.unlock();
        const int nb = (int)b.blocks.size();
        int mine = 0, err = 0;
        std::string msg;
        for (;;) {
            const int i = b.next.fetch_add(1);
            if (i >= nb) break;
            const Block &k = b.blocks[i];
            if (!err && k.isize) err = inflate_block(inf, b, k, b.out.data() + k.u_off, &msg);
            ++mine;
        }
        lk.lock();
        if (err && !b.err) {
            b.err = err;
            b.err_msg = msg;
        }
        b.done += mine;
        b.active -= 1;
        if (h->inflating == slot) h->inflating = -1;   // every block has been handed out
        if (b.done == nb && b.state == 1) {
            b.state = 2;
            h->cv_ready.notify_all();
        }
        h->cv_free.notify_all();
    }
}

// read one BGZF block header + payload into the batch; returns 1 ok, 0 clean EOF, <0 error
int read_block(b3c_bam *h, Batch &b, std::string *msg) {
    uint8_t hd[12];
    const size_t got = fread(hd, 1, 12, h->fp);
    if (got == 0) return 0;
    if (got != 12 || hd[0] != 0x1f || hd[1] != 0x8b || hd[2] != 8 || !(hd[3] & 4)) {
        *msg = "not a BGZF file (bad gzip member header)";
        return B3C_IO_ERR_FORMAT;
    }
    const int xlen = rd16(hd + 10);
    uint8_t extra[65536];
    if ((int)fread(extra, 1, xlen, h->fp) != xlen) {
        *msg = "truncated BGZF block";
        return B3C_IO_ERR_FORMAT;
    }
    int bsize = -1;
    for (int o = 0; o + 4 <= xlen;) {
        const int slen = rd16(extra + o + 2);
        if (extra[o] == 'B' && extra[o + 1] == 'C' && slen == 2 && o + 6 <= xlen) bsize = rd16(extra + o + 4);
        o += 4 + slen;
    }
    const long payload = (long)bsize + 1 - 12 - xlen - 8;
    if (bsize < 0 || payload < 0) {
        *msg = "not a BGZF file (no BC subfield)";
        return B3C_IO_ERR_FORMAT;
    }
    Block k;
    k.c_off = b.comp.size();
    k.c_len = (size_t)payload;
    b.comp.resize(k.c_off + payload + 8);
    if (fread(b.comp.data() + k.c_off, 1, payload + 8, h->fp) != (size_t)payload + 8) {
        *msg = "truncated BGZF block";
        return B3C_IO_ERR_FORMAT;
    }
    k.crc = rd32(b.comp.data() + k.c_off + payload);
    k.isize = rd32(b.comp.data() + k.c_off + payload + 4);
    if (k.isize > 65536) {
        *msg = "corrupt BGZF block (ISIZE > 64 KiB)";
        return B3C_IO_ERR_FORMAT;
    }
    b.comp.resize(k.c_off + payload);
    k.u_off = b.out.size();
    b.out.resize(k.u_off + k.isize);
    b.blocks.push_back(k);
    h->c_bytes += bsize + 1;
    h->u_bytes += k.isize;
    h->n_blocks += 1;
    return 1;
}

void reader_main(b3c_bam *h) {
    int slot = 0;
    for (;;) {
        Batch &b = h->ring[slot];
        {
            std::unique_lock<std::mutex> lk(h->mu);
            h->cv_free.wait(lk, [&] { return h->stop || (b.state == 0 && b.active == 0); });
            if (h->stop) return;
        }
        b.comp.clear();
        b.out.clear();
        b.blocks.clear();
        b.next.store(0);
        b.done = 0;
        b.err = 0;
        b.last = false;
        std::string msg;
        int rc = 1;
        while ((int)b.blocks.size() < BATCH_BLOCKS) {
            rc = read_block(h, b, &msg);
            if (rc <= 0) break;
        }
        if (rc <= 0) b.last = true;
        if (rc < 0) {
            b.err = rc;
            b.err_msg = msg;
        }
        {
            std::unique_lock<std::mutex> lk(h->mu);
            // one batch is handed out at a time: wait until the workers have drawn every block of the previous one
            h->cv_free.wait(lk, [&] { return h->stop || h->inflating < 0; });
            if (h->stop) return;
            if (b.blocks.empty()) {
                b.state = 2;
                h->cv_ready.notify_all();
            } else {
                b.state = 1;
                h->inflating = slot;
                h->cv_work.notify_all();
            }
        }
        if (b.last) return;
        slot = (slot + 1) % RING;
    }
}

// ---- the parser's view: a byte stream over the ready batches -----------------------------------------
// make batch `cur` available (blocks until it has been inflated); false at end of file or on error
bool acquire(b3c_bam *h) {
    if (h->cur_held) return true;
    if (h->eof) return false;
    Batch &b = h->ring[h->cur];
    std::unique_lock<std::mutex> lk(h->mu);
    h->cv_ready.wait(lk, [&] { return b.state == 2; });
    if (b.err) {
        h->status = b.err;
        set_err("%s: %s", h->path.c_str(), b.err_msg.c_str());
        h->eof = true;
        return false;
    }
    h->cur_held = true;
    h->pos = 0;
    return true;
}

void release(b3c_bam *h) {
    Batch &b = h->ring[h->cur];
    const bool last = b.last;
    {
        std::unique_lock<std::mutex> lk(h->mu);
        b.state = 0;
        h->cv_free.notify_all();
    }
    h->cur_held = false;
    if (last) h->eof = true;
    else h->cur = (h->cur + 1) % RING;
}

// n contiguous bytes at the cursor (consumed), or nullptr at end of file.  *partial is set when the file
// ends inside the requested span.
const uint8_t *take(b3c_bam *h, size_t n, bool *partial) {
    *partial = false;
    for (;;) {
        if (!acquire(h)) return nullptr;
        Batch &b = h->ring[h->cur];
        const size_t avail = b.out.size() - h->pos;
        if (avail >= n) {
            const uint8_t *p = b.out.data() + h->pos;
            h->pos += n;
            return p;
        }
        if (avail == 0) {
            release(h);
            continue;
        }
        // straddles batches: assemble in the carry buffer
        h->carry.assign(b.out.data() + h->pos, b.out.data() + b.out.size());
        release(h);
        while (h->carry.size() < n) {
            if (!acquire(h)) {
                *partial = true;
                return nullptr;
            }
            Batch &c = h->ring[h->cur];
            const size_t want = n - h->carry.size(), have = c.out.size() - h->pos;
            const size_t m = want < have ? want : have;
            h->carry.insert(h->carry.end(), c.out.data() + h->pos, c.out.data() + h->pos + m);
            h->pos += m;
            if (h->pos == c.out.size() && h->carry.size() < n) release(h);
        }
        return h->carry.data();
    }
}

int fail_format(b3c_bam *h, const char *what) {
    if (h->status == 0) {
        h->status = B3C_IO_ERR_FORMAT;
        set_err("%s: %s", h->path.c_str(), what);
    }
    return h->status;
}

int parse_header(b3c_bam *h, int require_queryname) {
    bool part;
    const uint8_t *p = take(h, 8, &part);
    if (!p || memcmp(p, "BAM\1", 4) != 0) return fail_format(h, "not a BAM file (bad magic)");
    const uint32_t l_text = rd32(p + 4);
    int64_t off = 8 + (int64_t)l_text + 4;
    if (l_text) {
        p = take(h, l_text, &part);
        if (!p) return fail_format(h, "truncated BAM header");
        h->text.assign((const char *)p, l_text);
        const size_t z = h->text.find('\0');
        if (z != std::string::npos) h->text.resize(z);
    }
    p = take(h, 4, &part);
    if (!p) return fail_format(h, "truncated BAM header");
    const int32_t n_ref = (int32_t)rd32(p);
    if (n_ref < 0) return fail_format(h, "negative reference count");
    h->ref_names.reserve(n_ref);
    h->ref_lens.reserve(n_ref);
    for (int32_t i = 0; i < n_ref; ++i) {
        p = take(h, 4, &part);
        if (!p) return fail_format(h, "truncated reference table");
        const uint32_t l_name = rd32(p);
        p = take(h, (size_t)l_name + 4, &part);
        if (!p || l_name == 0) return fail_format(h, "truncated reference table");
        h->ref_names.emplace_back((const char *)p, strnlen((const char *)p, l_name));
        h->ref_lens.push_back((int32_t)rd32(p + l_name));
        off += 4 + (int64_t)l_name + 4;
    }
    h->data_off = off;
    if (require_queryname) {
        // bam.header['HD']['SO'] == 'queryname' (contact_map.py:537-538)
        bool ok = false;
        size_t a = 0;
        while (a < h->text.size()) {
            size_t e = h->text.find('\n', a);
            if (e == std::string::npos) e = h->text.size();
            if (e - a >= 3 && h->text.compare(a, 3, "@HD") == 0) {
                size_t f = a;
                while (f < e) {
                    size_t t = h->text.find('\t', f);
                    if (t == std::string::npos || t > e) t = e;
                    if (t - f == 12 && h->text.compare(f, 12, "SO:queryname") == 0) ok = true;
                    f = t + 1;
                }
            }
            a = e + 1;
        }
        if (!ok) {
            h->status = B3C_IO_ERR_SORT;
            set_err("%s: BAM file must be sorted by read name", h->path.c_str());
            return h->status;
        }
    }
    return 0;
}

struct Aln {
    int32_t tid, pos;
    int64_t pos5;            // 5'-end position: pos, or pos + reference span for a reverse read (contact_map.py:757-758)
    uint16_t flag;
    bool match;
    const char *name;
    size_t name_len;
};

// next alignment of the stream: 1 ok, 0 end of file, <0 error
int next_alignment(b3c_bam *h, Aln *a) {
    bool part;
    const uint8_t *p = take(h, 4, &part);
    if (!p) return (part || h->status) ? fail_format(h, "truncated alignment record") : 0;
    const uint32_t bs = rd32(p);
    if (bs < 32) return fail_format(h, "alignment record shorter than its fixed fields");
    p = take(h, bs, &part);
    if (!p) return fail_format(h, "truncated alignment record");
    const uint32_t l_name = p[8], mapq = p[9], n_cig = rd16(p + 12);
    a->tid = (int32_t)rd32(p);
    a->pos = (int32_t)rd32(p + 4);
    a->flag = rd16(p + 14);
    if (32 + (size_t)l_name + 4 * (size_t)n_cig > bs) return fail_format(h, "alignment record overruns its block size");
    a->name = (const char *)p + 32;
    a->name_len = l_name ? strnlen(a->name, l_name) : 0;
    // the CIGAR: in the record, or -- beyond 65535 operations -- in the CG:B,I tag behind the placeholder
    // <l_seq>S<ref span>N (SAM specification, section 4.2.2); htslib / pysam hand the tag's operations to the caller
    const uint8_t *cg = p + 32 + l_name;
    uint32_t n_ops = n_cig;
    const uint32_t l_seq = rd32(p + 16);
    if (n_cig == 2 && (rd32(cg) & 0xf) == 4 && (rd32(cg) >> 4) == l_seq && (rd32(cg + 4) & 0xf) == 3) {
        const uint8_t *aux = cg + 8 + ((size_t)l_seq + 1) / 2 + l_seq, *end = p + bs;
        while (aux + 3 <= end) {
            const uint8_t t = aux[2];
            const uint8_t *v = aux + 3;
            size_t len = 0;
            auto size_of = [](uint8_t c) -> size_t {
                return (c == 'A' || c == 'c' || c == 'C') ? 1 : (c == 's' || c == 'S') ? 2 : (c == 'i' || c == 'I' || c == 'f') ? 4 : 0;
            };
            if (t == 'Z' || t == 'H') {
                const void *z = memchr(v, 0, (size_t)(end - v));
                if (!z) return fail_format(h, "unterminated string tag");
                len = (size_t)((const uint8_t *)z - v) + 1;
            } else if (t == 'B') {
                if (v + 5 > end) return fail_format(h, "truncated array tag");
                const size_t es = size_of(v[0]), cnt = rd32(v + 1);
                if (es == 0 || v + 5 + es * cnt > end) return fail_format(h, "malformed array tag");
                if (aux[0] == 'C' && aux[1] == 'G' && v[0] == 'I' && cnt > 0) {
                    cg = v + 5;
                    n_ops = (uint32_t)cnt;
                    break;
                }
                len = 5 + es * cnt;
            } else {
                len = size_of(t);
                if (len == 0) return fail_format(h, "unknown tag type");
            }
            aux = v + len;
        }
    }
    // _simple_match / _strong_match (contact_map.py:612-619)
    bool m = (int32_t)mapq >= h->min_mapq;
    if (m && h->strong > 0) {
        if (n_ops == 0) {
            m = false;                                               // r.cigarstring is None
        } else {
            const uint32_t op = rd32(cg + 4 * ((a->flag & 0x10) ? (n_ops - 1) : 0));
            m = (op & 0xf) == 0 && (int32_t)(op >> 4) >= h->strong;
        }
    }
    a->match = m;
    a->pos5 = a->pos;
    if ((h->extent || h->tip_size > 0) && (a->flag & 0x10)) {
        // r.alen = pysam reference_length: the CIGAR operations that consume the reference (M, D, N, =, X).  A mapped
        // reverse read without a CIGAR has alen None in the reference, whose `r.pos + r.alen` then raises: an error
        // here too, not a silent span of zero.
        if (n_ops == 0 && !(a->flag & 0x4))
            return fail_format(h, "mapped reverse read without a CIGAR: its 5' end is undefined (extent / tip records)");
        int64_t span = 0;
        const uint32_t n_cig = n_ops;
        for (uint32_t k = 0; k < n_cig; ++k) {
            const uint32_t op = rd32(cg + 4 * k), t = op & 0xf;
            if (t == 0 || t == 2 || t == 3 || t == 7 || t == 8) span += op >> 4;
        }
        a->pos5 += span;
    }
    return 1;
}

}  // namespace

extern "C" {

int b3c_io_version(void) { return 100; }
const char *b3c_io_last_error(void) { return b3cio::t_err; }

int b3c_bam_open(const char *path, int32_t n_threads, int32_t require_queryname, b3c_bam **out) {
    if (!path || !out) {
        set_err("b3c_bam_open: null argument");
        return B3C_IO_ERR_ARG;
    }
    *out = nullptr;
    FILE *fp = fopen(path, "rb");
    if (!fp) {
        set_err("%s: cannot open", path);
        return B3C_IO_ERR_OPEN;
    }
    b3c_bam *h = new b3c_bam();
    h->fp = fp;
    h->path = path;
    setvbuf(fp, nullptr, _IOFBF, 1 << 22);
    if (n_threads <= 0) n_threads = (int32_t)std::thread::hardware_concurrency();
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 64) n_threads = 64;
    for (int i = 0; i < n_threads; ++i) h->workers.emplace_back(worker_main, h);
    h->reader = std::thread(reader_main, h);
    const int rc = parse_header(h, require_queryname);
    if (rc != 0) {
        b3c_bam_close(h);
        return rc;
    }
    *out = h;
    return 0;
}

void b3c_bam_close(b3c_bam *h) {
    if (!h) return;
    {
        std::unique_lock<std::mutex> lk(h->mu);
        h->stop = true;
        h->cv_work.notify_all();
        h->cv_free.notify_all();
        h->cv_ready.notify_all();
    }
    if (h->reader.joinable()) h->reader.join();
    for (auto &t : h->workers) t.join();
    if (h->fp) fclose(h->fp);
    delete h;
}

int32_t b3c_bam_n_refs(const b3c_bam *h) { return h ? (int32_t)h->ref_names.size() : B3C_IO_ERR_ARG; }

const char *b3c_bam_ref_name(const b3c_bam *h, int32_t tid) {
    if (!h || tid < 0 || tid >= (int32_t)h->ref_names.size()) return nullptr;
    return h->ref_names[tid].c_str();
}

int64_t b3c_bam_ref_lengths(const b3c_bam *h, int64_t *h_lengths, int32_t capacity) {
    if (!h || (!h_lengths && capacity > 0)) return B3C_IO_ERR_ARG;
    const int64_t n = (int64_t)h->ref_lens.size();
    for (int64_t i = 0; i < n && i < capacity; ++i) h_lengths[i] = h->ref_lens[i];
    return n;
}

int64_t b3c_bam_header_text(const b3c_bam *h, char *h_text, int64_t capacity) {
    if (!h || (!h_text && capacity > 0)) return B3C_IO_ERR_ARG;
    const int64_t n = (int64_t)h->text.size();
    if (capacity > 0) {
        const int64_t m = n < capacity - 1 ? n : capacity - 1;
        memcpy(h_text, h->text.data(), m);
        h_text[m] = '\0';
    }
    return n;
}

int64_t b3c_bam_data_offset(const b3c_bam *h) { return h ? h->data_off : B3C_IO_ERR_ARG; }

int64_t b3c_bgzf_scan(const uint8_t *h_buf, int64_t n_bytes, int32_t at_eof, int64_t *h_offsets, int32_t *h_bsize,
                      int32_t *h_isize, int64_t capacity, int64_t *h_consumed) {
    if ((!h_buf && n_bytes > 0) || n_bytes < 0 || capacity < 0 || !h_consumed ||
        (capacity > 0 && (!h_offsets || !h_bsize || !h_isize))) {
        set_err("b3c_bgzf_scan: bad argument");
        return B3C_IO_ERR_ARG;
    }
    // the checks of read_block, on a buffer: a block cut off by the end of the buffer ends the scan, and is an error
    // only when the file ends there
    int64_t o = 0, n = 0;
    *h_consumed = 0;
    while (n < capacity && o < n_bytes) {
        const uint8_t *hd = h_buf + o;
        const int64_t left = n_bytes - o;
        if (left < 12) {
            if (!at_eof) break;
            set_err("not a BGZF file (bad gzip member header)");
            return B3C_IO_ERR_FORMAT;
        }
        if (hd[0] != 0x1f || hd[1] != 0x8b || hd[2] != 8 || !(hd[3] & 4)) {
            set_err("not a BGZF file (bad gzip member header)");
            return B3C_IO_ERR_FORMAT;
        }
        const int xlen = rd16(hd + 10);
        if (left < 12 + xlen) {
            if (!at_eof) break;
            set_err("truncated BGZF block");
            return B3C_IO_ERR_FORMAT;
        }
        int bsize = -1;
        for (int e = 0; e + 4 <= xlen;) {
            const int slen = rd16(hd + 12 + e + 2);
            if (hd[12 + e] == 'B' && hd[12 + e + 1] == 'C' && slen == 2 && e + 6 <= xlen) bsize = rd16(hd + 12 + e + 4);
            e += 4 + slen;
        }
        const long payload = (long)bsize + 1 - 12 - xlen - 8;
        if (bsize < 0 || payload < 0) {
            set_err("not a BGZF file (no BC subfield)");
            return B3C_IO_ERR_FORMAT;
        }
        if (left < (int64_t)bsize + 1) {
            if (!at_eof) break;
            set_err("truncated BGZF block");
            return B3C_IO_ERR_FORMAT;
        }
        const uint32_t isize = rd32(hd + bsize + 1 - 4);
        if (isize > 65536) {
            set_err("corrupt BGZF block (ISIZE > 64 KiB)");
            return B3C_IO_ERR_FORMAT;
        }
        h_offsets[n] = o;
        h_bsize[n] = bsize;
        h_isize[n] = (int32_t)isize;
        ++n;
        o += (int64_t)bsize + 1;
    }
    *h_consumed = o;
    return n;
}

int b3c_bam_set_filter(b3c_bam *h, int32_t min_mapq, int32_t strong, int32_t min_insert, const int32_t *h_tid2idx,
                       int32_t n_refs) {
    if (!h) return B3C_IO_ERR_ARG;
    if (h->started) {
        set_err("b3c_bam_set_filter: records have already been read");
        return B3C_IO_ERR_ARG;
    }
    if (min_insert > 0 && (!h_tid2idx || n_refs != (int32_t)h->ref_names.size())) {
        set_err("b3c_bam_set_filter: min_insert needs the tid -> index table of all %d references",
                (int)h->ref_names.size());
        return B3C_IO_ERR_ARG;
    }
    h->min_mapq = min_mapq;
    h->strong = strong < 0 ? 0 : strong;
    h->min_insert = min_insert < 0 ? 0 : min_insert;
    if (h_tid2idx) h->tid2idx.assign(h_tid2idx, h_tid2idx + n_refs);
    else if (!h->extent && h->tip_size <= 0) h->tid2idx.clear();      // the table of b3c_bam_set_extent / _set_tips is kept
    return 0;
}

static int64_t read_pairs_impl(b3c_bam *h, uint64_t *h_records, uint64_t *h_extent, int64_t capacity, uint8_t *h_tip10);

int64_t b3c_bam_read_pairs(b3c_bam *h, uint64_t *h_records, int64_t capacity) {
    return read_pairs_impl(h, h_records, nullptr, capacity, nullptr);
}

int b3c_bam_set_tips(b3c_bam *h, int64_t tip_size, const int32_t *h_tid2idx, int32_t n_refs) {
    if (!h || tip_size <= 0 || !h_tid2idx || n_refs != (int32_t)h->ref_names.size()) {
        set_err("b3c_bam_set_tips: needs a positive tip size and the tid -> index table of all references");
        return B3C_IO_ERR_ARG;
    }
    if (h->started || h->extent) {
        set_err("b3c_bam_set_tips: records have already been read, or extent records are on (the two do not combine)");
        return B3C_IO_ERR_ARG;
    }
    if (n_refs >= (1 << 30)) {
        set_err("b3c_bam_set_tips: doubled reference ids do not fit in 31 bits");
        return B3C_IO_ERR_ARG;
    }
    h->tid2idx.assign(h_tid2idx, h_tid2idx + n_refs);
    h->tip_size = tip_size;
    return 0;
}

int64_t b3c_bam_read_pairs_tips(b3c_bam *h, uint64_t *h_records, uint8_t *h_tip10, int64_t capacity) {
    if (!h || h->tip_size <= 0 || (!h_tip10 && capacity > 0)) {
        set_err("b3c_bam_read_pairs_tips: call b3c_bam_set_tips first");
        return B3C_IO_ERR_ARG;
    }
    return read_pairs_impl(h, h_records, nullptr, capacity, h_tip10);
}

int64_t b3c_bam_read_pairs_extent(b3c_bam *h, uint64_t *h_records, uint64_t *h_extent_records, int64_t capacity) {
    if (!h || !h->extent || (!h_extent_records && capacity > 0)) {
        set_err("b3c_bam_read_pairs_extent: call b3c_bam_set_extent first");
        return B3C_IO_ERR_ARG;
    }
    return read_pairs_impl(h, h_records, h_extent_records, capacity, nullptr);
}

int b3c_bam_set_extent(b3c_bam *h, const int32_t *h_tid2idx, int32_t n_refs, const int64_t *h_first_bin,
                       const int64_t *h_edge_ptr, const int64_t *h_upper_edges, int32_t n_seq) {
    if (!h || !h_tid2idx || !h_first_bin || !h_edge_ptr || !h_upper_edges || n_seq < 0 ||
        n_refs != (int32_t)h->ref_names.size()) {
        set_err("b3c_bam_set_extent: bad argument (the tid -> index table must cover all %d references)",
                h ? (int)h->ref_names.size() : 0);
        return B3C_IO_ERR_ARG;
    }
    if (h->started) {
        set_err("b3c_bam_set_extent: records have already been read");
        return B3C_IO_ERR_ARG;
    }
    for (int32_t t = 0; t < n_refs; ++t)
        if (h_tid2idx[t] >= n_seq) {
            set_err("b3c_bam_set_extent: index %d of reference %d is outside the %d sequences", h_tid2idx[t], t, n_seq);
            return B3C_IO_ERR_ARG;
        }
    for (int32_t i = 0; i < n_seq; ++i)
        if (h_edge_ptr[i + 1] <= h_edge_ptr[i] || h_first_bin[i] + (h_edge_ptr[i + 1] - h_edge_ptr[i]) >= 0x7fffffffll) {
            set_err("b3c_bam_set_extent: sequence %d has no bins, or bin numbers do not fit in 31 bits", i);
            return B3C_IO_ERR_ARG;
        }
    h->tid2idx.assign(h_tid2idx, h_tid2idx + n_refs);
    h->ext_first.assign(h_first_bin, h_first_bin + n_seq);
    h->ext_ptr.assign(h_edge_ptr, h_edge_ptr + n_seq + 1);
    h->ext_edges.assign(h_upper_edges, h_upper_edges + h_edge_ptr[n_seq]);
    h->extent = true;
    return 0;
}

// find_nearest_jit (contact_map.py:49-62): the bin whose upper edge is the first one >= x; past the end, the last
static uint64_t extent_bin(const b3c_bam *h, int32_t tid, int64_t x, int32_t n_refs) {
    if (tid < 0 || tid >= n_refs) return BAD_TID;
    const int32_t ix = h->tid2idx[tid];
    if (ix < 0) return BAD_TID;
    const int64_t lo = h->ext_ptr[ix], hi = h->ext_ptr[ix + 1];
    int64_t a = lo, b = hi;
    while (a < b) {
        const int64_t mid = (a + b) >> 1;
        if (h->ext_edges[mid] < x) a = mid + 1;
        else b = mid;
    }
    if (a == hi) a = hi - 1;
    return (uint64_t)(h->ext_first[ix] + (a - lo));
}

// _on_tip_withlocs (contact_map.py:631-670), one mate: which end of a sequence of length `len` the position p falls in
// (0 = head, 1 = tail), or -1.  Ends of `tip` bp when they do not overlap (len > 2 tip); otherwise the nearer end, and
// neither when p is exactly in the middle.
static int tip_of(int64_t p, int64_t len, int64_t tip) {
    if (len > 2 * tip) {
        if (p < tip) return 0;
        if (p > len - tip) return 1;
        return -1;
    }
    if (p < len - p) return 0;
    if (len - p < p) return 1;
    return -1;
}

static int64_t read_pairs_impl(b3c_bam *h, uint64_t *h_records, uint64_t *h_extent, int64_t capacity, uint8_t *h_tip10) {
    if (!h || (!h_records && capacity > 0) || capacity < 0) {
        set_err("b3c_bam_read_pairs: bad argument");
        return B3C_IO_ERR_ARG;
    }
    if (h->status) return h->status;
    h->started = true;
    const int32_t n_refs = (int32_t)h->ref_names.size();
    int64_t n = 0;
    while (n < capacity) {
        Aln a = {0, 0, 0, 0, false, nullptr, 0};
        const int rc = next_alignment(h, &a);
        if (rc < 0) return rc;
        if (rc == 0) {
            if (h->have_r1) {                                        // StopIteration with a mate pending (:730-731)
                h->n_orphan += 1;
                h->have_r1 = false;
            }
            break;
        }
        h->n_aln += 1;
        if (a.flag & (0x4 | 0x100 | 0x800)) continue;                // next_informative (:628)
        h->n_inf += 1;
        if (!h->have_r1 || h->r1_name.size() != a.name_len || memcmp(h->r1_name.data(), a.name, a.name_len) != 0) {
            if (h->have_r1) h->n_orphan += 1;                        // r1 = r2 (:729)
            h->have_r1 = true;
            h->r1_name.assign(a.name, a.name_len);
            h->r1_tid = a.tid;
            h->r1_pos = a.pos;
            h->r1_pos5 = a.pos5;
            h->r1_flag = a.flag;
            h->r1_match = a.match;
            continue;
        }
        // a pair: r1 is the pending record, r2 this one
        h->have_r1 = false;
        h->n_pairs += 1;
        const bool in1 = h->r1_tid >= 0 && h->r1_tid < n_refs, in2 = a.tid >= 0 && a.tid < n_refs;
        const bool pass = h->r1_match && a.match;
        if (h->min_insert > 0 && pass && in1 && in2 && h->tid2idx[h->r1_tid] >= 0 && h->tid2idx[a.tid] >= 0) {
            // after the exclusion and matcher tests (:733-739): swap on r1.is_read2 (:746), then proper pairs whose
            // r2.pos - r1.pos is below the threshold are dropped (:761-766)
            const bool swap = (h->r1_flag & 0x80) != 0;
            const uint16_t f1 = swap ? a.flag : h->r1_flag;
            const int32_t p1 = swap ? a.pos : h->r1_pos, p2 = swap ? h->r1_pos : a.pos;
            if ((f1 & 0x2) && (int64_t)p2 - (int64_t)p1 < (int64_t)h->min_insert) {
                h->n_short += 1;
                continue;
            }
        }
        uint64_t t1 = in1 ? (uint32_t)h->r1_tid : BAD_TID, t2 = in2 ? (uint32_t)a.tid : BAD_TID;
        if (h->tip_size > 0) {
            // Tip records: reference ids become 2 * tid + tip.  A pair that passed the exclusion and matcher tests
            // (:733-739) is assigned tips from the 5' positions (:757-758, :791); when either mate lies in neither end it
            // is dropped here and counted not_tip (:792-794).  The reference orders a pair by internal index (:774-777);
            // the accumulator does the same with the doubled ids.  On ONE sequence the tensor element is
            // [tip(read 1), tip(read 2)] in read order (:746, no swap for ix1 == ix2): the (tail, head) pairs are marked
            // in h_tip10, because the symmetric accumulator merges them with the (head, tail) ones.
            if (h_tip10) h_tip10[n] = 0;
            if (pass && in1 && in2 && h->tid2idx[h->r1_tid] >= 0 && h->tid2idx[a.tid] >= 0) {
                const int k1 = tip_of(h->r1_pos5, h->ref_lens[h->r1_tid], h->tip_size);
                const int k2 = tip_of(a.pos5, h->ref_lens[a.tid], h->tip_size);
                if (k1 < 0 || k2 < 0) {
                    h->n_not_tip += 1;
                    continue;
                }
                t1 = 2 * t1 + (uint64_t)k1;
                t2 = 2 * t2 + (uint64_t)k2;
                if (h->r1_tid == a.tid && h_tip10) {
                    const bool swap = (h->r1_flag & 0x80) != 0;                     // r1.is_read2 (:746)
                    const int ka = swap ? k2 : k1, kb = swap ? k1 : k2;
                    h_tip10[n] = (ka == 1 && kb == 0) ? 1 : 0;
                }
            } else {
                t1 = in1 ? 2 * t1 : BAD_TID;                                        // counted by the accumulator as
                t2 = in2 ? 2 * t2 : BAD_TID;                                        // ref_excluded / poor_match
            }
        }
        if (h_extent) {
            const uint64_t b1 = extent_bin(h, h->r1_tid, h->r1_pos5, n_refs), b2 = extent_bin(h, a.tid, a.pos5, n_refs);
            h_extent[n] = b1 | ((uint64_t)(pass ? 1u : 0u) << 31) | (b2 << 32);
        }
        h_records[n++] = t1 | ((uint64_t)(pass ? 1u : 0u) << 31) | (t2 << 32);
    }
    return n;
}

int b3c_bam_stats(const b3c_bam *h, int64_t *h_stats, int32_t n_stats) {
    if (!h || !h_stats || n_stats < 0) return B3C_IO_ERR_ARG;
    const int64_t v[9] = {h->n_aln, h->n_inf, h->n_pairs, h->n_short, h->n_orphan, h->n_blocks.load(), h->c_bytes.load(),
                          h->u_bytes.load(), h->n_not_tip};
    for (int i = 0; i < n_stats && i < 9; ++i) h_stats[i] = v[i];
    return 0;
}

}  // extern "C"
