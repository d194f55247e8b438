// Host side of SURVEY.md section 8 (f1) and (f3) in native code, behind the C ABI (include/apples_b200.h):
//
//   apples_fasta_*   FASTA / FASTQ -> one byte matrix [n][stride] (pinned host memory when a CUDA device is there), with
//                    the record semantics and alphabet normalisation of apples/fasta2dic.py:4-72 (readfq + fasta2dic):
//                    name = header up to the first blank, multi-line sequences, optional '+' quality block, sequences
//                    upper-cased (or lower-case masked to '-' with -X), letters outside the alphabet -> '-'.
//                    The matrix is what apples_place_batch_bytes / apples_set_reference_bytes take.
//   apples_jplace_write   result arrays -> the jplace text `json.dumps(result, sort_keys=True, indent=4)` writes for the
//                    joined per-query records (run_apples.py:106-118, jutil.py:1-19), byte for byte: Python float repr,
//                    ensure_ascii string escapes, the "first record is kept even when unplaceable" quirk of join_jplace.
//                    apples_jplace_write_k: the same with the ranked records of --keep-at-most K in each "p" list.
//
// Both are multi-threaded (std::thread): at config 5 the queries are 5 GB of text and a million records.  No CUDA kernel
// is involved; cudaHostAlloc is used only to make the matrix directly DMA-able.
#include <algorithm>
#include <atomic>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cuda_runtime.h>

#include "../../include/apples_b200.h"

struct apples_fasta {
    int64_t n = 0, max_len = 0, stride = 0;
    bool uniform = true;
    bool pinned = false;
    uint8_t* matrix = nullptr;
    std::vector<int64_t> lengths;
    std::string names;               // NUL-terminated names, concatenated
    std::vector<int64_t> name_off;   // n + 1 offsets into `names`
    std::string err;
};

namespace {

struct Rec {
    const char* name;   // header text after '>' / '@'
    int64_t name_len;
    const char* seq;    // first sequence line
    const char* seq_end;  // end of the sequence block (start of the next header / '+' line / EOF)
    int64_t len = 0;    // residues (line breaks removed)
};

inline const char* line_end(const char* p, const char* end) {
    const char* q = (const char*)memchr(p, '\n', (size_t)(end - p));
    return q ? q : end;
}

// strip the line terminator the way the Python twin does (rstrip('\r\n'))
inline const char* rstrip_crlf(const char* b, const char* e) {
    while (e > b && (e[-1] == '\n' || e[-1] == '\r')) --e;
    return e;
}

void set_err(char* err, int errlen, const std::string& msg) {
    if (err && errlen > 0) {
        snprintf(err, (size_t)errlen, "%s", msg.c_str());
    }
}

}  // namespace

extern "C" {

int apples_fasta_open(const char* path, int prot_flag, int mask_flag, int n_threads, int want_pinned, apples_fasta** out,
                      char* err, int errlen) {
    if (!out || !path) return -1;
    *out = nullptr;
    int fd = open(path, O_RDONLY);
    if (fd < 0) {
        set_err(err, errlen, std::string("cannot open ") + path);
        return -2;
    }
    struct stat st;
    if (fstat(fd, &st) != 0) {
        close(fd);
        set_err(err, errlen, "fstat failed");
        return -2;
    }
    const size_t size = (size_t)st.st_size;
    const char* data = nullptr;
    if (size) {
        data = (const char*)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (data == MAP_FAILED) {
            close(fd);
            set_err(err, errlen, "mmap failed");
            return -2;
        }
        madvise((void*)data, size, MADV_SEQUENTIAL);
    }
    close(fd);
    const char* end = data + size;
    if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    n_threads = std::min(n_threads, 64);

    // ---- pass 1: record boundaries.  Parallel scan for the lines that start with '>', '@' or '+'.  A file without '@' and
    // '+' lines is plain FASTA: every '>' line starts a record, so the boundaries are known without a sequential state
    // machine (5 GB of queries at config 5).  Anything else (FASTQ) takes readfq's sequential state machine below.
    std::vector<Rec> recs;
    bool plain_fasta = true;
    {
        std::vector<std::vector<const char*>> heads((size_t)n_threads);
        std::vector<char> other((size_t)n_threads, 0);
        auto scan = [&](int t) {
            const size_t b = size * (size_t)t / (size_t)n_threads, e = size * (size_t)(t + 1) / (size_t)n_threads;
            const char* p = data + b;
            const char* pe = data + e;
            if (b > 0) {   // first line start at or after b
                const char* q = (const char*)memchr(p - 1, '\n', (size_t)(end - (p - 1)));
                p = q ? q + 1 : end;
            }
            while (p < pe) {
                const char c = *p;
                if (c == '>') heads[(size_t)t].push_back(p);
                else if (c == '@' || c == '+') other[(size_t)t] = 1;
                const char* q = (const char*)memchr(p, '\n', (size_t)(end - p));
                p = q ? q + 1 : end;
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < n_threads; ++t) th.emplace_back(scan, t);
        scan(0);
        for (auto& t : th) t.join();
        for (int t = 0; t < n_threads; ++t) plain_fasta = plain_fasta && !other[(size_t)t];
        if (plain_fasta) {
            size_t total = 0;
            for (auto& h : heads) total += h.size();
            recs.resize(total);
            size_t k = 0;
            for (auto& h : heads)
                for (const char* p : h) recs[k++].name = p;   // header position for now
            // names, sequence ranges and lengths in parallel
            std::atomic<size_t> nx(0);
            // header positions (the next record's header ends this record's sequence block)
            std::vector<const char*> hp(recs.size());
            for (size_t i = 0; i < recs.size(); ++i) hp[i] = recs[i].name;
            auto fill2 = [&]() {
                for (;;) {
                    const size_t b = nx.fetch_add(1024);
                    if (b >= recs.size()) break;
                    const size_t e = std::min(recs.size(), b + 1024);
                    for (size_t i = b; i < e; ++i) {
                        const char* p = hp[i];
                        const char* stop = i + 1 < hp.size() ? hp[i + 1] : end;
                        const char* le = line_end(p, end);
                        const char* hb = p + 1;
                        const char* he = rstrip_crlf(hb, le);
                        const char* sp = (const char*)memchr(hb, ' ', (size_t)(he - hb));
                        Rec r;
                        r.name = hb;
                        r.name_len = (sp ? sp : he) - hb;
                        r.seq = le < end ? le + 1 : end;
                        if (r.seq > stop) r.seq = stop;
                        r.seq_end = stop;
                        int64_t len = 0;
                        for (const char* q = r.seq; q < stop;) {
                            const char* e2 = line_end(q, stop);
                            len += rstrip_crlf(q, e2) - q;
                            q = e2 < stop ? e2 + 1 : stop;
                        }
                        r.len = len;
                        recs[i] = r;
                    }
                }
            };
            std::vector<std::thread> th2;
            for (int t = 1; t < n_threads; ++t) th2.emplace_back(fill2);
            fill2();
            for (auto& t : th2) t.join();
        }
    }
    if (!plain_fasta) {
        // readfq's state machine (fasta2dic.py:4-39): a header is a line starting with '>' or '@' where a header is
        // expected; inside a sequence block a line starting with '@', '+' or '>' ends it; a '+' line starts a quality
        // block that is skipped until it is at least as long as the sequence.
        const char* p = data;
        while (p < end) {
            const char* le = line_end(p, end);
            if (le > p && (*p == '>' || *p == '@')) {
                Rec r;
                const char* hb = p + 1;
                const char* he = rstrip_crlf(hb, le);
                const char* sp = (const char*)memchr(hb, ' ', (size_t)(he - hb));
                r.name = hb;
                r.name_len = (sp ? sp : he) - hb;
                p = le < end ? le + 1 : end;
                r.seq = p;
                int64_t len = 0;
                bool plus = false;
                while (p < end) {
                    const char* e2 = line_end(p, end);
                    if (e2 > p && (*p == '>' || *p == '@' || *p == '+')) {
                        plus = *p == '+';
                        break;
                    }
                    len += rstrip_crlf(p, e2) - p;
                    p = e2 < end ? e2 + 1 : end;
                }
                r.seq_end = p;
                r.len = len;
                recs.push_back(r);
                if (plus) {
                    const char* e2 = line_end(p, end);
                    p = e2 < end ? e2 + 1 : end;
                    int64_t got = 0;
                    while (p < end && got < len) {
                        const char* e3 = line_end(p, end);
                        got += rstrip_crlf(p, e3) - p;
                        p = e3 < end ? e3 + 1 : end;
                    }
                }
            } else {
                p = le < end ? le + 1 : end;   // text before the first header / between records is ignored
            }
        }
    }

    apples_fasta* f = new apples_fasta();
    f->n = (int64_t)recs.size();
    f->lengths.resize(recs.size());
    f->name_off.resize(recs.size() + 1);
    int64_t max_len = 0, min_len = INT64_MAX, name_bytes = 0;
    for (size_t i = 0; i < recs.size(); ++i) {
        f->lengths[i] = recs[i].len;
        max_len = std::max(max_len, recs[i].len);
        min_len = std::min(min_len, recs[i].len);
        f->name_off[i] = name_bytes;
        name_bytes += recs[i].name_len + 1;
    }
    f->name_off[recs.size()] = name_bytes;
    f->names.resize((size_t)name_bytes);
    for (size_t i = 0; i < recs.size(); ++i) {
        memcpy(&f->names[(size_t)f->name_off[i]], recs[i].name, (size_t)recs[i].name_len);
        f->names[(size_t)f->name_off[i] + (size_t)recs[i].name_len] = '\0';
    }
    f->max_len = max_len;
    f->uniform = recs.empty() || min_len == max_len;
    f->stride = (max_len + 15) / 16 * 16;
    const size_t bytes = std::max<size_t>((size_t)f->n * (size_t)f->stride, 16);
    if (want_pinned && cudaHostAlloc((void**)&f->matrix, bytes, cudaHostAllocDefault) == cudaSuccess) {
        f->pinned = true;
    } else {
        cudaGetLastError();   // no device / no driver: plain memory
        f->matrix = (uint8_t*)malloc(bytes);
        if (!f->matrix) {
            delete f;
            if (size) munmap((void*)data, size);
            set_err(err, errlen, "out of memory");
            return -3;
        }
    }

    // ---- pass 2 (parallel): normalise and copy.  fasta2dic.py:52-72: upper() or lower-case -> '-' (mask), then the
    // letters outside the alphabet -> '-'.  Every other byte is kept as it is.
    uint8_t tab[256];
    for (int c = 0; c < 256; ++c) tab[c] = (uint8_t)c;
    for (int c = 'a'; c <= 'z'; ++c) tab[c] = mask_flag ? (uint8_t)'-' : (uint8_t)(c - 32);
    const char* invalid = prot_flag ? "BJOUXZ" : "BDEFHIJKLMNOPQRSUVWXYZ";
    for (const char* q = invalid; *q; ++q) {
        tab[(unsigned char)*q] = '-';
        if (!mask_flag) tab[(unsigned char)(*q + 32)] = '-';   // upper() first, then the translation
    }
    std::atomic<size_t> next(0);
    auto work = [&]() {
        const size_t chunk = 256;
        for (;;) {
            const size_t b = next.fetch_add(chunk);
            if (b >= recs.size()) break;
            const size_t e = std::min(recs.size(), b + chunk);
            for (size_t i = b; i < e; ++i) {
                uint8_t* dst = f->matrix + i * (size_t)f->stride;
                int64_t k = 0;
                const char* p = recs[i].seq;
                const char* se = recs[i].seq_end;
                while (p < se) {
                    const char* le = line_end(p, se);
                    const char* te = rstrip_crlf(p, le);
                    for (const char* c = p; c < te; ++c) dst[k++] = tab[(unsigned char)*c];
                    p = le < se ? le + 1 : se;
                }
                for (; k < f->stride; ++k) dst[k] = '-';
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < n_threads; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    if (size) munmap((void*)data, size);
    *out = f;
    return 0;
}

void apples_fasta_close(apples_fasta* f) {
    if (!f) return;
    if (f->matrix) {
        if (f->pinned) cudaFreeHost(f->matrix); else free(f->matrix);
    }
    delete f;
}

int64_t apples_fasta_count(const apples_fasta* f) { return f ? f->n : 0; }
int64_t apples_fasta_max_len(const apples_fasta* f) { return f ? f->max_len : 0; }
int64_t apples_fasta_stride(const apples_fasta* f) { return f ? f->stride : 0; }
int apples_fasta_uniform(const apples_fasta* f) { return f && f->uniform ? 1 : 0; }
int apples_fasta_pinned(const apples_fasta* f) { return f && f->pinned ? 1 : 0; }
const uint8_t* apples_fasta_matrix(const apples_fasta* f) { return f ? f->matrix : nullptr; }
const int64_t* apples_fasta_lengths(const apples_fasta* f) { return f ? f->lengths.data() : nullptr; }
const char* apples_fasta_names(const apples_fasta* f) { return f ? f->names.data() : nullptr; }
const int64_t* apples_fasta_name_offsets(const apples_fasta* f) { return f ? f->name_off.data() : nullptr; }

}  // extern "C"

// =================================================================================================================
// jplace writer
// =================================================================================================================
namespace {

// float.__repr__ (Python 3: shortest round-trip digits; fixed notation for 1e-4 <= |x| < 1e16, else exponent with at
// least two exponent digits; ".0" appended to integral values in fixed notation)
void py_float_repr(double x, std::string& out) {
    if (std::isnan(x)) { out += "NaN"; return; }            // json.dumps spelling
    if (std::isinf(x)) { out += x > 0 ? "Infinity" : "-Infinity"; return; }
    if (x == 0.0) { out += std::signbit(x) ? "-0.0" : "0.0"; return; }
    char buf[64];
    auto r = std::to_chars(buf, buf + sizeof buf, x, std::chars_format::scientific);   // shortest: d[.ddd]e[+-]XX
    const char* p = buf;
    if (*p == '-') { out += '-'; ++p; }
    char digits[32];
    int nd = 0;
    const char* e = p;
    while (e < r.ptr && *e != 'e') {
        if (*e != '.') digits[nd++] = *e;
        ++e;
    }
    int exp10 = 0;
    std::from_chars(e + 1 + (e[1] == '+' ? 1 : 0), r.ptr, exp10);
    const int decpt = exp10 + 1;   // position of the decimal point relative to the first digit
    if (decpt > 16 || decpt < -3) {
        out += digits[0];
        if (nd > 1) {
            out += '.';
            out.append(digits + 1, (size_t)(nd - 1));
        }
        out += 'e';
        const int ex = decpt - 1;
        out += ex < 0 ? '-' : '+';
        const int ax = ex < 0 ? -ex : ex;
        if (ax < 10) out += '0';
        out += std::to_string(ax);
    } else if (decpt <= 0) {
        out += "0.";
        out.append((size_t)(-decpt), '0');
        out.append(digits, (size_t)nd);
    } else if (decpt >= nd) {
        out.append(digits, (size_t)nd);
        out.append((size_t)(decpt - nd), '0');
        out += ".0";
    } else {
        out.append(digits, (size_t)decpt);
        out += '.';
        out.append(digits + decpt, (size_t)(nd - decpt));
    }
}

// json.encoder.encode_basestring_ascii of a UTF-8 string (quotes included); returns false on invalid UTF-8
bool json_escape_ascii(const char* s, size_t n, const char* suffix, std::string& out) {
    static const char* hex = "0123456789abcdef";
    auto put_u = [&](unsigned cp) {
        out += "\\u";
        out += hex[(cp >> 12) & 15]; out += hex[(cp >> 8) & 15]; out += hex[(cp >> 4) & 15]; out += hex[cp & 15];
    };
    out += '"';
    size_t i = 0;
    while (i < n) {
        const unsigned char c = (unsigned char)s[i];
        if (c < 0x80) {
            switch (c) {
                case '"': out += "\\\""; break;
                case '\\': out += "\\\\"; break;
                case '\n': out += "\\n"; break;
                case '\r': out += "\\r"; break;
                case '\t': out += "\\t"; break;
                case '\b': out += "\\b"; break;
                case '\f': out += "\\f"; break;
                default:
                    if (c < 0x20 || c == 0x7f) put_u(c); else out += (char)c;
            }
            ++i;
            continue;
        }
        const int extra = (c & 0xe0) == 0xc0 ? 1 : (c & 0xf0) == 0xe0 ? 2 : (c & 0xf8) == 0xf0 ? 3 : -1;
        if (extra < 0 || i + (size_t)extra >= n) return false;
        unsigned cp = extra == 1 ? (c & 0x1fu) : extra == 2 ? (c & 0x0fu) : (c & 0x07u);
        for (int k = 1; k <= extra; ++k) {
            const unsigned char cc = (unsigned char)s[i + (size_t)k];
            if ((cc & 0xc0) != 0x80) return false;
            cp = (cp << 6) | (cc & 0x3fu);
        }
        i += (size_t)extra + 1;
        if (cp >= 0x10000) {
            cp -= 0x10000;
            put_u(0xd800 + (cp >> 10));
            put_u(0xdc00 + (cp & 0x3ff));
        } else {
            put_u(cp);
        }
    }
    for (const char* q = suffix; q && *q; ++q) out += *q;
    out += '"';
    return true;
}

}  // namespace

extern "C" {

int apples_jplace_write(const char* path, const char* prefix, const char* suffix, int64_t n, const char* names,
                        const int64_t* name_off, const uint8_t* in_backbone, const int32_t* edge, const double* error,
                        const double* distal, const double* pendant, const int32_t* status, int exclude_intplace,
                        int n_threads, int64_t* n_written, char* err, int errlen) {
    return apples_jplace_write_k(path, prefix, suffix, n, names, name_off, in_backbone, edge, error, distal, pendant, status,
                                 exclude_intplace, 1, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, n_threads,
                                 n_written, err, errlen);
}

int apples_jplace_write_k(const char* path, const char* prefix, const char* suffix, int64_t n, const char* names,
                          const int64_t* name_off, const uint8_t* in_backbone, const int32_t* edge, const double* error,
                          const double* distal, const double* pendant, const int32_t* status, int exclude_intplace,
                          int32_t keep, const int32_t* alt_count, const int32_t* alt_edge, const double* alt_error,
                          const double* alt_distal, const double* alt_pendant, const uint8_t* alt_int0, int n_threads,
                          int64_t* n_written, char* err, int errlen) {
    if (!path || !prefix || !suffix || n < 0 || (n > 0 && (!names || !name_off || !edge || !error || !distal || !pendant || !status)))
        return -1;
    if (keep < 1 || keep > APPLES_MAX_KEEP ||
        (keep > 1 && n > 0 && (!alt_count || !alt_edge || !alt_error || !alt_distal || !alt_pendant || !alt_int0)))
        return -1;
    if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    n_threads = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(n_threads, 64), (n + 4095) / 4096));
    // which records are written (jutil.py:11-19): a single result is dropped when its edge is -1; of several, the first
    // is always kept and later ones with edge -1 are dropped
    auto final_edge = [&](int64_t i) -> int32_t {
        const int code = status[i] & APPLES_STATUS_CODE_MASK;
        if (code == APPLES_TOO_FEW_DISTANCES) return -1;
        if (code == APPLES_PLACED_MISPLACEMENT_FLAG && exclude_intplace) return -1;
        return edge[i];
    };
    std::vector<std::string> parts((size_t)n_threads);
    std::vector<int64_t> counts((size_t)n_threads, 0);
    std::atomic<int> bad(0);
    const int64_t per = (n + n_threads - 1) / std::max(n_threads, 1);
    auto work = [&](int t) {
        std::string& out = parts[(size_t)t];
        const int64_t b = (int64_t)t * per, e = std::min<int64_t>(n, b + per);
        out.reserve((size_t)std::max<int64_t>(0, e - b) * 330);
        for (int64_t i = b; i < e; ++i) {
            const int32_t fe = final_edge(i);
            if (fe == -1 && (n == 1 || i > 0)) continue;
            const int code = status[i] & APPLES_STATUS_CODE_MASK;
            out += counts[(size_t)t] || t > 0 ? ",\n" : "";
            out += "        {\n            \"n\": [\n                ";
            const char* nm = names + name_off[i];
            if (!json_escape_ascii(nm, strlen(nm), (in_backbone && in_backbone[i]) ? "-query" : nullptr, out)) bad.store(1);
            out += "\n            ],\n            \"p\": [\n                [\n                    ";
            out += std::to_string(fe);
            out += ",\n                    ";
            const bool plain = code == APPLES_ZERO_DIST_LEAF || code == APPLES_TOO_FEW_DISTANCES;
            if (plain) out += '0'; else py_float_repr(error[i], out);
            out += ",\n                    1,\n                    ";
            if (plain) out += '0'; else py_float_repr(distal[i], out);
            out += ",\n                    ";
            if (plain || (status[i] & APPLES_FLAG_PENDANT_INT0)) out += '0'; else py_float_repr(pendant[i], out);
            out += "\n                ]";
            // records 1.. of a least-squares placement (keep > 1): like_weight_ratio 0
            const int cnt = (keep > 1 && !plain && fe != -1) ? std::min<int32_t>(alt_count[i], keep) : 1;
            for (int j = 1; j < cnt; ++j) {
                const int64_t o = i * keep + j;
                out += ",\n                [\n                    ";
                out += std::to_string(alt_edge[o]);
                out += ",\n                    ";
                py_float_repr(alt_error[o], out);
                out += ",\n                    0,\n                    ";
                py_float_repr(alt_distal[o], out);
                out += ",\n                    ";
                if (alt_int0[o]) out += '0'; else py_float_repr(alt_pendant[o], out);
                out += "\n                ]";
            }
            out += "\n            ]\n        }";
            counts[(size_t)t]++;
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < n_threads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
    if (bad.load()) {
        set_err(err, errlen, "a query name is not valid UTF-8");
        return -4;
    }
    // chunks other than the first started with ",\n" unconditionally: drop it where nothing precedes
    int64_t total = 0;
    FILE* fp = fopen(path, "wb");
    if (!fp) {
        set_err(err, errlen, std::string("cannot open ") + path + " for writing");
        return -2;
    }
    bool ok = fwrite(prefix, 1, strlen(prefix), fp) == strlen(prefix);
    int64_t kept = 0;
    for (int t = 0; t < n_threads; ++t) kept += counts[(size_t)t];
    if (ok) ok = fputs(kept ? "[\n" : "[", fp) >= 0;   // json.dumps(indent=4): an empty list is "[]"
    bool any = false;
    for (int t = 0; t < n_threads && ok; ++t) {
        const std::string& s = parts[(size_t)t];
        if (s.empty()) continue;
        size_t skip = (!any && t > 0 && s.size() >= 2 && s[0] == ',' && s[1] == '\n') ? 2 : 0;
        ok = fwrite(s.data() + skip, 1, s.size() - skip, fp) == s.size() - skip;
        any = true;
        total += counts[(size_t)t];
    }
    if (ok) ok = fputs(kept ? "\n    ]" : "]", fp) >= 0;
    if (ok) ok = fwrite(suffix, 1, strlen(suffix), fp) == strlen(suffix);
    if (fclose(fp) != 0) ok = false;
    if (!ok) {
        set_err(err, errlen, "write failed");
        return -2;
    }
    if (n_written) *n_written = total;
    return 0;
}

}  // extern "C"

// =================================================================================================================
// newick reader / extended-newick writer (SURVEY.md section 8 a13: tree layout)
// =================================================================================================================
// apples_newick_parse: newick text -> flat arrays in post-order (node id = the reference's edge_index, util.py:57-69),
// with levels (util.py:72-88) and the smallest id of every subtree.  It is the native twin of
// apples_b200/tree.py BackboneTree.from_newick, which stays the definition of the accepted language: this parser handles
// well-formed input (balanced parentheses and brackets, closed quotes, plain decimal branch lengths) and answers
// APPLES_NEWICK_UNSUPPORTED for anything else, so that the caller falls back to the Python twin instead of guessing.
// apples_newick_extended: arrays -> the newick string with `{edge_index}` after every non-root node (jutil.py:22-96).
// A 200 000-leaf backbone takes 2 s + 0.8 s in Python and 25 ms + 25 ms here (run_apples.py set-up, once per run).
struct apples_newick {
    int64_t n = 0;
    int rooted = 0;
    std::vector<int32_t> parent, level, first;
    std::vector<double> elen;
    std::vector<uint8_t> has_length, has_label;
    std::string labels;
    std::vector<int64_t> label_off;   // n + 1
};

namespace {

inline bool nw_space(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13) || c == 0x1c || c == 0x1d || c == 0x1e || c == 0x1f; }  // str \s for ASCII
inline bool nw_label_char(unsigned char c) {
    return !(nw_space(c) || c == '(' || c == ')' || c == ',' || c == ':' || c == ';' || c == '[' || c == ']' || c == '\'');
}

// float(tok) for plain decimal tokens; false: leave the token to Python (inf, nan, underscores, hex, ...)
bool nw_parse_length(const char* b, const char* e, double& out) {
    if (b == e) return false;
    for (const char* p = b; p < e; ++p) {
        const char c = *p;
        if (!((c >= '0' && c <= '9') || c == '.' || c == 'e' || c == 'E' || c == '+' || c == '-')) return false;
    }
    const char* p = b;
    if (*p == '+') {
        ++p;
        if (p == e || *p == '-' || *p == '+') return false;
    }
    auto r = std::from_chars(p, e, out);
    return r.ec == std::errc() && r.ptr == e;
}

}  // namespace

extern "C" {

int apples_newick_parse(const char* text, int64_t len, apples_newick** out, char* err, int errlen) {
    if (!text || !out || len < 0) {
        set_err(err, errlen, "apples_newick_parse: bad arguments");
        return -1;
    }
    const char* b = text;
    const char* e = text + len;
    while (b < e && nw_space((unsigned char)*b)) ++b;            // s.strip()
    while (e > b && nw_space((unsigned char)e[-1])) --e;
    for (const char* p = b; p < e; ++p)
        if ((unsigned char)*p >= 0x80) {
            // non-ASCII text: str.strip / \s know more blanks than this parser (U+0085, U+00A0, U+2028, ...)
            bool blank_risk = false;
            const unsigned char c = (unsigned char)*p, d = p + 1 < e ? (unsigned char)p[1] : 0;
            if (c == 0xc2 && (d == 0x85 || d == 0xa0)) blank_risk = true;
            if (c == 0xe1 || c == 0xe2 || c == 0xe3) blank_risk = true;   // U+1680, U+2000-200A, U+2028/9, U+202F, U+205F, U+3000 live here
            if (blank_risk) return APPLES_NEWICK_UNSUPPORTED;
        }
    int rooted = (e - b >= 4 && memcmp(b, "[&R]", 4) == 0) ? 1 : 0;
    if (b < e && *b == '[') {
        const char* q = (const char*)memchr(b, ']', (size_t)(e - b));
        if (!q) return APPLES_NEWICK_UNSUPPORTED;                    // s.index(']') raises
        b = q + 1;
    }
    // creation (pre-order) arrays
    std::vector<int32_t> c_parent{-1};
    std::vector<double> c_len{0.0};
    std::vector<uint8_t> c_has_len{0}, c_has_label{0};
    std::vector<std::pair<const char*, const char*>> c_label{{nullptr, nullptr}};
    int64_t cur = 0;
    bool expect_len = false;
    auto add_node = [&](int32_t par) {
        c_parent.push_back(par);
        c_len.push_back(0.0);
        c_has_len.push_back(0);
        c_has_label.push_back(0);
        c_label.push_back({nullptr, nullptr});
        cur = (int64_t)c_parent.size() - 1;
    };
    const char* p = b;
    bool done = false;
    while (p < e && !done) {
        const unsigned char c = (unsigned char)*p;
        if (nw_space(c)) { ++p; continue; }
        switch (c) {
            case '(': add_node((int32_t)cur); ++p; break;
            case ',':
                if (c_parent[cur] < 0) return APPLES_NEWICK_UNSUPPORTED;
                add_node(c_parent[cur]);
                ++p;
                break;
            case ')':
                if (c_parent[cur] < 0) return APPLES_NEWICK_UNSUPPORTED;
                cur = c_parent[cur];
                ++p;
                break;
            case ':': expect_len = true; ++p; break;
            case ';': done = true; break;
            case '[': {
                const char* q = (const char*)memchr(p, ']', (size_t)(e - p));
                if (!q) return APPLES_NEWICK_UNSUPPORTED;
                p = q + 1;
                break;
            }
            case ']': return APPLES_NEWICK_UNSUPPORTED;
            default: {
                const char *tb, *te;
                bool quoted = false;
                if (c == '\'') {
                    const char* q = (const char*)memchr(p + 1, '\'', (size_t)(e - p - 1));
                    if (!q) return APPLES_NEWICK_UNSUPPORTED;
                    tb = p + 1;
                    te = q;
                    p = q + 1;
                    quoted = true;
                } else {
                    tb = p;
                    while (p < e && nw_label_char((unsigned char)*p)) ++p;
                    te = p;
                }
                if (expect_len) {
                    double x;
                    if (quoted || !nw_parse_length(tb, te, x)) return APPLES_NEWICK_UNSUPPORTED;
                    c_len[cur] = x;
                    c_has_len[cur] = 1;
                    expect_len = false;
                } else {
                    c_label[cur] = {tb, te};
                    c_has_label[cur] = 1;
                }
            }
        }
    }
    const int64_t n = (int64_t)c_parent.size();
    if (n > 0x7fffffff) {
        set_err(err, errlen, "apples_newick_parse: more than 2^31 nodes");
        return -1;
    }
    // children in creation order (= left to right), as a CSR
    std::vector<int32_t> cnt(n + 1, 0), kids(n > 1 ? n - 1 : 0);
    for (int64_t v = 1; v < n; ++v) cnt[c_parent[v] + 1]++;
    for (int64_t v = 0; v < n; ++v) cnt[v + 1] += cnt[v];
    {
        std::vector<int32_t> fill(cnt.begin(), cnt.end() - 1);
        for (int64_t v = 1; v < n; ++v) kids[fill[c_parent[v]]++] = (int32_t)v;
    }
    // post-order rank: children left to right, then the node (util.py:64-69)
    std::vector<int32_t> rank(n, 0);
    {
        std::vector<std::pair<int32_t, int32_t>> st;   // (node, next child position)
        st.push_back({0, cnt[0]});
        int32_t r = 0;
        while (!st.empty()) {
            auto& top = st.back();
            if (top.second < cnt[top.first + 1]) {
                const int32_t ch = kids[top.second++];
                st.push_back({ch, cnt[ch]});
            } else {
                rank[top.first] = r++;
                st.pop_back();
            }
        }
    }
    auto* t = new apples_newick();
    t->n = n;
    t->rooted = rooted;
    t->parent.assign(n, -1);
    t->elen.assign(n, 0.0);
    t->has_length.assign(n, 0);
    t->has_label.assign(n, 0);
    std::vector<int32_t> by_rank(n);
    for (int64_t v = 0; v < n; ++v) by_rank[rank[v]] = (int32_t)v;
    t->label_off.assign(n + 1, 0);
    for (int64_t r = 0; r < n; ++r) {
        const int32_t v = by_rank[r];
        if (c_parent[v] >= 0) t->parent[r] = rank[c_parent[v]];
        if (c_has_len[v]) {
            t->elen[r] = c_len[v];
            t->has_length[r] = 1;
        }
        if (c_has_label[v]) {
            t->has_label[r] = 1;
            t->labels.append(c_label[v].first, (size_t)(c_label[v].second - c_label[v].first));
        }
        t->label_off[r + 1] = (int64_t)t->labels.size();
    }
    // levels (root 0) and the smallest id of every subtree: parents have larger ids than their children
    t->level.assign(n, 0);
    t->first.resize(n);
    for (int64_t u = n - 2; u >= 0; --u) t->level[u] = t->level[t->parent[u]] + 1;
    for (int64_t u = 0; u < n; ++u) t->first[u] = (int32_t)u;
    for (int64_t u = 0; u + 1 < n; ++u) {
        const int32_t pp = t->parent[u];
        if (t->first[u] < t->first[pp]) t->first[pp] = t->first[u];
    }
    *out = t;
    return 0;
}

void apples_newick_free(apples_newick* t) { delete t; }
int64_t apples_newick_nodes(const apples_newick* t) { return t ? t->n : 0; }
int apples_newick_rooted(const apples_newick* t) { return t ? t->rooted : 0; }
const int32_t* apples_newick_parent(const apples_newick* t) { return t ? t->parent.data() : nullptr; }
const int32_t* apples_newick_level(const apples_newick* t) { return t ? t->level.data() : nullptr; }
const int32_t* apples_newick_first(const apples_newick* t) { return t ? t->first.data() : nullptr; }
const double* apples_newick_edge_length(const apples_newick* t) { return t ? t->elen.data() : nullptr; }
const uint8_t* apples_newick_has_length(const apples_newick* t) { return t ? t->has_length.data() : nullptr; }
const uint8_t* apples_newick_has_label(const apples_newick* t) { return t ? t->has_label.data() : nullptr; }
const char* apples_newick_labels(const apples_newick* t) { return t ? t->labels.data() : nullptr; }
const int64_t* apples_newick_label_offsets(const apples_newick* t) { return t ? t->label_off.data() : nullptr; }

int apples_newick_extended(int64_t n, const int32_t* parent, const double* elen, const uint8_t* has_length, const char* labels,
                           const int64_t* label_off, const uint8_t* has_label, int rooted, char** out_text, int64_t* out_len,
                           char* err, int errlen) {
    if (n <= 0 || !parent || !elen || !has_length || !label_off || !has_label || !out_text || !out_len) {
        set_err(err, errlen, "apples_newick_extended: bad arguments");
        return -1;
    }
    // children by increasing id (left to right)
    std::vector<int32_t> cnt(n + 1, 0), kids(n > 1 ? n - 1 : 0);
    for (int64_t v = 0; v < n; ++v) {
        if (parent[v] >= n || (parent[v] >= 0 && parent[v] <= v)) {
            set_err(err, errlen, "apples_newick_extended: parents must follow their children (post-order ids)");
            return -1;
        }
        if (parent[v] >= 0) cnt[parent[v] + 1]++;
    }
    for (int64_t v = 0; v < n; ++v) cnt[v + 1] += cnt[v];
    {
        std::vector<int32_t> fill(cnt.begin(), cnt.end() - 1);
        for (int64_t v = 0; v < n; ++v)
            if (parent[v] >= 0) kids[fill[parent[v]]++] = (int32_t)v;
    }
    std::string s;
    s.reserve((size_t)n * 24);
    if (rooted) s += "[&R] ";
    // tail of a node: label, ':' length, '{id}'
    auto close_node = [&](int32_t u) -> bool {
        if (has_label[u]) s.append(labels + label_off[u], (size_t)(label_off[u + 1] - label_off[u]));
        if (parent[u] >= 0) {
            if (has_length[u]) {
                const double x = elen[u];
                s += ':';
                if (std::isnan(x)) s += "nan";
                else if (std::isinf(x)) s += x > 0 ? "inf" : "-inf";
                else if (x == std::floor(x)) {           // x.is_integer(): str(int(x))
                    if (std::fabs(x) >= 9.0e18) return false;
                    s += std::to_string((long long)x);
                } else py_float_repr(x, s);
            }
            s += '{';
            s += std::to_string(u);
            s += '}';
        }
        return true;
    };
    std::vector<std::pair<int32_t, int32_t>> st;
    const int32_t root = (int32_t)(n - 1);
    st.push_back({root, cnt[root]});
    if (cnt[root + 1] > cnt[root]) s += '(';
    while (!st.empty()) {
        auto& top = st.back();
        const int32_t u = top.first;
        if (top.second < cnt[u + 1]) {
            if (top.second > cnt[u]) s += ',';
            const int32_t ch = kids[top.second++];
            if (cnt[ch + 1] > cnt[ch]) s += '(';
            st.push_back({ch, cnt[ch]});
        } else {
            if (cnt[u + 1] > cnt[u]) s += ')';
            if (!close_node(u)) return APPLES_NEWICK_UNSUPPORTED;
            st.pop_back();
        }
    }
    s += ';';
    char* buf = (char*)malloc(s.size() + 1);
    if (!buf) {
        set_err(err, errlen, "apples_newick_extended: out of memory");
        return -1;
    }
    memcpy(buf, s.data(), s.size() + 1);
    *out_text = buf;
    *out_len = (int64_t)s.size();
    return 0;
}

void apples_free_text(char* p) { free(p); }

}  // extern "C"
