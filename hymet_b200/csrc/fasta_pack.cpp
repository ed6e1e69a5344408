// fasta_pack.cpp -- see fasta_pack.h.  Host code, no CUDA.
//
// The packer is the end-to-end limiter (the GPU consumes > 100 Gbp/s), so sequence
// lines are converted 32 characters at a time with AVX2 when the host has it
// (runtime dispatch; the scalar loop is the same arithmetic one character at a time).
#include "fasta_pack.h"

#include <string.h>
#include <zlib.h>

#if defined(__x86_64__)
#include <immintrin.h>
#define HS_X86 1
#endif

namespace hs {

namespace {

struct Lut {
    uint8_t v[256];
    Lut()
    {
        for (int i = 0; i < 256; i++) v[i] = 4;  // not in the alphabet (S4) -> invalid position
        v['A'] = v['a'] = 0;                     // S3: case folded
        v['C'] = v['c'] = 1;
        v['G'] = v['g'] = 2;
        v['T'] = v['t'] = 3;
    }
};
const Lut kLut;

// Left-aligned accumulator: base i of the pending word sits at bits [62-2i, 63-2i],
// its invalid flag at bit (31-i).
struct Writer {
    uint64_t *seq;
    uint32_t *inv;
    uint64_t w = 0, acc = 0;
    uint32_t iacc = 0;
    int cnt = 0;
    uint64_t positions = 0;

    inline void push(uint32_t code)
    {
        acc |= (uint64_t)(code & 3u) << (62 - 2 * cnt);
        iacc |= (code >> 2) << (31 - cnt);
        if (++cnt == 32) {
            seq[w] = acc; inv[w] = iacc; w++;
            cnt = 0; acc = 0; iacc = 0;
        }
        positions++;
    }
    // n (1..32) bases: codes left-aligned in c, flags left-aligned in m, unused low bits zero
    inline void append(uint64_t c, uint32_t m, int n)
    {
        if (cnt) { acc |= c >> (2 * cnt); iacc |= m >> cnt; } else { acc = c; iacc = m; }
        if (cnt + n >= 32) {
            seq[w] = acc; inv[w] = iacc; w++;
            const int used = 32 - cnt;
            if (used < 32) { acc = c << (2 * used); iacc = m << used; } else { acc = 0; iacc = 0; }
            cnt = cnt + n - 32;
        } else {
            cnt += n;
        }
        positions += (uint64_t)n;
    }
    inline void finish()
    {
        if (cnt) {
            seq[w] = acc;
            inv[w] = iacc | ((1u << (32 - cnt)) - 1u);  // padding is invalid
            w++;
            cnt = 0; acc = 0; iacc = 0;
        }
    }
};

void line_scalar(Writer &wr, const unsigned char *p, size_t L)
{
    for (size_t q = 0; q < L; q++) wr.push(kLut.v[p[q]]);
}

#ifdef HS_X86
// 32 characters -> 64 bits of 2-bit codes (first base most significant) + 32 invalid flags.
__attribute__((target("avx2"))) inline void convert32(__m256i v, uint64_t &codes, uint32_t &bad)
{
    const __m256i up = _mm256_and_si256(v, _mm256_set1_epi8((char)0xDF));            // fold case (S3)
    const __m256i c1 = _mm256_and_si256(_mm256_srli_epi16(up, 1), _mm256_set1_epi8(3));  // A0 C1 T2 G3
    const __m256i code = _mm256_xor_si256(c1, _mm256_and_si256(_mm256_srli_epi16(c1, 1), _mm256_set1_epi8(1)));  // A0 C1 G2 T3
    const __m256i letters = _mm256_setr_epi8('A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                             'A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0);
    const __m256i ok = _mm256_cmpeq_epi8(up, _mm256_shuffle_epi8(letters, code));   // S4: exactly A/C/G/T
    // reverse byte order inside each 128-bit half so movemask puts base 0 at the top
    const __m256i rev = _mm256_setr_epi8(15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0,
                                         15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0);
    const uint32_t mm = ~(uint32_t)_mm256_movemask_epi8(_mm256_shuffle_epi8(ok, rev));
    bad = (mm << 16) | (mm >> 16);
    // four codes -> one byte (first base in the top two bits), then 8 bytes -> big-endian u64
    const __m256i w16 = _mm256_maddubs_epi16(_mm256_and_si256(code, ok),  // invalid positions carry code 0
                                             _mm256_set1_epi32(0x01041040));  // (c0*64+c1*16), (c2*4+c3)
    const __m256i w32 = _mm256_madd_epi16(w16, _mm256_set1_epi16(1));
    const __m256i b16 = _mm256_packus_epi32(w32, w32);
    const __m256i b8 = _mm256_packus_epi16(b16, b16);
    const uint64_t lo = (uint32_t)_mm256_extract_epi32(b8, 0), hi = (uint32_t)_mm256_extract_epi32(b8, 4);
    codes = __builtin_bswap64(lo | (hi << 32));
}

__attribute__((target("avx2"))) void line_avx2(Writer &wr, const unsigned char *p, size_t L, const unsigned char *safe_end)
{
    size_t off = 0;
    if (L >= 32) {
        // full vectors: the bit offset inside the pending word is constant along the line,
        // so the accumulator stays in registers and the loop has no branches
        uint64_t acc = wr.acc, w = wr.w;
        uint32_t iacc = wr.iacc;
        uint64_t *seq = wr.seq;
        uint32_t *inv = wr.inv;
        const int r = wr.cnt;
        if (r == 0) {
            for (; off + 32 <= L; off += 32, w++) {
                uint64_t c; uint32_t b;
                convert32(_mm256_loadu_si256((const __m256i *)(p + off)), c, b);
                seq[w] = c; inv[w] = b;
            }
        } else {
            for (; off + 32 <= L; off += 32, w++) {
                uint64_t c; uint32_t b;
                convert32(_mm256_loadu_si256((const __m256i *)(p + off)), c, b);
                seq[w] = acc | (c >> (2 * r)); inv[w] = iacc | (b >> r);
                acc = c << (64 - 2 * r); iacc = b << (32 - r);
            }
        }
        wr.acc = acc; wr.iacc = iacc; wr.w = w;
        wr.positions += off;
    }
    const int n = (int)(L - off);
    if (n) {
        __m256i v;
        if (p + off + 32 <= safe_end) {
            v = _mm256_loadu_si256((const __m256i *)(p + off));
        } else {  // never read past the caller's buffer
            unsigned char tmp[32] = {0};
            memcpy(tmp, p + off, (size_t)n);
            v = _mm256_loadu_si256((const __m256i *)tmp);
        }
        uint64_t c; uint32_t b;
        convert32(v, c, b);
        wr.append(c & (~0ull << (64 - 2 * n)), b & (~0u << (32 - n)), n);
    }
}

// Sequence text 64 bytes at a time, across line boundaries (AVX-512 VBMI2 hosts).  The line-by-line
// path above tops out near 3 GB/s per thread on 80-column FASTA (memchr + two full vectors + a masked
// tail per line) and was the end-to-end limiter of the hybrid ingest.  Here a block of ordinary
// sequence text -- nothing below 'A' except '\n' -- has its newlines squeezed out by VPCOMPRESSB and its
// byte order reversed by VPERMB, after which the conversion of convert32() yields the 128 code bits
// and 64 flags first-base-most-significant with no further shuffling.  Anything else in a block (a
// header or '+' line, CR, digits, '-', '*' ...) stops the run BEFORE that block and the line loop takes
// over, so every rule of the format stays in one place.
// Consumes whole 64-byte blocks starting at p (a position inside a sequence line or at a line start
// whose first byte the caller has already classified as sequence); returns the bytes consumed.
#define HS_AVX512_TARGET __attribute__((target("avx512f,avx512bw,avx512vl,avx512vbmi,avx512vbmi2,bmi2,popcnt")))

// 64 newline-free characters -> two packed words + their flags.  `c` holds base i of word h at byte
// 32h + 31 - i (rev32 below), so the dword-to-byte narrowing leaves the 16 code bytes in memory order
// and the compare mask IS the two flag words: no scalar shuffling at all.
HS_AVX512_TARGET inline void convert64(__m512i c, __m128i &codes, uint64_t &bad)
{
    const __m512i letters = _mm512_broadcast_i32x4(_mm_setr_epi8('A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0));
    const __m512i up = _mm512_and_si512(c, _mm512_set1_epi8((char)0xDF));                                   // fold case (S3)
    const __m512i c1 = _mm512_and_si512(_mm512_srli_epi16(up, 1), _mm512_set1_epi8(3));                      // A0 C1 T2 G3
    const __m512i code = _mm512_xor_si512(c1, _mm512_and_si512(_mm512_srli_epi16(c1, 1), _mm512_set1_epi8(1)));  // A0 C1 G2 T3
    const __mmask64 ok = _mm512_cmpeq_epi8_mask(up, _mm512_shuffle_epi8(letters, code));                    // S4: exactly A/C/G/T
    // four codes -> one byte; the later base of a pair sits in the LOWER byte: weights 1,4 | 16,64
    const __m512i w16 = _mm512_maddubs_epi16(_mm512_maskz_mov_epi8(ok, code), _mm512_set1_epi32(0x40100401));
    codes = _mm512_cvtepi32_epi8(_mm512_madd_epi16(w16, _mm512_set1_epi16(1)));
    bad = ~(uint64_t)ok;
}

HS_AVX512_TARGET inline __m512i rev32_index()
{
    return _mm512_set_epi8(
        32, 33, 34, 35, 36, 37, 38, 39, 40, 41, 42, 43, 44, 45, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61, 62, 63,
        0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31);
}

// up to 64 newline-free characters at any bit offset of the pending word (head and tail of a run)
HS_AVX512_TARGET void append_chars(Writer &wr, const unsigned char *q, int m)
{
    if (m <= 0) return;
    const __mmask64 have = m >= 64 ? ~0ull : ((1ull << m) - 1ull);
    __m128i codes;
    uint64_t bad;
    convert64(_mm512_permutexvar_epi8(rev32_index(), _mm512_maskz_loadu_epi8(have, q)), codes, bad);
    const int n0 = m < 32 ? m : 32, n1 = m - n0;
    wr.append((uint64_t)_mm_extract_epi64(codes, 0), (uint32_t)bad & (~0u << (32 - n0)), n0);   // absent bytes converted to code 0
    if (n1) wr.append((uint64_t)_mm_extract_epi64(codes, 1), (uint32_t)(bad >> 32) & (~0u << (32 - n1)), n1);
}

// Sequence text 64 bytes at a time, across line boundaries (AVX-512 VBMI2 hosts).  The line-by-line
// path above tops out near 3 GB/s per thread on 80-column FASTA (memchr + two full vectors + a masked
// tail per line, variable shifts into the pending word) and was the end-to-end limiter of the hybrid
// ingest.  Two stages over a 4 KB scratch that stays in L1:
//   1. blocks of ordinary sequence text -- nothing below 'A' except '\n' -- have their newlines
//      squeezed out by VPCOMPRESSB and are stored back to back;
//   2. once the pending word has been completed, every 64 characters of the scratch ARE two whole
//      output words: convert64 and two stores, no carried state.
// Anything else in a block (a header or '+' line, CR, digits, '-', '*' ...) stops the run BEFORE that
// block and the line loop takes over, so every rule of the format stays in one place.
// Consumes whole 64-byte blocks starting at p (inside a sequence line, or at a line start whose first
// byte the caller has classified as sequence); returns the bytes consumed.
HS_AVX512_TARGET size_t run_avx512(Writer &wr, const unsigned char *p, size_t n, uint64_t &kept_out)
{
    constexpr size_t kScratch = 4096;
    alignas(64) unsigned char tmp[kScratch + 128];   // a 64-byte store at fill <= kScratch, a 64-byte load at q <= fill
    const __m512i rev = rev32_index();
    const __m512i vnl = _mm512_set1_epi8('\n'), vA = _mm512_set1_epi8('A');
    size_t off = 0, fill = 0;
    uint64_t kept = 0;
    bool stop = false, aligned = wr.cnt == 0;
    while (!stop && off + 64 <= n) {
        while (off + 64 <= n && fill <= kScratch) {
            _mm_prefetch((const char *)(p + off + 4096), _MM_HINT_T0);   // measured: 4.5 -> 6.4 GB/s per thread out of cache
            const __m512i v = _mm512_loadu_si512((const void *)(p + off));
            const __mmask64 nl = _mm512_cmpeq_epi8_mask(v, vnl);
            if (_mm512_cmplt_epu8_mask(v, vA) != nl) { stop = true; break; }   // something other than letters and newlines
            _mm512_storeu_si512((void *)(tmp + fill), _mm512_maskz_compress_epi8(~nl, v));
            fill += (size_t)__builtin_popcountll(~(uint64_t)nl);
            off += 64;
        }
        size_t q = 0;
        if (!aligned) {
            const size_t need = (size_t)(32 - wr.cnt);
            if (fill < need) continue;               // (only when the run is ending: the tail append takes them)
            append_chars(wr, tmp, (int)need);
            wr.positions -= need;                    // counted once, below
            q = need;
            aligned = true;
        }
        uint64_t *seq = wr.seq + wr.w;
        uint32_t *inv = wr.inv + wr.w;
        size_t words = 0;
        for (; q + 64 <= fill; q += 64, words += 2) {
            __m128i codes;
            uint64_t bad;
            convert64(_mm512_permutexvar_epi8(rev, _mm512_loadu_si512((const void *)(tmp + q))), codes, bad);
            // staging buffers are written once and read by the DMA engine only: streaming stores skip the
            // read-for-ownership of lines the CPU never looks at again (measured on the 16-vCPU B200 host:
            // e2e 13.6 -> 12.7 ms per Gbp)
            _mm_stream_si64((long long *)(seq + words), _mm_extract_epi64(codes, 0));
            _mm_stream_si64((long long *)(seq + words + 1), _mm_extract_epi64(codes, 1));
            _mm_stream_si32((int *)(inv + words), (int)(uint32_t)bad);
            _mm_stream_si32((int *)(inv + words + 1), (int)(uint32_t)(bad >> 32));
        }
        wr.w += words;
        kept += q;
        // the characters left over (< 64) move to the front for the next round
        const __m512i rest = _mm512_loadu_si512((const void *)(tmp + q));
        _mm512_storeu_si512((void *)tmp, rest);
        fill -= q;
    }
    if (fill) {
        // fewer than 64 (or, if the pending word was never completed, fewer than 32 + 64) left
        const int first = fill > 64 ? 64 : (int)fill;
        append_chars(wr, tmp, first);
        if (fill > 64) append_chars(wr, tmp + 64, (int)(fill - 64));
        wr.positions -= fill;
        kept += fill;
    }
    _mm_sfence();
    wr.positions += kept;
    kept_out = kept;
    return off;
}
#endif

int g_pack_level = -1;   // -1: best the host has; 0 scalar, 1 AVX2 lines, 2 AVX-512 runs (tests pin it)

}  // namespace

void set_pack_level(int level) { g_pack_level = level; }

int pack_level()
{
#ifdef HS_X86
    static const int best = (__builtin_cpu_supports("avx512vbmi2") && __builtin_cpu_supports("avx512vbmi") &&
                             __builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl") &&
                             __builtin_cpu_supports("bmi2")) ? 2 : (__builtin_cpu_supports("avx2") ? 1 : 0);
#else
    static const int best = 0;
#endif
    return (g_pack_level < 0 || g_pack_level > best) ? best : g_pack_level;
}

uint64_t pack_text_span(const char *t, size_t n, uint64_t *seq, uint32_t *inv, PackStats *st)
{
    Writer wr{seq, inv};
    const int level = pack_level();
    const bool have_avx2 = level >= 1;
    const unsigned char *safe_end = (const unsigned char *)t + n;
    enum { SEEK_HDR, IN_SEQ } state = SEEK_HDR;
    bool fastq = false;
    uint64_t rec_len = 0, n_records = 0, n_seq = 0;
    size_t i = 0;
    while (i < n) {
        const char *nl = (const char *)memchr(t + i, '\n', n - i);
        size_t j = nl ? (size_t)(nl - t) : n;  // line = [i, j)
        const char c0 = t[i];
        if (c0 == '>' || c0 == '@') {
            // header line: one invalid position keeps k-mers from bridging records (S6)
            state = IN_SEQ;
            fastq = (c0 == '@');
            rec_len = 0;
            wr.push(4);
            n_records++;
            i = j + 1;
            continue;
        }
        if (state == SEEK_HDR) { i = j + 1; continue; }
        if (c0 == '+') {
            i = j + 1;  // the '+' line
            if (fastq) {  // quality block: as many symbols as the sequence had
                uint64_t q = 0;
                while (i < n && q < rec_len) {
                    if (t[i] != '\n' && t[i] != '\r') q++;
                    i++;
                }
                nl = i < n ? (const char *)memchr(t + i, '\n', n - i) : nullptr;
                i = nl ? (size_t)(nl - t) + 1 : n;
            }
            state = SEEK_HDR;
            continue;
        }
#ifdef HS_X86
        if (level >= 2 && n - i >= 64) {
            // as many 64-byte blocks of plain sequence text as there are from here; if the run ends inside
            // a line, the rest of that line is sequence too (its first byte was classified above)
            uint64_t kept = 0;
            const size_t adv = run_avx512(wr, (const unsigned char *)t + i, n - i, kept);
            if (adv) {
                rec_len += kept;
                n_seq += kept;
                i += adv;
                if (t[i - 1] == '\n') continue;   // at a line start again: classify the next line
                if (i >= n) break;
                nl = (const char *)memchr(t + i, '\n', n - i);
                j = nl ? (size_t)(nl - t) : n;
            }
        }
#endif
        size_t L = j - i;
        if (L && t[i + L - 1] == '\r') L--;  // kseq: one trailing CR dropped, everything else kept
        const unsigned char *p = (const unsigned char *)t + i;
#ifdef HS_X86
        if (have_avx2) line_avx2(wr, p, L, safe_end); else
#endif
            line_scalar(wr, p, L);
        rec_len += L;
        n_seq += L;
        i = j + 1;
    }
    wr.finish();
    if (st) { st->n_records += n_records; st->n_seq_bases += n_seq; st->n_positions += wr.positions; }
    return wr.w;
}

// Offsets of the header lines AS pack_text_span SEES THEM, thinned to at least min_gap bytes apart (the first
// one is always there).  Same control flow as the packer without the packing: a line that starts with '>' or
// '@' outside a FASTQ quality block is a header and resets the packer completely, so the text can be cut in
// front of any of them -- which is what makes FASTQ splittable although '@' also starts quality lines.
std::vector<size_t> record_starts(const char *t, size_t n, size_t min_gap)
{
    std::vector<size_t> out;
    enum { SEEK_HDR, IN_SEQ } state = SEEK_HDR;
    bool fastq = false;
    uint64_t rec_len = 0;
    size_t i = 0;
    while (i < n) {
        const char *nl = (const char *)memchr(t + i, '\n', n - i);
        const size_t j = nl ? (size_t)(nl - t) : n;
        const char c0 = t[i];
        if (c0 == '>' || c0 == '@') {
            if (out.empty() || i - out.back() >= min_gap) out.push_back(i);
            state = IN_SEQ;
            fastq = (c0 == '@');
            rec_len = 0;
            i = j + 1;
            continue;
        }
        if (state == SEEK_HDR) { i = j + 1; continue; }
        if (c0 == '+') {
            i = j + 1;
            if (fastq) {
                uint64_t q = 0;
                while (i < n && q < rec_len) {
                    if (t[i] != '\n' && t[i] != '\r') q++;
                    i++;
                }
                nl = i < n ? (const char *)memchr(t + i, '\n', n - i) : nullptr;
                i = nl ? (size_t)(nl - t) + 1 : n;
            }
            state = SEEK_HDR;
            continue;
        }
        size_t L = j - i;
        if (L && t[i + L - 1] == '\r') L--;
        rec_len += L;
        i = j + 1;
    }
    return out;
}

std::vector<std::pair<size_t, size_t>> split_records(const char *t, size_t n, int parts, size_t min_span)
{
    std::vector<std::pair<size_t, size_t>> out;
    size_t first = 0;
    while (first < n && (t[first] == '\n' || t[first] == '\r')) first++;
    if (parts < 1) parts = 1;
    if (first < n && t[first] != '>' && parts > 1) {
        // FASTQ ('@' also occurs in quality lines): cut where the packer's own walk sees a header
        size_t span = n / (size_t)parts + 1;
        if (span < min_span) span = min_span;
        const std::vector<size_t> starts = record_starts(t, n, span);
        size_t beg = 0;
        for (size_t q = 1; q < starts.size(); q++) {
            if (starts[q] <= beg) continue;
            out.emplace_back(beg, starts[q]);
            beg = starts[q];
        }
        if (beg < n || out.empty()) out.emplace_back(beg, n);
        return out;
    }
    size_t span = n / (size_t)parts + 1;
    if (span < min_span) span = min_span;
    size_t beg = 0;
    while (beg < n) {
        size_t end = beg + span;
        if (end >= n || parts == 1) {
            end = n;
        } else {
            // advance to the next line that starts a record
            for (;;) {
                const char *nl = (const char *)memchr(t + end, '\n', n - end);
                if (!nl) { end = n; break; }
                end = (size_t)(nl - t) + 1;
                if (end >= n || t[end] == '>') break;
            }
        }
        out.emplace_back(beg, end);
        beg = end;
    }
    return out;
}

bool slurp_file(const std::string &path, std::vector<char> &out, std::string &err)
{
    gzFile f = path == "-" ? gzdopen(0, "rb") : gzopen(path.c_str(), "rb");
    if (!f) { err = "could not open " + path; return false; }
    gzbuffer(f, 1 << 20);
    size_t len = out.size();
    for (;;) {
        if (out.size() - len < (1u << 22)) out.resize(out.size() ? out.size() * 2 : (1u << 24));
        int r = gzread(f, out.data() + len, 1u << 22);
        if (r < 0) { err = "read error on " + path; gzclose(f); return false; }
        if (r == 0) break;
        len += (size_t)r;
    }
    gzclose(f);
    out.resize(len);
    return true;
}

}  // namespace hs
