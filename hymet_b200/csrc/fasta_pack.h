// fasta_pack.h -- FASTA/FASTQ text -> 2-bit packed query chunks (host side).
//
// Replaces the kseq reader + '*'-joined chunks of `mash screen` (SURVEY.md 8a
// rows a6/a7; the binary is invoked at /root/reference/scripts/mash.sh:14).
// Record boundaries become one invalid position, exactly like mash's '*'.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace hs {

struct PackStats {
    uint64_t n_records = 0;    // sequence records seen
    uint64_t n_seq_bases = 0;  // characters inside records (what "query bases" counts)
    uint64_t n_positions = 0;  // packed positions written (bases + separators)
};

// Upper bound on packed 64-bit words needed for `n_text` bytes of FASTA/FASTQ text.
inline uint64_t pack_words_bound(uint64_t n_text) { return n_text / 32 + 4; }

// Pack one span of text that starts at a record header (or before the first one).
// seq/inv must hold pack_words_bound(n) words.  The tail of the last word is
// flagged invalid.  Returns the number of words written.
uint64_t pack_text_span(const char *text, size_t n, uint64_t *seq, uint32_t *inv, PackStats *st);

// Which implementation pack_text_span uses: 0 scalar, 1 AVX2 line by line, 2 AVX-512 (VBMI2) runs of
// 64-byte blocks across lines.  Default -1 = the best the host supports; tests pin lower levels to
// compare them bit for bit.
void set_pack_level(int level);
int pack_level();

// Offsets of the header lines as pack_text_span sees them ('>' / '@' at a line start outside a FASTQ
// quality block), thinned to >= min_gap bytes apart.  The text may be cut in front of any of them.
std::vector<size_t> record_starts(const char *text, size_t n, size_t min_gap);

// Split [text, text+n) into about `parts` spans that each begin at a record header: a line starting with
// '>' (FASTA), or a header found by record_starts (FASTQ, where '@' may also start a quality line).
std::vector<std::pair<size_t, size_t>> split_records(const char *text, size_t n, int parts, size_t min_span);

// Whole file (plain or gzip, "-" = stdin) into memory.
bool slurp_file(const std::string &path, std::vector<char> &out, std::string &err);

}  // namespace hs
