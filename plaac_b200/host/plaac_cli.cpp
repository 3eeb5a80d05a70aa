// plaac -- host program with plaac.jar's command line, header block and output columns, scoring through
// libplaac_cuda.so (include/plaac_cuda.h).  C++ stand-in for the Java host of the north star: this image has no
// JDK, so the host side above the C ABI is written in C++ and mirrors plaac.java's CLI (main :302-530),
// FASTA reader (fastareader :4302-4375), summary table (scoreallfastas :653-950) and per-residue table
// (plotsomefastas :587-649).  All scoring happens on the GPU; there is no CPU scoring path in this file.
//
// Extra options (all start with "--" so they cannot collide with the jar's single-letter flags):
//   --gpus N        shard every batch over the first N GPUs (plaac_score_multi)
//   --device D      GPU index when --gpus is 1 (default 0)
//   --batch-mb M    residues per scoring batch in MiB (default 256; the file-to-table fast path cuts 64 MiB pieces unless
//                   the table is ranked)
//   --compat-F      keep the jar's -F bug (plaac.java:388 reads the -B file name)
//   --rank          print the rows of every scoring batch in the web front end's order (COREscore desc, LLR desc, no-CORE
//                   rows last; web/lib/server.rb:222-229), computed on the GPU (plaac_rank); --rank-core prints only the
//                   rows with a CORE.  A file that fits one batch (--batch-mb) is ranked as a whole.
//   --gpu-ingest    parse the FASTA on the GPU as well (plaac_score_fasta): the file goes to the device as raw bytes in
//                   record-aligned pieces of --batch-mb, pieces round-robin over --gpus, rows formatted on all host
//                   threads; summary table only.  The default for regular files of at least 1 MB; --host-reader forces
//                   the reader of this program instead
//   --variants FILE score sequence variants of the -i records instead of the records (plaac_score_variants): one line
//                   per variant, "SEQid<TAB>spec", spec = WT or comma-separated substitutions <ref><pos><alt> with a
//                   1-based position (D262V or D262V,P275S); SEQid is matched against record names as -p matches them.
//                   One row per variant, named <name>:<SPEC>, in record order and within a record in file order
//   --saturate      every single substitution of every -i record (wild type first, then positions in ascending order,
//                   at each one the 20 residues A..Y other than the one there)
//   --effects COLS  with --variants or --saturate: print per variant only the change of the listed summary columns
//                   against the wild type (plaac_score_variant_effects) instead of its row.  COLS is a comma-separated
//                   list of LLR COREscore PRDscore HMMall HMMvit FImeanhydro FImeancharge FImeancombo PAPAcombo PAPAprop
//                   PAPAfi PAPAllr PAPAllr2 (printed as d<NAME>, variant minus wild type) and COREchange (1 gained,
//                   -1 lost, 0 unchanged)
//   --segments FILE also write every prion-like segment of each record's Viterbi parse (each maximal run of PrD-state
//                   residues; plaac_score_segments) to FILE as a table: SEQid SEGstart SEGend SEGlen SEGscore PRD, 1-based
//                   positions, SEGscore the PRDscore sum over the segment, PRD 1 for the segment that is the row's PrD.
//                   One line per segment, in record order (also with --rank); the summary table is unchanged
//   --null FILE --replicates K [--seed S] [--null-columns COLS]
//                   also score K composition-preserving shuffles of every record on the GPU (plaac_score_shuffles) and
//                   write to FILE one line per printed record, in record order: SEQid NULLreps, then n<NAME> p<NAME> per
//                   column, n the shuffles whose value (NaN lowest) reaches the record's and p = (1+n)/(1+K) (%.6g).
//                   COLS: the names of --effects with hasCORE (shuffles with a CORE, no p column) for COREchange;
//                   default COREscore,LLR,HMMall.  A record's shuffles are those of its index in its batch (--batch-mb),
//                   so the file depends on --seed and, for inputs beyond one batch, on --batch-mb; the summary table is
//                   unchanged
//   --stop-hits H   with --null and --replicates K: the sequential null of Besag and Clifford
//                   (plaac_score_shuffles_seq).  A record's column stops once H of its shuffles have reached it, after at
//                   most K shuffles, so a protein far from significance costs about H shuffles instead of K.  The file
//                   is then SEQid, followed by r<NAME> n<NAME> p<NAME> per column: r the shuffles scored for the column,
//                   n the ones that reached the record (H if it stopped), p = H/r if it stopped and (1+n)/(1+K)
//                   otherwise (%.6g); hasCORE gets r and n and no p
#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <map>
#include <memory>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "plaac_cuda.h"

namespace {

const char kAaNames[] = "XACDEFGHIKLMNPQRSTVWY*";  // plaac.java:26

// ---------------------------------------------------------------------------------------------- Java formatting
// java.util.Formatter %.<d>f takes the SHORTEST decimal digits that identify the double (the digits
// Double.toString prints) and rounds THOSE half-up (sun.misc.FormattedFloatingDecimal.applyPrecision); C's printf
// rounds the exact binary value half-even.  NaN -> "NaN", infinities -> "Infinity" / "-Infinity".
std::string jfmt_exact(double x, int d)
{
    if (std::isnan(x)) return "NaN";
    if (std::isinf(x)) return x > 0 ? "Infinity" : "-Infinity";
    char sci[64];
    auto r = std::to_chars(sci, sci + sizeof(sci), std::fabs(x), std::chars_format::scientific);
    *r.ptr = 0;
    // sci = D[.DDDD]e[+-]XX
    std::string digits;
    const char* p = sci;
    for (; *p && *p != 'e'; p++)
        if (*p != '.') digits.push_back(*p);
    int exp10 = std::atoi(p + 1);  // value = 0.D1D2... * 10^(exp10+1)
    const int point = exp10 + 1;   // number of digits before the decimal point (may be <= 0)
    // digit at absolute decimal position q (q >= 0: q-th digit before the point from the left; fractional: index point+k)
    auto digit_at = [&](int idx) -> int { return (idx >= 0 && idx < (int)digits.size()) ? digits[idx] - '0' : 0; };
    const int keep = point + d;  // number of leading digits kept
    std::string out;             // kept digits, left-padded with zeros when point <= 0
    if (keep <= 0) {
        // everything is below the last printed place; round half up on the first dropped digit
        const bool up = (keep == 0) && digit_at(0) >= 5;
        out.assign((size_t)d + 1, '0');
        if (up) out.back() = '1';
    } else {
        for (int i = 0; i < keep; i++) out.push_back((char)('0' + digit_at(i)));
        if (digit_at(keep) >= 5) {
            int i = (int)out.size() - 1;
            while (i >= 0 && out[i] == '9') out[i--] = '0';
            if (i >= 0)
                out[i]++;
            else
                out.insert(out.begin(), '1');
        }
        // make sure there is at least one integer digit
        const int intdigits = (int)out.size() - d;
        if (intdigits <= 0) out.insert(0, (size_t)(1 - intdigits), '0');
    }
    std::string s;
    if (std::signbit(x)) s.push_back('-');
    s.append(out, 0, out.size() - d);
    if (d > 0) {
        s.push_back('.');
        s.append(out, out.size() - d, d);
    }
    return s;
}

// Fast path of the same rule.  Rounding the shortest digits half-up differs from rounding the exact binary value only
// when the shortest decimal form of x has exactly d+1 fractional digits and ends in 5 (a shorter form rounds to itself;
// with a longer form no (d+1)-digit boundary can lie between x and its shortest form, or that boundary would BE the
// shortest form).  Those x have x * 10^d within rounding noise of k + 0.5, so everything else goes through
// std::to_chars(fixed, d), which rounds the exact value correctly; candidates near k + 0.5 take the exact routine.
void put_fixed(std::string& out, double x, int d)
{
    static const double kPow10[] = {1, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9};
    const double ax = std::fabs(x);
    if (d >= 0 && d <= 9 && ax < 1e9) {  // (also false for NaN)
        const double y = ax * kPow10[d];
        const double f = y - std::floor(y);
        // y < 2e12: the half ulp of x and the rounding of the product move y by < 4.4e-4 together, below the margin
        if (y < 2e12 && std::fabs(f - 0.5) > 1e-3) {
            char buf[48];
            auto r = std::to_chars(buf, buf + sizeof(buf), x, std::chars_format::fixed, d);
            out.append(buf, (size_t)(r.ptr - buf));
            return;
        }
    }
    out += jfmt_exact(x, d);
}

std::string jfmt(double x, int d)
{
    std::string s;
    put_fixed(s, x, d);
    return s;
}

void put_int(std::string& out, long v)
{
    char buf[24];
    auto r = std::to_chars(buf, buf + sizeof(buf), v);
    out.append(buf, (size_t)(r.ptr - buf));
}

// Double.toString for the alpha echo of plaac.java:505 (plain notation for 1e-3 <= |x| < 1e7, else d.dddE[-]x).
std::string jdouble(double x)
{
    if (std::isnan(x)) return "NaN";
    if (std::isinf(x)) return x > 0 ? "Infinity" : "-Infinity";
    if (x == 0) return std::signbit(x) ? "-0.0" : "0.0";
    char buf[64];
    const double ax = std::fabs(x);
    std::string s = std::signbit(x) ? "-" : "";
    if (ax >= 1e-3 && ax < 1e7) {
        auto r = std::to_chars(buf, buf + sizeof(buf), ax, std::chars_format::fixed);
        *r.ptr = 0;
        s += buf;
        if (s.find('.') == std::string::npos) s += ".0";
        return s;
    }
    auto r = std::to_chars(buf, buf + sizeof(buf), ax, std::chars_format::scientific);
    *r.ptr = 0;
    std::string m(buf);
    const size_t e = m.find('e');
    std::string mant = m.substr(0, e);
    const int ex = std::atoi(m.c_str() + e + 1);
    if (mant.find('.') == std::string::npos) mant += ".0";
    return s + mant + "E" + std::to_string(ex);
}

// ---------------------------------------------------------------------------------------------- FASTA reader
// fastareader, plaac.java:4302-4375.  readLine semantics: \n, \r or \r\n end a line.  Sequence lines are NOT
// trimmed (the jar discards the result of line.trim()); a blank line ends the record and everything up to the next
// '>' line is skipped; the name is everything after '>' (trimmed only when found by hasmorefastas).
class FastaReader {
public:
    // The file is mapped and scanned in memory: one get() per character through an ifstream made the reader the slowest
    // part of the program (the jar reads the input twice -- background counts, then scoring -- and so does this host).
    explicit FastaReader(const std::string& path)
    {
        const int fd = ::open(path.c_str(), O_RDONLY);
        struct stat st;
        if (fd >= 0 && ::fstat(fd, &st) == 0 && S_ISREG(st.st_mode)) {
            good_ = true;
            size_ = (size_t)st.st_size;
            if (size_ > 0) {
                void* m = ::mmap(nullptr, size_, PROT_READ, MAP_PRIVATE, fd, 0);
                if (m == MAP_FAILED)
                    good_ = false;
                else {
                    data_ = (const char*)m;
                    ::madvise(m, size_, MADV_SEQUENTIAL);
                }
            }
        } else if (fd >= 0) {
            // not a regular file (a pipe, /dev/stdin): read it through
            good_ = true;
            char tmp[1 << 16];
            ssize_t k;
            while ((k = ::read(fd, tmp, sizeof(tmp))) > 0) own_.append(tmp, (size_t)k);
            data_ = own_.data();
            size_ = own_.size();
        }
        if (fd >= 0) ::close(fd);
        if (!good_) std::printf("# Couldn't open %s\n", path.c_str());
    }
    ~FastaReader()
    {
        if (data_ && own_.empty() && size_ > 0) ::munmap((void*)data_, size_);
    }
    FastaReader(const FastaReader&) = delete;
    FastaReader& operator=(const FastaReader&) = delete;
    bool hasmore()
    {
        if (!good_) return false;
        if (ondeck_) return true;
        std::string_view line;
        while (readline(line)) {
            if (!line.empty() && line[0] == '>') {
                name_ = trim(line).substr(1);
                return true;
            }
        }
        return false;
    }
    const std::string& name() const { return name_; }  // valid after hasmore() until the next next()
    // Reads the record's sequence; the NEXT record's name becomes current (as in the jar, the caller must take
    // name() before calling next()).
    void next(std::string& seq)
    {
        seq.clear();
        std::string_view line;
        while (readline(line)) {
            if (line.empty()) {
                ondeck_ = false;
                return;
            }
            if (line[0] == '>') {
                ondeck_ = true;
                name_.assign(line.substr(1));
                return;
            }
            seq.append(line);
        }
        ondeck_ = false;
    }

private:
    static std::string trim(std::string_view s)
    {
        size_t a = 0, b = s.size();
        while (a < b && (unsigned char)s[a] <= ' ') a++;  // String.trim(): code points <= U+0020
        while (b > a && (unsigned char)s[b - 1] <= ' ') b--;
        return std::string(s.substr(a, b - a));
    }
    // BufferedReader.readLine: a line ends with \n, \r or \r\n; the last line may end with the file
    bool readline(std::string_view& line)
    {
        if (pos_ >= size_) return false;
        const char* b = data_ + pos_;
        const char* e = data_ + size_;
        const char* p = b;
        while (p < e && *p != '\n' && *p != '\r') p++;
        line = std::string_view(b, (size_t)(p - b));
        if (p < e) p += (*p == '\r' && p + 1 < e && p[1] == '\n') ? 2 : 1;
        pos_ = (size_t)(p - data_);
        return true;
    }
    const char* data_ = nullptr;
    size_t size_ = 0, pos_ = 0;
    std::string own_;
    bool good_ = false, ondeck_ = false;
    std::string name_;
};

void strip_stop(std::string& s)
{
    if (!s.empty() && s.back() == '*') s.pop_back();  // plaac.java:758 / :624
}

// computeaafreq :1655-1666 + countaas :1698-1706 + isvalidprotein :1732-1739 (on the UNSTRIPPED sequence).
// The jar counts in 32-bit ints; this host uses 64-bit counters (identical below 2^31 residues per bin).
bool bg_counts_from_fasta(const std::string& path, double out[PLAAC_NAA])
{
    int64_t cnt[PLAAC_NAA] = {0};
    FastaReader fr(path);
    std::string seq;
    std::vector<uint8_t> codes;
    while (fr.hasmore()) {
        fr.next(seq);
        const size_t m = seq.size();
        if (m == 0) continue;  // the jar throws on aa[m-1]; skip instead
        codes.resize(m);
        plaac_encode_host(seq.data(), (int64_t)m, codes.data());
        bool valid = codes[m - 1] != 0;
        for (size_t i = 1; valid && i + 1 < m; i++) valid = codes[i] != 0 && codes[i] != 21;
        if (!valid) continue;
        for (size_t i = 0; i < m; i++) cnt[codes[i]]++;
    }
    for (int i = 0; i < PLAAC_NAA; i++) out[i] = (double)cnt[i];
    return true;
}

// read_aa_params :2684-2713: 22 lines "value [# name]".
void read_aa_params(const std::string& path, double out[PLAAC_NAA])
{
    for (int i = 0; i < PLAAC_NAA; i++) out[i] = 0;
    std::ifstream in(path);
    if (!in.good()) {
        std::printf("# Couldn't open %s\n", path.c_str());
        return;
    }
    std::string line;
    for (int i = 0; i < PLAAC_NAA && std::getline(in, line); i++) {
        char name[64] = {0}, hash[8] = {0};
        double v = 0;
        const int n = std::sscanf(line.c_str(), "%lf %7s %63s", &v, hash, name);
        if (n >= 1) out[i] = v;
        if (n >= 3 && name[0] != kAaNames[i])
            std::printf("# warning: %s does not have expected name in line%d\n", path.c_str(), i + 1);
    }
}

void print_aa_params(const double v[PLAAC_NAA])  // :2665-2670
{
    for (int i = 0; i < PLAAC_NAA; i++) std::printf("%s # %c\n", jfmt(v[i], 6).c_str(), kAaNames[i]);
}

std::string aaparams2string(const double* v)  // :2717-2723
{
    std::string s;
    for (int i = 0; i < PLAAC_NAA; i++) {
        s.push_back(kAaNames[i]);
        s += "=" + jfmt(v[i], 5) + ";";
    }
    return s;
}

// submatrix(int[],r1,r2) clamping rules (:1445-1456) + aa2string.
std::string aa_sub(const uint8_t* aa, int m, int r1, int r2)
{
    if (m <= 0) return "";
    if (r1 < 0) r1 = 0;
    if (r2 < r1) r2 = r1;
    if (r1 >= m) r1 = m - 1;
    if (r2 >= m) r2 = m - 1;
    std::string s;
    for (int i = r1; i <= r2; i++) s.push_back(kAaNames[aa[i]]);
    return s;
}

// Column documentation printed by -d (plaac.java:661-711); web/views/_plaac_headers.haml is generated from it.
const char* const kColumnDocs[] = {
    "SEQid: sequence name from fasta file",
    "MW: Michelitsh-Weissman [PNAS 2000] score --- maximum number of N + Q in window of at most 80 AA",
    "MWstart: index of start position of window with max MW score.",
    "MWend: index of end position of window with max MW score",
    "MWlen: length of window used for MW score [smaller of 80 and PROTlen].",
    "LLR: max sum of PLAAC log-likelihood ratios (base 4) in window of size c [NaN if PROTlen < c]",
    "LLRstart: index of start position of window with max LLR score [-1 if PROTlen < c]",
    "LLRend: index of end position of window with max LLR score [-1 if PROTlen < c]",
    "LLRlen: length of window used for LLR score [should be c]",
    "NLLR: normalized LLR score, i.e. LLR/LLRlen [NaN if PROTlen < c]",
    "VITmaxrun: maximum length of consecutive PrD state in Viterbi parse",
    "COREscore: max sum of PLAAC LLRs in window of size c contained entirely within Viterbi parse [NaN if VITmaxrun < c]",
    "COREstart: index of start position of window with max COREscore [-1 if VITmaxrun < c]",
    "COREend: index of end position of window with max COREscore [-2 if VITmaxrun < c]",
    "CORElen: length of window used for CORElen [should be either c or 0]",
    "PRDscore: sum of PLAAC LLRs in full region of Viterbi parse containing CORE region, if any [NaN otherwise].",
    "PRDstart: index of start position of window with PRDscore [-1 if VITmaxrun < c]",
    "PRDend: index of end position of window with PRDscore [-2 if VITmaxrun < c]",
    "PRDlen: length of window used for PRDscore",
    "PROTlen: number of AAs in protein, not including terminal stop codon if any.",
    "HMMall: log-likelihood ratio for sequence under two-state HMM vs. one-state background HMM",
    "HMMvit: log-likelihood ratio for sequence under Viterbi parse of two-state HMM vs. one-state background HMM",
    "COREaa: AA sequence at which COREscore is attained [- if VITmaxrun < c]",
    "STARTaa: first 15 AA of PRDaa [- if VITmaxrun < c]",
    "ENDaa: last 15 AA of PRDaa [- if VITmaxrun < c]",
    "PRDaa: AA sequence at which PRDscore is attained [- if VITmaxrun < c]",
    "FInumaa: number of AAs predicted to be disordered by FoldIndex [Prilusky et al, Bioinformatics, 2005] (exludes runs of under 5 AA)",
    "FImeanhydro: hydropathy score <H> for entire protein [Uversky et al, Proteins, 2000]",
    "FImeancharge: mean charge <R> for entire protein [Uversky et al, Proteins, 2000]",
    "FImeancombo: disorder score for entire protein: 2.785<H> - |<R>| - 1.151 [Uversky et al, Proteins, 2000]",
    "FImaxrun: length of longest run of predicted disorder by FoldIndex",
    "PAPAcombo: signed distance to PAPA decision surface [as in King et al Brain Res 2012]",
    "PAPAprop: maximal score of PAPA prion propensities (averges of averages) in region with negative FI score [Toombs et al MBC 2012]",
    "PAPAfi: FI score (averages of averages) at PAPAcen",
    "PAPAllr: PLAAC LLR score (average) at PAPAcen",
    "PAPAllr2: PLAAC LLR score (average of averages) at PAPAcen",
    "PAPAcen: index of center of window at which PAPAprop is obtained",
    "PAPAaa: AA sequence of width W centered at PAPAcen",
};

const char kSummaryHeader[] =
    "SEQid\tMW\tMWstart\tMWend\tMWlen\tLLR\tLLRstart\tLLRend\tLLRlen\tNLLR\tVITmaxrun\tCOREscore\tCOREstart\tCOREend\t"
    "CORElen\tPRDscore\tPRDstart\tPRDend\tPRDlen\tPROTlen\tHMMall\tHMMvit\tCOREaa\tSTARTaa\tENDaa\tPRDaa\tFInumaa\t"
    "FImeanhydro\tFImeancharge\tFImeancombo\tFImaxrun\tPAPAcombo\tPAPAprop\tPAPAfi\tPAPAllr\tPAPAllr2\tPAPAcen\tPAPAaa";

double inf2nan(double x) { return std::isinf(x) ? NAN : x; }  // :1008

struct Options {
    std::string inputfile, bgfile, bgfreqfile, fgfreqfile, plotlist, hmmdotfile;
    int corelength = 60, ww1 = 41, ww2 = 41, ww3 = 41, hmmtype = 1;
    double alpha = 1.0;
    bool printheaders = false, printparameters = true, adjustprolines = true;
    int gpus = 1, device = 0;
    int64_t batch_res = (int64_t)256 << 20;
    bool batch_set = false;  // --batch-mb given
    bool compat_F = false;
    bool gpu_ingest = false, host_reader = false;
    bool rank = false, rank_core_only = false;
    std::string variants_file;  // --variants
    bool saturate = false;      // --saturate
    std::string effects;        // --effects, as given
    bool effects_set = false;
    int32_t effects_mask = 0;   // PLAAC_EFFECT_* bits of --effects
    std::string segments_file;  // --segments
    FILE* seg_out = nullptr;    // ... open
    std::string null_file;      // --null
    FILE* null_out = nullptr;   // ... open
    int64_t replicates = 0;     // --replicates
    uint64_t seed = 0;          // --seed
    std::string null_columns = "COREscore,LLR,HMMall";  // --null-columns, as given
    bool replicates_set = false, seed_set = false, null_columns_set = false;
    const char* stop_hits_arg = nullptr;  // --stop-hits, as given
    int64_t stop_hits = 0;                // ... parsed (0: the fixed null)
    int32_t null_mask = 0;      // plaac_null.columns of --null-columns
};

// --effects names, bit k = PLAAC_EFFECT_* bit k (the doubles of plaac_summary in declaration order, then COREchange)
const char* const kEffectNames[] = {"LLR",          "COREscore",   "PRDscore",  "HMMall",   "HMMvit",
                                    "FImeanhydro",  "FImeancharge", "FImeancombo", "PAPAcombo", "PAPAprop",
                                    "PAPAfi",       "PAPAllr",     "PAPAllr2",  "COREchange"};
constexpr int kEffectCoreChange = 13;
// --null-columns names: those of --effects, with hasCORE (replicates with a CORE) for bit 13
const char* const kNullNames[] = {"LLR",          "COREscore",   "PRDscore",  "HMMall",   "HMMvit",
                                  "FImeanhydro",  "FImeancharge", "FImeancombo", "PAPAcombo", "PAPAprop",
                                  "PAPAfi",       "PAPAllr",     "PAPAllr2",  "hasCORE"};

// Comma-separated column names of option `opt` (--effects or --null-columns) -> mask; 0 after printing the message.
int32_t parse_columns(const std::string& list, const char* opt, const char* const (&names)[14])
{
    int32_t mask = 0;
    size_t a = 0;
    while (a <= list.size()) {
        size_t b = list.find(',', a);
        if (b == std::string::npos) b = list.size();
        const std::string name = list.substr(a, b - a);
        int k = 0;
        while (k <= kEffectCoreChange && name != names[k]) k++;
        if (k > kEffectCoreChange) {
            if (name.empty())
                std::fprintf(stderr, "plaac: %s: empty column name in '%s'\n", opt, list.c_str());
            else
                std::fprintf(stderr, "plaac: %s: unknown column '%s'\n", opt, name.c_str());
            std::fprintf(stderr, "plaac: %s takes a comma-separated list of", opt);
            for (int j = 0; j <= kEffectCoreChange; j++) std::fprintf(stderr, " %s", names[j]);
            std::fprintf(stderr, "\n");
            return 0;
        }
        mask |= 1 << k;
        a = b + 1;
    }
    return mask;
}

struct Scorers {
    std::vector<plaac_ctx*> ctx;
    ~Scorers()
    {
        for (auto c : ctx) plaac_destroy(c);
    }
};

struct Batch {
    std::vector<std::string> names, ids;  // ids: ORDER column of the per-residue table
    std::vector<uint8_t> codes;
    std::vector<int64_t> offsets{0};
    void clear()
    {
        names.clear();
        ids.clear();
        codes.clear();
        offsets.assign(1, 0);
    }
    int64_t nprot() const { return (int64_t)names.size(); }
    void add(const std::string& name, const std::string& id, const std::string& seq)
    {
        const size_t o = codes.size();
        codes.resize(o + seq.size());
        plaac_encode_host(seq.data(), (int64_t)seq.size(), codes.data() + o);
        offsets.push_back((int64_t)codes.size());
        names.push_back(name);
        ids.push_back(id);
    }
};

int die(const Scorers& S, int rc, const char* what)
{
    const char* msg = "";
    for (auto c : S.ctx)
        if (*plaac_last_error(c)) msg = plaac_last_error(c);
    if (!*msg) msg = plaac_last_error(nullptr);
    std::fprintf(stderr, "plaac: %s failed (%d): %s\n", what, rc, msg);
    return 2;
}

// Substitutions of a sequence variant (positions ascending): the string columns of its row are the wild type's cut with
// these patched in, so a row costs no more than its printed residues.
struct SubList {
    const int32_t* pos = nullptr;
    const uint8_t* code = nullptr;
    int64_t n = 0;
};

// One row of the summary table (plaac.java:899-945) appended to `out`.
void aa_sub_into(std::string& out, const uint8_t* aa, int m, int r1, int r2, const SubList& subs = SubList())
{
    if (m <= 0) return;
    if (r1 < 0) r1 = 0;
    if (r2 < r1) r2 = r1;
    if (r1 >= m) r1 = m - 1;
    if (r2 >= m) r2 = m - 1;
    const size_t o = out.size();
    for (int i = r1; i <= r2; i++) out.push_back(kAaNames[aa[i]]);
    for (const int32_t* p = std::lower_bound(subs.pos, subs.pos + subs.n, r1); p < subs.pos + subs.n && *p <= r2; p++)
        out[o + (size_t)(*p - r1)] = kAaNames[subs.code[p - subs.pos]];
}

void append_summary_row(const Options& o, std::string_view name, const plaac_summary& s, const uint8_t* aa, std::string& out,
                        const SubList& subs = SubList())
{
    const int n = s.prot_len;
    if (n < 1) return;  // :762
    const int llrlen = s.llr_end - s.llr_start + 1;
    const double llr = inf2nan(s.llr);
    const int prdlen = s.prd_end - s.prd_start + 1;
    out.append(name);
    auto I = [&](long v) { out.push_back('\t'), put_int(out, v); };
    auto F = [&](double v) { out.push_back('\t'), put_fixed(out, v, 3); };
    I(s.mw_score), I(s.mw_start + 1), I(s.mw_end + 1), I(s.mw_end - s.mw_start + 1);
    F(llr), I(s.llr_start + 1), I(s.llr_end + 1), I(llrlen), F(llr / (double)llrlen), I(s.vit_maxrun);
    F(inf2nan(s.core_score)), I(s.core_start + 1), I(s.core_end + 1), I(s.core_end - s.core_start + 1);
    F(s.prd_score), I(s.prd_start + 1), I(s.prd_end + 1), I(prdlen), I(n), F(s.hmm_all), F(s.hmm_vit);
    if (prdlen >= o.corelength) {  // :915-931
        out.push_back('\t'), aa_sub_into(out, aa, n, s.core_start, s.core_end, subs);
        out.push_back('\t'), aa_sub_into(out, aa, n, s.prd_start, s.prd_start + 14, subs);
        out.push_back('\t'), aa_sub_into(out, aa, n, s.prd_end - 14, s.prd_end, subs);
        out.push_back('\t'), aa_sub_into(out, aa, n, s.prd_start, s.prd_end, subs);
    } else
        out += "\t-\t-\t-\t-";
    I(s.fi_numaa), F(s.fi_meanhydro), F(s.fi_meancharge), F(s.fi_meancombo), I(s.fi_maxrun);
    F(inf2nan(s.papa_combo)), F(s.papa_prop), F(s.papa_fi), F(s.papa_llr), F(s.papa_llr2), I(s.papa_center + 1);
    out.push_back('\t'), aa_sub_into(out, aa, n, s.papa_center - o.ww2 / 2, s.papa_center + o.ww2 / 2, subs);
    out.push_back('\n');
}

void print_summary_row(const Options& o, const std::string& name, const plaac_summary& s, const uint8_t* aa, std::string& line)
{
    line.clear();
    append_summary_row(o, name, s, aa, line);
    std::fwrite(line.data(), 1, line.size(), stdout);
}

// --segments: the records of the batch and the segments of their Viterbi parses; the segment table is written here.
int score_segment_batch(const Options& o, Scorers& S, Batch& B, std::vector<plaac_summary>& sum)
{
    const int64_t np = B.nprot();
    std::vector<int64_t> first((size_t)np + 1);
    std::vector<int32_t> st, en;
    std::vector<double> sc;
    plaac_segments G = {};
    for (int64_t cap = np;;) {  // (a second pass only for a batch with more segments than records)
        st.resize((size_t)std::max<int64_t>(cap, 1)), en.resize(st.size()), sc.resize(st.size());
        G = {cap, first.data(), st.data(), en.data(), sc.data(), 0};
        const int rc = plaac_score_segments(S.ctx[0], B.codes.data(), B.offsets.data(), np, sum.data(), &G);
        if (rc != PLAAC_OK) return die(S, rc, "plaac_score_segments");
        if (G.count <= cap) break;
        cap = G.count;
    }
    std::string out;
    for (int64_t i = 0; i < np; i++) {
        const plaac_summary& r = sum[(size_t)i];
        for (int64_t k = first[(size_t)i]; k < first[(size_t)i + 1]; k++) {
            out.append(B.names[(size_t)i]);
            auto I = [&](long v) { out.push_back('\t'), put_int(out, v); };
            I(st[(size_t)k] + 1), I(en[(size_t)k] + 1), I(en[(size_t)k] - st[(size_t)k] + 1);
            out.push_back('\t'), put_fixed(out, sc[(size_t)k], 3);
            I(st[(size_t)k] == r.prd_start && en[(size_t)k] == r.prd_end ? 1 : 0);
            out.push_back('\n');
        }
    }
    if (std::fwrite(out.data(), 1, out.size(), o.seg_out) != out.size() || std::fflush(o.seg_out) != 0) {
        std::fprintf(stderr, "plaac: cannot write %s\n", o.segments_file.c_str());
        return 2;
    }
    return 0;
}

// --null: the records of the batch (plaac_score_shuffles' observed records) and, per printed record in record order,
// the counts of its shuffles that reach it and the p-values (1 + n) / (1 + K); the table is written here.
int score_null_batch(const Options& o, Scorers& S, Batch& B, std::vector<plaac_summary>& sum)
{
    const int64_t np = B.nprot();
    const int k = __builtin_popcount((unsigned)o.null_mask);
    std::vector<int64_t> counts((size_t)np * (size_t)k);
    std::vector<int64_t> scored(o.stop_hits > 0 ? counts.size() : 0);
    plaac_null N = {};
    N.replicates = o.replicates;
    N.seed = o.seed;
    N.columns = o.null_mask;
    N.nsel = -1;
    N.counts = counts.data();
    if (o.stop_hits > 0) {
        const int rc = plaac_score_shuffles_seq(S.ctx[0], B.codes.data(), B.offsets.data(), np, &N, o.stop_hits, scored.data(),
                                                sum.data());
        if (rc != PLAAC_OK) return die(S, rc, "plaac_score_shuffles_seq");
    } else {
        const int rc = plaac_score_shuffles(S.ctx[0], B.codes.data(), B.offsets.data(), np, &N, sum.data());
        if (rc != PLAAC_OK) return die(S, rc, "plaac_score_shuffles");
    }
    std::string out;
    char buf[64];
    for (int64_t i = 0; i < np; i++) {
        const plaac_summary& r = sum[(size_t)i];
        if (r.prot_len < 1 || (o.rank_core_only && !(r.core_score == r.core_score))) continue;  // (rows not printed)
        out.append(B.names[(size_t)i]);
        if (o.stop_hits == 0) out.push_back('\t'), put_int(out, (long)o.replicates);
        int c = 0;
        for (int b = 0; b <= kEffectCoreChange; b++) {
            if (!((o.null_mask >> b) & 1)) continue;
            const size_t at = (size_t)i * (size_t)k + (size_t)c++;
            const int64_t n = counts[at];
            if (o.stop_hits > 0) out.push_back('\t'), put_int(out, (long)scored[at]);
            out.push_back('\t'), put_int(out, (long)n);
            if (b != kEffectCoreChange) {
                const double p = o.stop_hits > 0 && n == o.stop_hits ? (double)n / (double)scored[at]
                                                                      : (double)(1 + n) / (double)(1 + o.replicates);
                std::snprintf(buf, sizeof(buf), "\t%.6g", p);
                out += buf;
            }
        }
        out.push_back('\n');
    }
    if (std::fwrite(out.data(), 1, out.size(), o.null_out) != out.size() || std::fflush(o.null_out) != 0) {
        std::fprintf(stderr, "plaac: cannot write %s\n", o.null_file.c_str());
        return 2;
    }
    return 0;
}

int score_summary_batch(const Options& o, Scorers& S, Batch& B)
{
    if (B.nprot() == 0) return 0;
    std::vector<plaac_summary> sum((size_t)B.nprot());
    if (o.seg_out) {
        if (const int rs = score_segment_batch(o, S, B, sum)) return rs;
    } else if (o.null_out) {
        if (const int rs = score_null_batch(o, S, B, sum)) return rs;
    } else {
        const int rc = plaac_score_multi(S.ctx.data(), (int)S.ctx.size(), B.codes.data(), B.offsets.data(), B.nprot(),
                                         sum.data(), nullptr);
        if (rc != PLAAC_OK) return die(S, rc, "plaac_score");
    }
    std::string line;
    if (o.rank) {
        std::vector<int32_t> order((size_t)B.nprot());
        int64_t ncore = 0;
        const int rr = plaac_rank(S.ctx[0], sum.data(), B.nprot(), 0, order.data(), &ncore);
        if (rr != PLAAC_OK) return die(S, rr, "plaac_rank");
        const int64_t nshow = o.rank_core_only ? ncore : B.nprot();
        for (int64_t k = 0; k < nshow; k++) {
            const size_t i = (size_t)order[(size_t)k];
            print_summary_row(o, B.names[i], sum[i], B.codes.data() + B.offsets[i], line);
        }
        B.clear();
        return 0;
    }
    for (int64_t i = 0; i < B.nprot(); i++)
        print_summary_row(o, B.names[(size_t)i], sum[(size_t)i], B.codes.data() + B.offsets[(size_t)i], line);
    B.clear();
    return 0;
}

// ---------------------------------------------------------------------------------------------- file-to-table fast path
// The whole file is mapped once and cut into pieces that end right before a '>' line; every piece goes to the GPU as
// raw bytes and is parsed, encoded, counted (background) and scored there (plaac_score_fasta: reader semantics of
// fastareader :4302-4375, tested against the host reader).  The host only cuts, formats the rows on all its threads
// into one buffer per piece, and writes.  Pieces go round-robin to the GPUs of --gpus.
// The jar trims a record name only when the reader found it after an empty line or at the file start (:4362); for the
// first record of a later piece that context lies in the text before the piece, which is looked at directly.
struct MappedFile {
    const char* data = nullptr;
    size_t size = 0;
    bool good = false, mapped = false;
    std::string own;
    explicit MappedFile(const std::string& path)
    {
        const int fd = ::open(path.c_str(), O_RDONLY);
        struct stat st;
        if (fd >= 0 && ::fstat(fd, &st) == 0 && S_ISREG(st.st_mode)) {
            good = true;
            size = (size_t)st.st_size;
            if (size > 0) {
                void* m = ::mmap(nullptr, size, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
                if (m == MAP_FAILED)
                    good = false;
                else {
                    data = (const char*)m;
                    mapped = true;
                }
            }
        } else if (fd >= 0) {  // a pipe, /dev/stdin: read it through
            good = true;
            char tmp[1 << 16];
            ssize_t k;
            while ((k = ::read(fd, tmp, sizeof(tmp))) > 0) own.append(tmp, (size_t)k);
            data = own.data();
            size = own.size();
        }
        if (fd >= 0) ::close(fd);
    }
    ~MappedFile()
    {
        if (mapped) ::munmap((void*)data, size);
    }
    MappedFile(const MappedFile&) = delete;
    MappedFile& operator=(const MappedFile&) = delete;
};

// PLAAC_CLI_TIMING=1: phase times on stderr
struct Phase {
    static double now()
    {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec + ts.tv_nsec * 1e-9;
    }
    static bool on()
    {
        static const bool v = getenv("PLAAC_CLI_TIMING") != nullptr;
        return v;
    }
    static void mark(const char* what)
    {
        static double t0 = now(), last = t0;
        if (!on()) return;
        const double t = now();
        std::fprintf(stderr, "[plaac %8.3f s  +%7.3f] %s\n", t - t0, t - last, what);
        last = t;
    }
};

int host_threads()
{
    cpu_set_t set;
    int n = 0;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
    if (n <= 0) n = (int)std::thread::hardware_concurrency();
    return std::max(1, std::min(n, 64));
}

// f(tid, lo, hi) over [0, n) cut into one contiguous range per thread
template <class F>
void parallel_ranges(size_t n, int nthreads, F f)
{
    nthreads = (int)std::max<size_t>(1, std::min<size_t>((size_t)nthreads, n));
    std::vector<std::thread> th;
    const size_t per = (n + nthreads - 1) / nthreads;
    for (int t = 1; t < nthreads; t++) {
        const size_t lo = std::min(n, t * per), hi = std::min(n, lo + per);
        if (hi > lo) th.emplace_back([=] { f(t, lo, hi); });
    }
    f(0, 0, std::min(n, per));
    for (auto& t : th) t.join();
}

// Is the record that starts at text[pos] (a '>' at a line start) found by nextfasta in the jar, i.e. does the latest
// header-or-empty line before it open a record?  Then its name is printed untrimmed.
bool opened_by_previous_record(const char* text, size_t pos)
{
    size_t e = pos;  // a line start: the text before it ends with a line terminator
    while (e > 0) {
        size_t le = e;  // end of the previous line without its terminator (\n, \r or \r\n as BufferedReader.readLine sees them)
        if (text[le - 1] == '\n') {
            le--;
            if (le > 0 && text[le - 1] == '\r') le--;
        } else if (text[le - 1] == '\r')
            le--;
        size_t ls = le;
        while (ls > 0 && text[ls - 1] != '\n' && text[ls - 1] != '\r') ls--;
        if (ls == le) return false;        // an empty line: the reader is between records
        if (text[ls] == '>') return true;  // a header line: the record it opened is still open
        e = ls;
    }
    return false;  // file start: hasmorefastas finds the first record (trimmed)
}

struct PieceBuffers {  // reused from piece to piece (never zero-filled)
    size_t cap_rec = 0, cap_bytes = 0;
    std::unique_ptr<plaac_summary[]> sum;
    std::unique_ptr<uint8_t[]> codes, flags;
    std::unique_ptr<int64_t[]> offsets, npos;
    std::unique_ptr<int32_t[]> nlen, order;
    void reserve(size_t nrec, size_t nbytes)
    {
        if (nrec > cap_rec) {
            cap_rec = nrec + nrec / 8 + 16;
            sum.reset(new plaac_summary[cap_rec]);
            flags.reset(new uint8_t[cap_rec + 16]);
            offsets.reset(new int64_t[cap_rec + 1]);
            npos.reset(new int64_t[cap_rec]);
            nlen.reset(new int32_t[cap_rec]);
            order.reset(new int32_t[cap_rec]);
        }
        if (nbytes > cap_bytes) {
            cap_bytes = nbytes + nbytes / 8 + 64;
            codes.reset(new uint8_t[cap_bytes]);
        }
    }
};

struct PieceResult {
    std::vector<std::string> parts;  // the rows, one string per formatting thread, in order
    double bg[PLAAC_NAA] = {0};
    int rc = 0;
    int64_t nrec = 0, nshow = 0;
    bool ranked = false;
};

// GPU stage of one piece [lo, hi) of the text on ctx: parse + score (+ rank) on the GPU; results in B.
void piece_gpu(const Options& o, plaac_ctx* ctx, const char* text, size_t lo, size_t hi, bool count_only, int nthreads,
               PieceBuffers& B, PieceResult& R)
{
    const size_t nbytes = hi - lo;
    // upper bound of the record count: '>' characters (counted on all threads; memchr runs at memory speed)
    std::vector<size_t> part((size_t)nthreads, 0);
    parallel_ranges(nbytes, nthreads, [&](int t, size_t a, size_t b) {
        size_t c = 0;
        const char* p = text + lo + a;
        const char* e = text + lo + b;
        while (p < e && (p = (const char*)memchr(p, '>', (size_t)(e - p)))) c++, p++;
        part[(size_t)t] = c;
    });
    size_t maxrec = 1;
    for (size_t c : part) maxrec += c;
    B.reserve(maxrec, nbytes + 16);
    memset(B.flags.get(), 0, maxrec + 8);
    plaac_fasta_index idx;
    R.rc = plaac_score_fasta(ctx, text + lo, (int64_t)nbytes, (int64_t)maxrec, B.sum.get(), B.codes.get(), B.offsets.get(),
                             B.npos.get(), B.nlen.get(), B.flags.get(), &idx, R.bg);
    Phase::mark("piece: plaac_score_fasta");
    if (R.rc != PLAAC_OK || count_only) return;
    R.nrec = R.nshow = idx.nrec;
    if (o.rank && idx.nrec > 0) {
        int64_t ncore = 0;
        R.rc = plaac_rank(ctx, B.sum.get(), idx.nrec, 0, B.order.get(), &ncore);
        if (R.rc != PLAAC_OK) return;
        R.ranked = true;
        if (o.rank_core_only) R.nshow = ncore;
    }
}

// Host stage: the rows of the piece, formatted on `nthreads` threads.
void piece_format(const Options& o, const char* text, size_t lo, int nthreads, const PieceBuffers& B, PieceResult& R)
{
    if (R.rc != PLAAC_OK || R.nshow <= 0) return;
    const int32_t* order = R.ranked ? B.order.get() : nullptr;
    const bool first_untrimmed = lo > 0 && opened_by_previous_record(text, lo);
    R.parts.assign((size_t)nthreads, std::string());
    parallel_ranges((size_t)R.nshow, nthreads, [&](int t, size_t a, size_t b) {
        std::string& s = R.parts[(size_t)t];
        s.reserve((b - a) * 320);
        for (size_t k = a; k < b; k++) {
            const size_t r = order ? (size_t)order[k] : k;
            std::string_view name(text + lo + (size_t)B.npos[r], (size_t)B.nlen[r]);
            bool trim = (B.flags[r] & 1) != 0;
            if (r == 0 && first_untrimmed) trim = false;  // found by nextfasta in the jar: untrimmed
            if (trim)
                while (!name.empty() && (unsigned char)name.back() <= ' ') name.remove_suffix(1);
            append_summary_row(o, name, B.sum[r], B.codes.get() + B.offsets[r], s);
        }
    });
    Phase::mark("piece: rows formatted");
}

// Piece boundaries: every piece ends right before a '>' that starts a line (or at the end of the text).
std::vector<size_t> cut_pieces(const char* text, size_t size, size_t piece)
{
    std::vector<size_t> cuts{0};
    size_t start = 0;
    while (start < size) {
        size_t want = start + piece;
        if (want >= size) {
            cuts.push_back(size);
            break;
        }
        // last record start in (start, want]; if there is none, the first one after want
        size_t cut = 0;
        for (size_t k = want; k > start + 1; k--)
            if (text[k] == '>' && (text[k - 1] == '\n' || text[k - 1] == '\r')) {
                cut = k;
                break;
            }
        if (cut == 0) {
            cut = size;
            const char* p = text + want;
            const char* e = text + size;
            while (p < e && (p = (const char*)memchr(p, '>', (size_t)(e - p)))) {
                if (p[-1] == '\n' || p[-1] == '\r') {
                    cut = (size_t)(p - text);
                    break;
                }
                p++;
            }
        }
        cuts.push_back(cut);
        start = cut;
    }
    if (cuts.size() == 1) cuts.push_back(size);
    return cuts;
}

// Runs all pieces.  count_only: background counts only (bg_total).  sink(rows of one formatting thread) is called in
// output order from the calling thread.  One GPU: the GPU stage of piece k+1 runs on a second host thread while this
// thread formats and hands over piece k.  Several GPUs: piece k on ctx k % G, one host thread per ctx.
template <class Sink>
int score_fasta_gpu(const Options& o, Scorers& S, const MappedFile& F, bool count_only, double* bg_total, Sink sink)
{
    // Piece size: --batch-mb if given; else 64 MiB of text, which pipelines better than one 256 MiB piece after another
    // (measured, 1.5 GB file: 0.95 s instead of 1.25 s after the driver's start-up); a ranked table keeps the larger
    // default, because a file that fits one piece is ranked as a whole.
    const int64_t piece = (o.batch_set || o.rank) ? o.batch_res : std::min<int64_t>(o.batch_res, (int64_t)64 << 20);
    const std::vector<size_t> cuts = cut_pieces(F.data, F.size, (size_t)std::max<int64_t>(piece, 1 << 20));
    const size_t npieces = cuts.size() - 1;
    const int G = (int)S.ctx.size();
    const int nthreads = std::max(1, host_threads() / std::max(1, std::min<int>(G, (int)npieces)));
    auto hand_over = [&](PieceResult& R) -> int {
        if (R.rc != PLAAC_OK) return die(S, R.rc, "plaac_score_fasta");
        if (bg_total)
            for (int i = 0; i < PLAAC_NAA; i++) bg_total[i] += R.bg[i];
        if (!count_only)
            for (auto& p : R.parts) sink(p);
        return 0;
    };
    if (G <= 1 || npieces <= 1) {
        PieceBuffers B[2];
        PieceResult R[2];
        piece_gpu(o, S.ctx[0], F.data, cuts[0], cuts[1], count_only, nthreads, B[0], R[0]);
        for (size_t k = 0; k < npieces; k++) {
            const int cur = (int)(k & 1), nxt = cur ^ 1;
            std::thread ahead;
            if (k + 1 < npieces && R[cur].rc == PLAAC_OK) {
                R[nxt] = PieceResult();
                ahead = std::thread([&, k, nxt] {
                    piece_gpu(o, S.ctx[0], F.data, cuts[k + 1], cuts[k + 2], count_only, nthreads, B[nxt], R[nxt]);
                });
            }
            if (!count_only) piece_format(o, F.data, cuts[k], nthreads, B[cur], R[cur]);
            const int rc = hand_over(R[cur]);
            if (ahead.joinable()) ahead.join();
            if (rc) return rc;
        }
        return 0;
    }
    std::vector<PieceResult> res(npieces);
    std::vector<std::thread> th;
    for (int g = 0; g < G; g++)
        th.emplace_back([&, g] {
            PieceBuffers B;
            for (size_t k = (size_t)g; k < npieces; k += (size_t)G) {
                piece_gpu(o, S.ctx[(size_t)g], F.data, cuts[k], cuts[k + 1], count_only, nthreads, B, res[k]);
                if (!count_only) piece_format(o, F.data, cuts[k], nthreads, B, res[k]);
            }
        });
    for (auto& t : th) t.join();
    for (size_t k = 0; k < npieces; k++) {
        const int rc = hand_over(res[k]);
        if (rc) return rc;
    }
    return 0;
}

int score_residue_batch(const Options&, Scorers& S, Batch& B)
{
    if (B.nprot() == 0) return 0;
    const size_t N = (size_t)B.offsets.back();
    std::vector<uint8_t> u8(2 * N + 1);
    std::vector<double> f64(10 * N + 1);
    plaac_residue_out r;
    r.vit = u8.data();
    r.map = u8.data() + N;
    double** f[10] = {&r.charge, &r.hydro, &r.fi, &r.plaac, &r.papa, &r.fix2, &r.plaacx2, &r.papax2, &r.post_bg, &r.post_prd};
    for (int k = 0; k < 10; k++) *f[k] = f64.data() + (size_t)k * N;
    const int rc = plaac_score_multi(S.ctx.data(), (int)S.ctx.size(), B.codes.data(), B.offsets.data(), B.nprot(), nullptr, &r);
    if (rc != PLAAC_OK) return die(S, rc, "plaac_score");
    std::string line;
    for (int64_t p = 0; p < B.nprot(); p++) {
        const int64_t lo = B.offsets[(size_t)p], hi = B.offsets[(size_t)p + 1];
        for (int64_t t = lo; t < hi; t++) {  // :635-643
            line.clear();
            line += B.ids[(size_t)p] + "\t" + B.names[(size_t)p] + "\t" + std::to_string(t - lo + 1) + "\t";
            line.push_back(kAaNames[B.codes[(size_t)t]]);
            line += "\t" + std::to_string((int)r.vit[t]) + "\t" + std::to_string((int)r.map[t]) + "\t";
            line += jfmt(r.charge[t], 4) + "\t" + jfmt(r.hydro[t], 4) + "\t" + jfmt(r.fi[t], 8) + "\t" + jfmt(r.plaac[t], 4) + "\t" +
                    jfmt(r.papa[t], 8) + "\t" + jfmt(r.fix2[t], 8) + "\t" + jfmt(r.plaacx2[t], 4) + "\t" + jfmt(r.papax2[t], 8);
            line += "\t" + jfmt(r.post_bg[t], 4) + "\t" + jfmt(r.post_prd[t], 4) + "\n";
            std::fwrite(line.data(), 1, line.size(), stdout);
        }
        std::puts("########################################################");  // :645
    }
    B.clear();
    return 0;
}

// readhashtable :1866-1893 for the plot list: name [\t synonym]; ORDER = 1-based line number.
void read_plot_list(const std::string& path, std::map<std::string, std::string>& syn, std::map<std::string, std::string>& order)
{
    std::ifstream in(path);
    if (!in.good()) {
        std::printf("# Couldn't open %s\n", path.c_str());
        return;
    }
    std::string line;
    int i = 1;
    while (std::getline(in, line)) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        const size_t tab = line.find('\t');
        const std::string key = line.substr(0, tab);
        std::string val = key;
        if (tab != std::string::npos) {
            const size_t tab2 = line.find('\t', tab + 1);
            val = line.substr(tab + 1, tab2 == std::string::npos ? std::string::npos : tab2 - tab - 1);
        }
        syn[key] = val;
        order[key] = std::to_string(i);
        i++;
    }
}

// ---------------------------------------------------------------------------------------------- sequence variants
// One line of a --variants file.
struct VariantLine {
    int line = 0;
    std::string spec;                  // upper-cased, as printed after "<name>:"
    std::vector<int32_t> pos;          // 0-based, ascending
    std::vector<uint8_t> ref, alt;     // codes
};

struct VariantFile {
    std::vector<VariantLine> lines;
    std::map<std::string, std::vector<int>> by_id;  // SEQid -> indices into lines, in file order
    std::map<std::string, bool> matched;
};

int letter_code(char c)
{
    const char u = (char)std::toupper((unsigned char)c);
    const char* p = std::strchr(kAaNames, u);
    return (u && p) ? (int)(p - kAaNames) : -1;
}

// Syntax only (needs no record and no device); false after printing the message.
bool read_variant_file(const std::string& path, VariantFile& V)
{
    std::ifstream in(path);
    if (!in.good()) {
        std::fprintf(stderr, "plaac: cannot open variant file %s\n", path.c_str());
        return false;
    }
    std::string line;
    for (int ln = 1; std::getline(in, line); ln++) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (line.empty()) continue;
        auto bad = [&](const std::string& why) {
            std::fprintf(stderr, "plaac: %s line %d: %s\n", path.c_str(), ln, why.c_str());
            return false;
        };
        const size_t tab = line.find('\t');
        if (tab == std::string::npos || tab == 0) return bad("expected SEQid<TAB>spec");
        VariantLine L;
        L.line = ln;
        L.spec = line.substr(tab + 1);
        for (char& c : L.spec) c = (char)std::toupper((unsigned char)c);
        if (L.spec != "WT") {
            std::vector<std::pair<int32_t, std::pair<uint8_t, uint8_t>>> subs;
            size_t a = 0;
            while (a <= L.spec.size()) {
                size_t b = L.spec.find(',', a);
                if (b == std::string::npos) b = L.spec.size();
                const std::string tok = L.spec.substr(a, b - a);
                if (tok.size() < 3) return bad("substitution '" + tok + "' is not <ref><pos><alt>");
                const int r = letter_code(tok.front()), t = letter_code(tok.back());
                if (r < 0 || t < 0) return bad("unknown residue letter in '" + tok + "'");
                const std::string num = tok.substr(1, tok.size() - 2);
                long long p = 0;
                const auto res = std::from_chars(num.data(), num.data() + num.size(), p);
                if (res.ec != std::errc() || res.ptr != num.data() + num.size() || p < 1 || p > 0x7fffffff)
                    return bad("substitution '" + tok + "' has no valid 1-based position");
                subs.push_back({(int32_t)(p - 1), {(uint8_t)r, (uint8_t)t}});
                a = b + 1;
            }
            std::sort(subs.begin(), subs.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
            for (size_t k = 0; k < subs.size(); k++) {
                if (k > 0 && subs[k].first == subs[k - 1].first)
                    return bad("position " + std::to_string(subs[k].first + 1) + " is substituted twice");
                L.pos.push_back(subs[k].first);
                L.ref.push_back(subs[k].second.first);
                L.alt.push_back(subs[k].second.second);
            }
        }
        const std::string id = line.substr(0, tab);
        V.by_id[id].push_back((int)V.lines.size());
        V.matched[id] = false;
        V.lines.push_back(std::move(L));
    }
    return true;
}

// Variants of the current batch over its reference records, and the names of their rows.
struct VariantBatch {
    Batch ref;
    std::vector<int32_t> protein;
    std::vector<int64_t> first_sub{0};
    std::vector<int32_t> pos;
    std::vector<uint8_t> code;
    std::vector<std::string> rows;
    int64_t nres = 0;
    void clear()
    {
        ref.clear();
        protein.clear();
        first_sub.assign(1, 0);
        pos.clear();
        code.clear();
        rows.clear();
        nres = 0;
    }
};

// --effects: one row per variant, its name and the changes of the selected columns.
int score_effect_batch(const Options& o, Scorers& S, VariantBatch& B)
{
    const int64_t nvar = (int64_t)B.protein.size();
    const int k = __builtin_popcount((unsigned)o.effects_mask);
    std::vector<double> eff((size_t)nvar * (size_t)k);
    const plaac_variants V = {nvar, B.protein.data(), B.first_sub.data(), B.pos.data(), B.code.data()};
    const int rc = plaac_score_variant_effects(S.ctx[0], B.ref.codes.data(), B.ref.offsets.data(), B.ref.nprot(), &V,
                                               o.effects_mask, eff.data(), nullptr);
    if (rc != PLAAC_OK) return die(S, rc, "plaac_score_variant_effects");
    const bool last_is_core = (o.effects_mask >> kEffectCoreChange) & 1;  // (the highest bit: the last column)
    std::string out;
    for (int64_t v = 0; v < nvar; v++) {
        out += B.rows[(size_t)v];
        const double* e = eff.data() + (size_t)v * (size_t)k;
        for (int c = 0; c < k; c++) {
            out.push_back('\t');
            if (last_is_core && c == k - 1)
                put_int(out, (long)e[c]);
            else
                put_fixed(out, e[c], 3);
        }
        out.push_back('\n');
        if (out.size() >= ((size_t)1 << 20)) {
            std::fwrite(out.data(), 1, out.size(), stdout);
            out.clear();
        }
    }
    std::fwrite(out.data(), 1, out.size(), stdout);
    B.clear();
    return 0;
}

int score_variant_batch(const Options& o, Scorers& S, VariantBatch& B)
{
    const int64_t nvar = (int64_t)B.protein.size();
    if (nvar == 0) {
        B.clear();
        return 0;
    }
    if (o.effects_mask) return score_effect_batch(o, S, B);
    std::vector<plaac_summary> sum((size_t)nvar);
    const plaac_variants V = {nvar, B.protein.data(), B.first_sub.data(), B.pos.data(), B.code.data()};
    const int rc = plaac_score_variants(S.ctx[0], B.ref.codes.data(), B.ref.offsets.data(), B.ref.nprot(), &V, sum.data());
    if (rc != PLAAC_OK) return die(S, rc, "plaac_score_variants");
    std::string out;
    for (int64_t v = 0; v < nvar; v++) {
        const int64_t f = B.first_sub[(size_t)v];
        const SubList subs{B.pos.data() + f, B.code.data() + f, B.first_sub[(size_t)v + 1] - f};
        append_summary_row(o, B.rows[(size_t)v], sum[(size_t)v], B.ref.codes.data() + B.ref.offsets[(size_t)B.protein[(size_t)v]], out, subs);
        if (out.size() >= ((size_t)1 << 20)) {
            std::fwrite(out.data(), 1, out.size(), stdout);
            out.clear();
        }
    }
    std::fwrite(out.data(), 1, out.size(), stdout);
    B.clear();
    return 0;
}

// --variants / --saturate: the -i records through this program's reader, their variants scored batch by batch.
int score_variants_file(const Options& o, Scorers& S, VariantFile* VF)
{
    VariantBatch B;
    FastaReader fr(o.inputfile);
    std::string seq, name;
    std::vector<uint8_t> aa;
    while (fr.hasmore()) {
        name = fr.name();
        fr.next(seq);
        if (seq.empty()) continue;
        strip_stop(seq);
        if (seq.empty()) continue;
        aa.resize(seq.size());
        plaac_encode_host(seq.data(), (int64_t)seq.size(), aa.data());
        const int64_t len = (int64_t)seq.size();
        std::vector<int> mine;
        if (VF) {
            for (const std::string& id : {name, ">" + name}) {
                auto it = VF->by_id.find(id);
                if (it == VF->by_id.end()) continue;
                mine.insert(mine.end(), it->second.begin(), it->second.end());
                VF->matched[id] = true;
            }
            if (mine.empty()) continue;
            std::sort(mine.begin(), mine.end());
            for (int k : mine) {  // every line of this record is checked before any of its variants is scored
                const VariantLine& L = VF->lines[(size_t)k];
                for (size_t j = 0; j < L.pos.size(); j++) {
                    if (L.pos[j] >= len) {
                        std::fprintf(stderr, "plaac: %s line %d: position %d is beyond the end of %s (%lld residues)\n",
                                     o.variants_file.c_str(), L.line, L.pos[j] + 1, name.c_str(), (long long)len);
                        return 2;
                    }
                    if (aa[(size_t)L.pos[j]] != L.ref[j]) {
                        std::fprintf(stderr, "plaac: %s line %d: %s has %c at position %d, not %c\n", o.variants_file.c_str(),
                                     L.line, name.c_str(), kAaNames[aa[(size_t)L.pos[j]]], L.pos[j] + 1, kAaNames[L.ref[j]]);
                        return 2;
                    }
                }
            }
        }
        int32_t p = -1;  // this record's index in B.ref, once one of its variants is in the batch
        auto add = [&](const std::string& spec, const int32_t* ps, const uint8_t* cs, size_t n) -> int {
            if (p < 0) {
                B.ref.add(name, "", seq);
                p = (int32_t)B.ref.nprot() - 1;
            }
            B.protein.push_back(p);
            B.pos.insert(B.pos.end(), ps, ps + n);
            B.code.insert(B.code.end(), cs, cs + n);
            B.first_sub.push_back((int64_t)B.pos.size());
            B.rows.push_back(name + ":" + spec);
            B.nres += len;
            if (B.nres >= o.batch_res || (int64_t)B.protein.size() >= (4 << 20)) {
                p = -1;
                return score_variant_batch(o, S, B);
            }
            return 0;
        };
        int rc = 0;
        if (VF) {
            for (int k : mine) {
                const VariantLine& L = VF->lines[(size_t)k];
                if ((rc = add(L.spec, L.pos.data(), L.alt.data(), L.pos.size()))) return rc;
            }
        } else {
            if ((rc = add("WT", nullptr, nullptr, 0))) return rc;
            for (int32_t i = 0; i < (int32_t)len; i++)
                for (uint8_t c = 1; c <= 20; c++) {
                    if (c == aa[(size_t)i]) continue;
                    const std::string spec = kAaNames[aa[(size_t)i]] + std::to_string(i + 1) + kAaNames[c];
                    if ((rc = add(spec, &i, &c, 1))) return rc;
                }
        }
    }
    if (VF)
        for (const auto& m : VF->matched)
            if (!m.second) {
                std::fprintf(stderr, "plaac: %s line %d: %s is the name of no record of %s\n", o.variants_file.c_str(),
                             VF->lines[(size_t)VF->by_id.at(m.first).front()].line, m.first.c_str(), o.inputfile.c_str());
                return 2;
            }
    return score_variant_batch(o, S, B);
}

void usage()
{
    std::puts("------------------------------------------------------------");
    std::puts("plaac (B200/CUDA host): same command line and output tables as plaac.jar.");
    std::puts("------------------------------------------------------------");
    std::puts("USAGE: plaac -i input.fa > output.txt");
    std::puts("  -c core_length   minimal contiguous prion-like domain length for the HMM parses (default 60)");
    std::puts("  -B bg_freqs.txt  background AA frequencies/counts, one per line, in the order");
    std::puts("                   X, A, C, D, E, F, G, H, I, K, L, M, N, P, Q, R, S, T, V, W, Y, *");
    std::puts("  -b background.fa FASTA used to compute background AA frequencies (default: the input file);");
    std::puts("                   with -b or -B but no -i the counts are printed in -B format");
    std::puts("  -a alpha         weight of the S. cerevisiae background in the mix (0..1, default 1.0)");
    std::puts("  -F fg_freqs.txt  prion-like AA frequencies in the -B format (default: 28 S. cerevisiae domains)");
    std::puts("  -w window_size   FoldIndex window (default 41)");
    std::puts("  -W Window_size   PAPA window (default 41)");
    std::puts("  -d               print documentation of the output columns");
    std::puts("  -s               skip the run-time parameter block");
    std::puts("  -p list.txt|all  per-residue table for the listed proteins (one name per line) or for all");
    std::puts("  --gpus N, --device D, --batch-mb M, --rank, --rank-core, --gpu-ingest, --host-reader   (this host only)");
    std::puts("  --variants FILE  score the variants listed in FILE (SEQid<TAB>WT or D262V,P275S) instead of the records");
    std::puts("  --saturate       score every single substitution of every record");
    std::puts("  --effects COLS   with --variants or --saturate: print only each variant's change against the wild type in");
    std::puts("                   the listed columns (comma-separated: LLR COREscore PRDscore HMMall HMMvit FImeanhydro");
    std::puts("                   FImeancharge FImeancombo PAPAcombo PAPAprop PAPAfi PAPAllr PAPAllr2, printed as d<NAME>;");
    std::puts("                   COREchange: 1 CORE gained, -1 lost, 0 unchanged)");
    std::puts("  --segments FILE  also write every prion-like segment (maximal run of PrD-state residues of the Viterbi");
    std::puts("                   parse) of every record to FILE: SEQid SEGstart SEGend SEGlen SEGscore PRD");
    std::puts("  --null FILE --replicates K [--seed S] [--null-columns COLS]");
    std::puts("                   also score K composition-preserving shuffles of every record and write to FILE, per record,");
    std::puts("                   SEQid NULLreps and n<NAME> p<NAME> per column: the shuffles that reach the record's score");
    std::puts("                   (NaN lowest) and the empirical p-value (1+n)/(1+K).  COLS as --effects, with hasCORE (the");
    std::puts("                   shuffles with a CORE, no p) in place of COREchange; default COREscore,LLR,HMMall");
    std::puts("  --stop-hits H    with --null: stop a record's column once H shuffles have reached it (at most K shuffles;");
    std::puts("                   sequential p-values of Besag and Clifford).  FILE then holds SEQid and r<NAME> n<NAME>");
    std::puts("                   p<NAME> per column: r shuffles scored, n = H if it stopped, p = H/r if it stopped, else");
    std::puts("                   (1+n)/(1+K)");
    std::puts("  --compat-F       -F reads the -B file, as plaac.jar does (plaac.java:388); without it -F reads its own file,");
    std::puts("                   so the parameter block and every score differ from the jar's for the same command line");
}

}  // namespace

int main(int argc, char** argv)
{
    Options o;
    std::vector<std::string> args;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto val = [&](const char* name) -> const char* {
            if (i + 1 >= argc) {
                std::fprintf(stderr, "plaac: %s needs a value\n", name);
                std::exit(2);
            }
            return argv[++i];
        };
        if (a == "--gpus")
            o.gpus = std::atoi(val("--gpus"));
        else if (a == "--device")
            o.device = std::atoi(val("--device"));
        else if (a == "--batch-mb")
            o.batch_res = (int64_t)std::atoll(val("--batch-mb")) << 20, o.batch_set = true;
        else if (a == "--compat-F")
            o.compat_F = true;
        else if (a == "--rank")
            o.rank = true;
        else if (a == "--rank-core")
            o.rank = o.rank_core_only = true;
        else if (a == "--gpu-ingest")
            o.gpu_ingest = true;
        else if (a == "--host-reader")
            o.host_reader = true;
        else if (a == "--variants")
            o.variants_file = val("--variants");
        else if (a == "--saturate")
            o.saturate = true;
        else if (a == "--effects")
            o.effects = val("--effects"), o.effects_set = true;
        else if (a == "--segments")
            o.segments_file = val("--segments");
        else if (a == "--null")
            o.null_file = val("--null");
        else if (a == "--replicates")
            o.replicates = std::atoll(val("--replicates")), o.replicates_set = true;
        else if (a == "--seed")
            o.seed = std::strtoull(val("--seed"), nullptr, 10), o.seed_set = true;
        else if (a == "--null-columns")
            o.null_columns = val("--null-columns"), o.null_columns_set = true;
        else if (a == "--stop-hits")
            o.stop_hits_arg = val("--stop-hits");
        else if (a == "--format-check") {
            // test hook: lines "decimals value" on stdin -> the Java-formatted value on stdout
            int d;
            char tok[128];
            while (std::scanf("%d %127s", &d, tok) == 2) {
                if (d < 0)
                    std::puts(jdouble(std::strtod(tok, nullptr)).c_str());
                else
                    std::puts(jfmt(std::strtod(tok, nullptr), d).c_str());
            }
            return 0;
        }
        else
            args.push_back(a);
    }
    // plaac.java:337-353: options are consumed pairwise; the last token is examined only if it is -d or -s
    size_t i = 0;
    const size_t n = args.size();
    while (i + 1 < n || (i < n && (args[i] == "-d" || args[i] == "-s"))) {
        const std::string& a = args[i];
        if (a == "-i") o.inputfile = args[++i];
        else if (a == "-b") o.bgfile = args[++i];
        else if (a == "-B") o.bgfreqfile = args[++i];
        else if (a == "-F") o.fgfreqfile = args[++i];
        else if (a == "-c") o.corelength = std::atoi(args[++i].c_str());
        else if (a == "-w") o.ww1 = std::atoi(args[++i].c_str());
        else if (a == "-W") o.ww2 = std::atoi(args[++i].c_str());
        else if (a == "-a") o.alpha = std::atof(args[++i].c_str());
        else if (a == "-m") o.hmmtype = std::atoi(args[++i].c_str());
        else if (a == "-p") o.plotlist = args[++i];
        else if (a == "-h") o.hmmdotfile = args[++i];
        else if (a == "-d") o.printheaders = true;
        else if (a == "-s") o.printparameters = false;
        else std::printf("# skipping unknown option %s\n", a.c_str());
        i++;
    }
    o.ww3 = o.ww2;  // :355

    if (!o.segments_file.empty()) {
        const char* clash = !o.plotlist.empty()        ? "-p"
                            : !o.variants_file.empty() ? "--variants"
                            : o.saturate               ? "--saturate"
                            : o.gpu_ingest             ? "--gpu-ingest"
                            : o.gpus > 1               ? "--gpus > 1"
                                                       : nullptr;
        if (clash) {
            std::fprintf(stderr, "plaac: --segments cannot be combined with %s\n", clash);
            return 2;
        }
        o.host_reader = true;  // segments come with the records of plaac_score_segments, not the GPU reader's
    }
    if (!o.null_file.empty()) {
        const char* clash = !o.plotlist.empty()        ? "-p"
                            : !o.variants_file.empty() ? "--variants"
                            : o.saturate               ? "--saturate"
                            : !o.segments_file.empty() ? "--segments"
                            : o.gpu_ingest             ? "--gpu-ingest"
                            : o.gpus > 1               ? "--gpus > 1"
                                                       : nullptr;
        if (clash) {
            std::fprintf(stderr, "plaac: --null cannot be combined with %s\n", clash);
            return 2;
        }
        if (o.replicates < 1) {
            std::fprintf(stderr, "plaac: --null needs --replicates K with K >= 1\n");
            return 2;
        }
        if (!(o.null_mask = parse_columns(o.null_columns, "--null-columns", kNullNames))) return 2;
        if (o.stop_hits_arg) {
            const char* e = o.stop_hits_arg + std::strlen(o.stop_hits_arg);
            const auto [end, ec] = std::from_chars(o.stop_hits_arg, e, o.stop_hits);
            if (ec != std::errc() || end != e || end == o.stop_hits_arg) {
                std::fprintf(stderr, "plaac: --stop-hits needs an integer H, got '%s'\n", o.stop_hits_arg);
                return 2;
            }
            if (o.stop_hits < 1) {
                std::fprintf(stderr, "plaac: --stop-hits needs H >= 1, got %lld\n", (long long)o.stop_hits);
                return 2;
            }
        }
        o.host_reader = true;  // the shuffles come with the records of plaac_score_shuffles, not the GPU reader's
    } else if (o.replicates_set || o.seed_set || o.null_columns_set || o.stop_hits_arg) {
        std::fprintf(stderr, "plaac: %s needs --null FILE\n",
                     o.replicates_set ? "--replicates" : o.seed_set ? "--seed" : o.null_columns_set ? "--null-columns" : "--stop-hits");
        return 2;
    }
    const bool variants = o.saturate || !o.variants_file.empty();
    VariantFile vfile;
    if (variants) {
        const char* clash = o.saturate && !o.variants_file.empty() ? "--variants"
                            : !o.plotlist.empty()                  ? "-p"
                            : o.rank                               ? "--rank / --rank-core"
                            : o.gpu_ingest                         ? "--gpu-ingest"
                            : o.gpus > 1                           ? "--gpus > 1"
                                                                   : nullptr;
        if (clash) {
            std::fprintf(stderr, "plaac: %s cannot be combined with %s\n", o.saturate ? "--saturate" : "--variants", clash);
            return 2;
        }
        if (o.effects_set && !(o.effects_mask = parse_columns(o.effects, "--effects", kEffectNames))) return 2;
        if (!o.variants_file.empty() && !read_variant_file(o.variants_file, vfile)) return 2;
        o.host_reader = true;  // the work is the quadratic scoring, not the reading
    } else if (o.effects_set) {
        std::fprintf(stderr, "plaac: --effects needs --variants FILE or --saturate\n");
        return 2;
    }

    // The file-to-table fast path (GPU ingest) is the default for regular input files of at least 1 MB in summary mode;
    // --host-reader forces the reader of this program, --gpu-ingest the GPU one.
    bool fast = false;
    if (o.plotlist.empty() && !o.inputfile.empty() && !o.host_reader) {
        struct stat st;
        fast = o.gpu_ingest || (::stat(o.inputfile.c_str(), &st) == 0 && S_ISREG(st.st_mode) && st.st_size >= (1 << 20));
    }
    o.gpu_ingest = fast;
    const bool input_bg = o.bgfreqfile.empty() && o.bgfile.empty() && !o.inputfile.empty();  // :382-384

    // background counts :374-384
    double bgf[PLAAC_NAA] = {0};
    if (!o.bgfreqfile.empty())
        read_aa_params(o.bgfreqfile, bgf);
    else if (!o.bgfile.empty())
        bg_counts_from_fasta(o.bgfile, bgf);
    else if (!o.inputfile.empty() && !fast)
        bg_counts_from_fasta(o.inputfile, bgf);  // (fast path: counted on the GPU, below)
    double fgfile[PLAAC_NAA];
    const double* fg = nullptr;
    if (!o.fgfreqfile.empty()) {
        // plaac.java:388 reads bgfreqfile here (a bug); --compat-F reproduces it
        read_aa_params(o.compat_F ? o.bgfreqfile : o.fgfreqfile, fgfile);
        fg = fgfile;
        if (!o.compat_F)
            std::puts("# note: -F read from the -F file; plaac.jar reads the -B file here (plaac.java:388), --compat-F does the same");
    }
    if ((!o.bgfile.empty() || !o.bgfreqfile.empty()) && o.inputfile.empty()) {  // :393-403
        print_aa_params(bgf);
        return 0;
    }
    if (o.inputfile.empty()) {
        usage();
        return 0;
    }
    if (o.alpha > 1 || o.alpha < 0) {
        std::puts("# warning: invalid alpha; using alpha = 1.0");
        o.alpha = 1.0;
    }

    plaac_params P;
    double info[4][PLAAC_NAA];
    int rc = 0;
    auto make_params = [&]() -> int {
        rc = plaac_params_init(&P, o.alpha, bgf, fg, o.corelength, o.ww1, o.ww2, o.ww3, o.adjustprolines ? 1 : 0, &info[0][0]);
        if (rc != PLAAC_OK) std::fprintf(stderr, "plaac: plaac_params_init failed (%d)\n", rc);
        return rc;
    };
    auto print_preamble = [&]() {
        if (o.printparameters) {  // :503-514
            std::puts("############################ parameters at run-time ####################################");
            std::printf("## alpha=%s; corelength=%d; ww1=%d; ww2=%d; ww3=%d; adjustprolines=%s;\n", jdouble(o.alpha).c_str(),
                        o.corelength, o.ww1, o.ww2, o.ww3, o.adjustprolines ? "true" : "false");
            std::printf("## fg_used: {%s}\n", aaparams2string(info[0]).c_str());
            std::printf("## bg_scer: {%s}\n", aaparams2string(info[1]).c_str());
            std::printf("## bg_input: {%s}\n", aaparams2string(info[2]).c_str());
            std::printf("## bg_used: {%s}\n", aaparams2string(info[3]).c_str());
            std::printf("## plaac_llr: {%s}\n", aaparams2string(P.llr).c_str());
            std::printf("## papa_lods: {%s}\n", aaparams2string(P.papa_lod).c_str());
            std::puts("#######################################################################################");
        }
        if (!o.hmmdotfile.empty()) std::puts("# -h (GraphViz export of the HMM) is not part of this host; ignored");
    };
    auto print_table_head = [&]() {
        if (o.printheaders) {  // :661-711
            std::puts("############################ Description of output columns ############################");
            for (const char* d : kColumnDocs) std::printf("## %s\n", d);
            std::puts("#######################################################################################");
        }
        std::puts(kSummaryHeader);
        std::fflush(stdout);
    };

    Scorers S;
    auto open_devices = [&]() -> int {
        const int ndev = plaac_device_count();
        if (ndev <= 0) {
            std::fprintf(stderr, "plaac: no CUDA device (%s); this program has no CPU scoring path\n", plaac_last_error(nullptr));
            return 2;
        }
        if (o.gpus < 1) o.gpus = 1;
        if (o.gpus > ndev) o.gpus = ndev;
        for (int g = 0; g < o.gpus; g++) {
            plaac_ctx* c = nullptr;
            rc = plaac_create(&c, o.gpus == 1 ? o.device : g, &P);
            if (rc != PLAAC_OK) {
                std::fprintf(stderr, "plaac: plaac_create failed (%d): %s\n", rc, plaac_last_error(nullptr));
                return 2;
            }
            S.ctx.push_back(c);
        }
        Phase::mark("devices open");
        return 0;
    };
    auto close_devices = [&]() {
        for (auto c : S.ctx) plaac_destroy(c);
        S.ctx.clear();
    };

    if (fast) {
        Phase::mark("start");
        MappedFile F(o.inputfile);
        Phase::mark("file mapped");
        if (!F.good) {
            // the jar prints the message once per attempt to open the file (background pass, scoring pass)
            if (input_bg) std::printf("# Couldn't open %s\n", o.inputfile.c_str());
            if (make_params()) return 2;
            print_preamble();
            print_table_head();
            std::printf("# Couldn't open %s\n", o.inputfile.c_str());
            return 0;
        }
        auto to_stdout = [](const std::string& rows) { std::fwrite(rows.data(), 1, rows.size(), stdout); };
        if (input_bg && o.alpha < 1) {
            // the tables depend on the input's own composition: count first (GPU, provisional tables), then score
            if (make_params()) return 2;
            if ((rc = open_devices())) return rc;
            if ((rc = score_fasta_gpu(o, S, F, true, bgf, to_stdout))) return rc;
            close_devices();
        }
        if (input_bg && !(o.alpha < 1)) {
            // alpha = 1: the input's composition only feeds the "## bg_input" line of the preamble, which is printed before
            // the table.  One pass: score with the (composition-independent) tables, hold the rows, print the preamble
            // with the counts that pass produced, then the rows.
            if (make_params()) return 2;
            if ((rc = open_devices())) return rc;
            std::vector<std::string> held;
            rc = score_fasta_gpu(o, S, F, false, bgf, [&](std::string& rows) { held.push_back(std::move(rows)); });
            if (rc) return rc;
            if (make_params()) return 2;  // same tables, bg_input filled in
            print_preamble();
            print_table_head();
            for (const auto& h : held) std::fwrite(h.data(), 1, h.size(), stdout);
            std::fflush(stdout);
            Phase::mark("rows written");
            return 0;
        }
        if (make_params()) return 2;
        print_preamble();
        print_table_head();
        if ((rc = open_devices())) return rc;
        rc = score_fasta_gpu(o, S, F, false, nullptr, to_stdout);
        std::fflush(stdout);
        Phase::mark("rows written");
        return rc;
    }

    if (make_params()) return 2;
    print_preamble();
    if (variants) {
        if (o.effects_mask) {
            std::string head = "SEQid";
            for (int k = 0; k <= kEffectCoreChange; k++)
                if ((o.effects_mask >> k) & 1) head += std::string("\t") + (k == kEffectCoreChange ? "" : "d") + kEffectNames[k];
            std::puts(head.c_str());
            std::fflush(stdout);
        } else {
            print_table_head();
        }
        if ((rc = open_devices())) return rc;
        rc = score_variants_file(o, S, o.saturate ? nullptr : &vfile);
        std::fflush(stdout);
        return rc;
    }
    Batch B;
    std::string seq, name;
    std::unique_ptr<FILE, int (*)(FILE*)> seg_file(nullptr, std::fclose);
    if (!o.segments_file.empty()) {
        seg_file.reset(std::fopen(o.segments_file.c_str(), "w"));
        if (!seg_file) {
            std::fprintf(stderr, "plaac: cannot open %s for writing\n", o.segments_file.c_str());
            return 2;
        }
        o.seg_out = seg_file.get();
        std::fputs("SEQid\tSEGstart\tSEGend\tSEGlen\tSEGscore\tPRD\n", o.seg_out);
    }
    std::unique_ptr<FILE, int (*)(FILE*)> null_file(nullptr, std::fclose);
    if (!o.null_file.empty()) {
        null_file.reset(std::fopen(o.null_file.c_str(), "w"));
        if (!null_file) {
            std::fprintf(stderr, "plaac: cannot open %s for writing\n", o.null_file.c_str());
            return 2;
        }
        o.null_out = null_file.get();
        std::string head = o.stop_hits > 0 ? "SEQid" : "SEQid\tNULLreps";
        for (int b = 0; b <= kEffectCoreChange; b++)
            if ((o.null_mask >> b) & 1)
                head += (o.stop_hits > 0 ? std::string("\tr") + kNullNames[b] : std::string()) + "\tn" + kNullNames[b] +
                        (b == kEffectCoreChange ? "" : std::string("\tp") + kNullNames[b]);
        head += "\n";
        std::fputs(head.c_str(), o.null_out);
    }
    if (o.plotlist.empty()) {
        print_table_head();
        if ((rc = open_devices())) return rc;
        FastaReader fr(o.inputfile);
        while (fr.hasmore()) {
            name = fr.name();
            fr.next(seq);
            if (seq.empty()) continue;  // the jar throws on sb.charAt(-1) (:758); skip the record instead
            strip_stop(seq);
            if (seq.empty()) continue;  // :762
            B.add(name, "", seq);
            if ((int64_t)B.codes.size() >= o.batch_res || B.nprot() >= (4 << 20))
                if ((rc = score_summary_batch(o, S, B))) return rc;
        }
        if ((rc = score_summary_batch(o, S, B))) return rc;
    } else {
        std::map<std::string, std::string> syn, order;
        const bool plotall = o.plotlist == "all";
        if (!plotall) read_plot_list(o.plotlist, syn, order);
        std::puts("ORDER\tSEQid\tAANUM\tAA\tVIT\tMAP\tCHARGE\tHYDRO\tFI\tPLAAC\tPAPA\tFIx2\tPLAACx2\tPAPAx2\tHMM.background\tHMM.PrD-like");
        std::fflush(stdout);
        if ((rc = open_devices())) return rc;
        FastaReader fr(o.inputfile);
        int genecount = 1;
        const int64_t res_batch = std::min<int64_t>(o.batch_res, (int64_t)32 << 20);
        while (fr.hasmore()) {
            name = fr.name();
            fr.next(seq);
            if (!(plotall || syn.count(name) || syn.count(">" + name))) continue;  // :617
            std::string nm = name, id = std::to_string(genecount);
            if (syn.count(name)) nm = syn[name];
            if (order.count(name)) id = order[name];
            if (seq.empty()) continue;  // the jar throws (:624)
            strip_stop(seq);
            genecount++;
            B.add(nm, id, seq);
            if ((int64_t)B.codes.size() >= res_batch)
                if ((rc = score_residue_batch(o, S, B))) return rc;
        }
        if ((rc = score_residue_batch(o, S, B))) return rc;
    }
    return 0;
}
