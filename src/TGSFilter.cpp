// tgsfilter — drop-in CLI host over libtgsf_cuda (B200).
//
// Written from scratch against include/tgsf.h; mirrors the reference CLI's observable behaviour for
// the filter / QC path: argv grammar, defaults and clamps of TGSFilter_cmd (T.cpp:198-503), the
// pre-pass (GetFilterParameterTask, T.cpp:869-1216; parameter resolution in main, T.cpp:3058-3126),
// FASTQ/FASTA records on stdout or -o (T.cpp:2020-2053) and the INFO: lines on stderr
// (T.cpp:3071-3098, 3214-3235).  ("T.cpp" = reference src/TGSFilter.cpp.)
//
// The thread/queue runtime of the reference (1 reader + N workers + 1 writer, T.cpp:1808-1916) is
// replaced by: parse -> pinned varlen batches -> tgsf_submit (async, two batches in flight per GPU,
// batches dealt round-robin over the GPUs) -> tgsf_collect -> records in input order (= -t 1).
//
// Downsampling (-g/-d/-r/-R, -F) follows DownSampleTask's selection (T.cpp:2297-2344) over the
// filtered records.  BAM/SAM input is parsed by the ingest pipeline itself (src/pipeline.hpp; BGZF blocks decoded
// in parallel), without htslib.
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <iostream>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/uio.h>
#include <unistd.h>

#include "../include/tgsf.h"
#include "../include/tgsf_layout.h"
#include "pipeline.hpp"
#include "report.hpp"

using std::cerr;
using std::endl;
using std::string;

namespace {

// ---- parameters: Para_A24 (T.cpp:82-172) -------------------------------------------------------
struct Params {
    string InFile, OutFile, readType, AdapterFile;
    int MinLen = 1000, MaxLen = 2147483647;
    float MinQ = -1, MaxQ = 255;
    int BCNum = 100000, BCLen = 150;
    float EndBias = 1;
    int HeadTrim = -1, TailTrim = -1;
    bool ONLYAD = false;
    int ADNum = 100000, EndLen = 150, EndMatchLen = 4, MidMatchLen = 35, ExtraLen = 50;
    float EndSim = 0, MidSim = 0;
    bool discard = false;
    uint64_t GenomeSize = 0;
    int DesiredDepth = 0, DesiredNum = 0;
    float DesiredFrac = 0;
    bool Downsample = false, Filter = true;
    int Kmer = 11, MinRepeat = 0;
    bool OnlyQC = false, FastaOut = false;
    int n_thread = 16, Infq = 3, Outfq = 3;
    bool OUTGZ = false;
    int compLevel = 6;
    int gpus = 1;                 // --gpus (extension; TGSF_GPUS env)
    string ContamFile;            // --contam (extension): drop pieces that share k-mers with this FASTA
    int ContamK = 17;             // --contam-k
    float ContamFrac = 0.05f;     // --contam-frac
    uint64_t batch_bases = 64ull << 20; // bases per batch (TGSF_BATCH_MB)
};

int usage() {
    std::cout << "Usage: tgsfilter -i TGS.raw.fq.gz -x ont -o TGS.clean.fq.gz\n"
                 " Input/Output options:\n"
                 "   -i   <str>   input of fasta/fastq file\n"
                 "   -x   <str>   read type (ont|clr|hifi)\n"
                 "   -o   <str>   output of fasta/fastq file instead of stdout\n"
                 " Basic filter options:\n"
                 "   -l   <int>   min length of read to out [1000]\n"
                 "   -L   <int>   max length of read to out\n"
                 "   -q  <float>  min Phred average quality score\n"
                 "   -Q  <float>  max Phred average quality score\n"
                 "   -n   <int>   read number for base content check [100000]\n"
                 "   -e   <int>   read end length for base content check [150]\n"
                 "   -b  <float>  bias (%) of adjacent base content at read end [1]\n"
                 "   -5   <int>   trim bases from the 5' end of the read\n"
                 "   -3   <int>   trim bases from the 3' end of the read\n"
                 " Adapter filter options:\n"
                 "   -a   <str>   adapter sequence file \n"
                 "   -A           disable reads filter, only for adapter identify\n"
                 "   -N   <int>   read number for adapter identify [100000]\n"
                 "   -E   <int>   read end length for adapter trim [150]\n"
                 "   -m   <int>   min match length for end adapter [15]\n"
                 "   -M   <int>   min match length for middle adapter [35]\n"
                 "   -T   <int>   extra trim length for middle adpter on both side [50]\n"
                 "   -s  <float>  min similarity for end adapter\n"
                 "   -S  <float>  min similarity for middle adapter\n"
                 "   -D           discard reads with middle adapter instead of split\n"
                 " Downsampling options:\n"
                 "   -g   <str>   genome size (k/m/g)\n"
                 "   -d   <int>   downsample to the desired coverage (requires -g) \n"
                 "   -r   <int>   downsample to the desired number of reads \n"
                 "   -R  <float>  downsample to the desired fraction of reads \n"
                 "   -F           disable reads filter, only for downsampling\n"
                 "   -k   <int>   kmer size for repeat evaluations [11] \n"
                 "   -p   <int>   min repeat length of reads [0] \n"
                 " Other options:\n"
                 "   --qc         disable all filter, only for quality control \n"
                 "   -f           force FASTA output (discard quality) \n"
                 "   -c   <int>   compression level (0-9) for compressed output [6]\n"
                 "   -t   <int>   host threads for compressing/writing the output [16] (filtering runs on the GPU)\n"
                 "   --gpus <int> number of GPUs to shard batches over [1]\n"
                 " Contaminant screen options:\n"
                 "   --contam <str>        FASTA[.gz] of contaminant sequences; pieces sharing enough k-mers are discarded\n"
                 "   --contam-k <int>      k-mer size of the contaminant screen, 11-31 [17]\n"
                 "   --contam-frac <float> min fraction of a piece's k-mers found in the set to discard it [0.05]\n"
                 "   -h           show help [b200 host of v1.11]\n\n";
    return 1;
}

uint64_t genome_size(const string &g) { // GetGenomeSize, T.cpp:178-196
    if (g.empty()) return 0;
    char u = (char)std::tolower((unsigned char)g.back());
    double v = atof(g.c_str());
    if (u == 'k') v *= 1e3;
    else if (u == 'm') v *= 1e6;
    else if (u == 'g') v *= 1e9;
    return (uint64_t)v;
}

// TGSFilter_cmd, T.cpp:198-503: every '-' is removed from the flag token, so --qc == -qc.
int parse_cmd(int argc, char **argv, Params *P) {
    if (argc <= 2) { usage(); return 1; }
    for (int i = 1; i < argc; i++) {
        if (argv[i][0] != '-') { cerr << "Error: command option error! please check." << endl; return 1; }
        string flag = argv[i];
        flag.erase(std::remove(flag.begin(), flag.end(), '-'), flag.end());
        auto need = [&]() -> bool {
            if (i + 1 == argc) { cerr << "Error: Lack Argument for [ -" << flag << " ]" << endl; return false; }
            i++;
            return true;
        };
        if (flag == "i") { if (!need()) return 1; P->InFile = argv[i]; }
        else if (flag == "o") { if (!need()) return 1; P->OutFile = argv[i]; }
        else if (flag == "x") { if (!need()) return 1; P->readType = argv[i]; }
        else if (flag == "l") { if (!need()) return 1; P->MinLen = atoi(argv[i]); if (P->MinLen < 100) P->MinLen = 100; }
        else if (flag == "L") { if (!need()) return 1; P->MaxLen = atoi(argv[i]); }
        else if (flag == "q") { if (!need()) return 1; P->MinQ = atof(argv[i]); }
        else if (flag == "Q") { if (!need()) return 1; P->MaxQ = atof(argv[i]); }
        else if (flag == "n") { if (!need()) return 1; P->BCNum = atoi(argv[i]); }
        else if (flag == "e") { if (!need()) return 1; P->BCLen = atoi(argv[i]); }
        else if (flag == "b") { if (!need()) return 1; P->EndBias = atof(argv[i]); }
        else if (flag == "5") { if (!need()) return 1; P->HeadTrim = atoi(argv[i]); }
        else if (flag == "3") { if (!need()) return 1; P->TailTrim = atoi(argv[i]); }
        else if (flag == "a") { if (!need()) return 1; P->AdapterFile = argv[i]; }
        else if (flag == "A") { P->ONLYAD = true; }
        else if (flag == "N") { if (!need()) return 1; P->ADNum = atoi(argv[i]); }
        else if (flag == "E") { if (!need()) return 1; P->EndLen = atoi(argv[i]); }
        else if (flag == "m") { if (!need()) return 1; P->EndMatchLen = atoi(argv[i]); }
        else if (flag == "M") { if (!need()) return 1; P->MidMatchLen = atoi(argv[i]); }
        else if (flag == "T") { if (!need()) return 1; P->ExtraLen = atoi(argv[i]); }
        else if (flag == "s") {
            if (!need()) return 1;
            P->EndSim = atof(argv[i]);
            if (P->EndSim < 0.7) { P->EndSim = 0.7; cerr << "Warning: re set -s to : " << P->EndSim << endl; }
        }
        else if (flag == "S") {
            if (!need()) return 1;
            P->MidSim = atof(argv[i]);
            if (P->MidSim < 0.8) { P->MidSim = 0.8; cerr << "Warning: reset -S to : " << P->MidSim << endl; }
        }
        else if (flag == "D") { P->discard = true; }
        else if (flag == "g") { if (!need()) return 1; P->GenomeSize = genome_size(argv[i]); if (P->GenomeSize == 0) return 1; }
        else if (flag == "d") { if (!need()) return 1; P->DesiredDepth = atoi(argv[i]); }
        else if (flag == "r") { if (!need()) return 1; P->DesiredNum = atoi(argv[i]); }
        else if (flag == "R") { if (!need()) return 1; P->DesiredFrac = atof(argv[i]); }
        else if (flag == "k") { if (!need()) return 1; P->Kmer = atoi(argv[i]); }
        else if (flag == "p") { if (!need()) return 1; P->MinRepeat = atoi(argv[i]); }
        else if (flag == "F") { P->Filter = false; }
        else if (flag == "qc") { P->OnlyQC = true; }
        else if (flag == "c") { if (!need()) return 1; P->compLevel = atoi(argv[i]); }
        else if (flag == "f") { P->FastaOut = true; }
        else if (flag == "t") { if (!need()) return 1; P->n_thread = atoi(argv[i]); }
        else if (flag == "gpus") { if (!need()) return 1; P->gpus = std::max(1, atoi(argv[i])); }
        else if (flag == "contam") { if (!need()) return 1; P->ContamFile = argv[i]; }
        else if (flag == "contamk") { if (!need()) return 1; P->ContamK = atoi(argv[i]); }
        else if (flag == "contamfrac") { if (!need()) return 1; P->ContamFrac = (float)atof(argv[i]); }
        else if (flag == "help" || flag == "h") { usage(); return 1; }
        else { cerr << "Error: UnKnow argument -" << flag << endl; return 1; }
    }
    if (P->InFile.empty()) { cerr << "Error: lack argument for the must: -i " << endl; exit(-1); }
    if (access(P->InFile.c_str(), 0) != 0) { cerr << "Error: Can't find this file for -i " << P->InFile << endl; exit(-1); }
    if (P->ContamK < 11 || P->ContamK > 31) { cerr << "Error: --contam-k must be in [11,31]" << endl; exit(-1); }
    const long long contam_ppm = llround((double)P->ContamFrac * 1e6); // as tgsf_set_contaminants computes it
    if (!(P->ContamFrac == P->ContamFrac) || contam_ppm < 1 || contam_ppm > 1000000) {
        cerr << "Error: --contam-frac must be in (0,1]" << endl;
        exit(-1);
    }
    if (!P->ContamFile.empty()) {
        if (P->OnlyQC || P->ONLYAD || !P->Filter) {
            cerr << "Error: --contam screens filtered reads and cannot be combined with --qc, -A or -F" << endl;
            exit(-1);
        }
        if (access(P->ContamFile.c_str(), R_OK) != 0) { cerr << "Error: Can't find this file for --contam " << P->ContamFile << endl; exit(-1); }
    }
    if (P->OnlyQC) P->Filter = false;
    if (P->Filter) {
        if (P->readType.empty()) { cerr << "Error: lack argument for the must: -x " << endl; exit(-1); }
        const string rt = P->readType;
        if (rt == "CLR" || rt == "clr") { cerr << "INFO: read type: PacBio continuous long read (clr)." << endl; P->readType = "clr"; }
        else if (rt == "HIFI" || rt == "hifi" || rt == "CCS" || rt == "ccs") { cerr << "INFO: read type: PacBio highly accurate long reads (hifi)." << endl; P->readType = "hifi"; }
        else if (rt == "ONT" || rt == "ont") { cerr << "INFO: read type: NanoPore reads (ont)." << endl; P->readType = "ont"; }
        else { cerr << "Error: read type should be : clr/hifi/ccs/ont or CLR/HIFI/CCS/ONT." << endl; exit(-1); }
        if (P->MidSim == 0) P->MidSim = P->readType == "hifi" ? 0.95 : 0.9;          // T.cpp:439-447
        if (P->EndSim == 0) P->EndSim = P->readType == "hifi" ? 0.9 : P->readType == "clr" ? 0.8 : 0.75;
        cerr << "INFO: min similarity for middle adapter: " << P->MidSim << endl;
        cerr << "INFO: min similarity for end adapter: " << P->EndSim << endl;
    }
    if (P->DesiredNum > 0 || P->DesiredFrac > 0) { // T.cpp:463-480
        P->Downsample = true;
    } else if (P->GenomeSize > 0 || P->DesiredDepth > 0) {
        if (P->GenomeSize > 0 && P->DesiredDepth > 0) P->Downsample = true;
        else if (P->GenomeSize > 0) { cerr << "Error: The desired depth was required, along with the genome size!" << endl; exit(-1); }
        else { cerr << "Error: The genome size was required, along with the desired depth!" << endl; exit(-1); }
    }
    if (!P->Filter && !P->Downsample && !P->OnlyQC) {
        cerr << "Error: Please set functional parameters for filter, downsampling or quality control." << endl;
        exit(-1);
    }
    return 0;
}

// Contaminant FASTA (multi-line, plain or gzip): records back to back in seq, offs[i]..offs[i+1].
bool load_contam_fasta(const string &path, std::vector<uint8_t> &seq, std::vector<uint64_t> &offs) {
    gzFile f = gzopen(path.c_str(), "rb");
    if (!f) return false;
    gzbuffer(f, 1 << 20);
    seq.clear();
    offs.assign(1, 0);
    std::vector<char> line(1 << 16);
    bool in_rec = false, at_bol = true, header = false;
    int n;
    while ((n = gzread(f, line.data(), (unsigned)line.size())) > 0) {
        for (int i = 0; i < n; ++i) {
            const char ch = line[(size_t)i];
            if (ch == '\n') { at_bol = true; header = false; continue; }
            if (at_bol && ch == '>') {
                if (in_rec) offs.push_back(seq.size());
                in_rec = true;
                header = true;
            } else if (!header && ch != '\r' && ch != ' ' && ch != '\t') {
                in_rec = true;
                seq.push_back((uint8_t)ch);
            }
            at_bol = false;
        }
    }
    const bool ok = n == 0;
    gzclose(f);
    if (in_rec) offs.push_back(seq.size());
    return ok;
}

string file_ext(const string &p) { size_t d = p.rfind('.'); return d == string::npos ? "" : p.substr(d + 1); }
int file_type(const string &path) { // GetFileType, T.cpp:839-857
    string ext = file_ext(path);
    if (ext == "gz") ext = file_ext(path.substr(0, path.rfind('.')));
    if (ext == "fa" || ext == "fasta") return 0;
    if (ext == "fq" || ext == "fastq") return 1;
    if (ext == "sam" || ext == "SAM" || ext == "bam" || ext == "BAM") return 2;
    return 3;
}

char g_comp[256];
string rev_comp(const string &s) { // rev_comp_seq, T.cpp:860-867
    string r;
    r.reserve(s.size());
    for (int i = (int)s.size() - 1; i >= 0; --i) r += g_comp[(unsigned char)s[i]];
    return r;
}

// ---- FASTA / FASTQ reader: 4-line FASTQ, 2-line FASTA, like FastxReader (T.cpp:521-782) ----------
class FastxReader {
public:
    explicit FastxReader(const string &path) : isFastq_(file_type(path) == 1) {
        if (file_type(path) == 2) { // BAM / SAM: the ingest parser's record reader (src/pipeline.hpp)
            sambam_.reset(new ingest::FastParser(path, true, true));
            if (!sambam_->ok()) sambam_.reset();
            return;
        }
        f_ = gzopen(path.c_str(), "rb"); // transparent for plain files, multi-member aware
        if (f_) gzbuffer(f_, 1 << 20);
        buf_.resize(1 << 20);
    }
    ~FastxReader() { if (f_) gzclose(f_); }
    bool ok() const { return f_ != nullptr || sambam_ != nullptr; }
    // false at end of input or on a malformed record (the reference stops there too)
    bool read(string &name, string &seq, string &qual) {
        if (sambam_) {
            ingest::FastParser::Rec r;
            if (!sambam_->next(r)) return false;
            name.assign(r.name, r.name_len);
            seq.assign(r.seq, r.seq_len);
            qual.assign(r.qual, r.qual_len);
            return true;
        }
        if (!f_) return false;
        if (isFastq_) {
            string strand;
            for (int i = 0; i < 5; i++) {
                if (!line(name)) return false;
                if (!name.empty() && name[0] == '@') {
                    if (!line(seq) || !line(strand)) return false;
                    if (!strand.empty() && strand[0] == '+' && !seq.empty()) break;
                }
            }
            if (name.empty()) { cerr << "Error: input format wrong!" << endl; return false; }
            name = name.substr(1);
            if (!line(qual) || qual.empty()) { cerr << "Error: quality are empty:" << name << endl; return false; }
            if (qual.size() != seq.size()) { cerr << "warning: sequence and quality have different length:" << name << endl; return false; }
            return true;
        }
        for (int i = 0; i < 3; i++) {
            if (!line(name)) return false;
            if (!name.empty() && name[0] == '>') break;
        }
        if (name.empty()) { cerr << "Error: input format wrong!" << endl; return false; }
        name = name.substr(1);
        if (!line(seq) || seq.empty()) { cerr << "Error: sequence are empty:" << name << endl; return false; }
        qual.clear();
        return true;
    }

private:
    bool fill() {
        int n = gzread(f_, buf_.data(), (unsigned)buf_.size());
        if (n <= 0) return false;
        pos_ = 0;
        len_ = (size_t)n;
        return true;
    }
    bool line(string &out) {
        out.clear();
        while (true) {
            if (pos_ == len_ && !fill()) return !out.empty();
            const char *p = buf_.data() + pos_;
            const char *nl = (const char *)memchr(p, '\n', len_ - pos_);
            if (nl) {
                out.append(p, nl - p);
                pos_ += (size_t)(nl - p) + 1;
                if (!out.empty() && out.back() == '\r') out.pop_back();
                return true;
            }
            out.append(p, len_ - pos_);
            pos_ = len_;
        }
    }
    gzFile f_ = nullptr;
    std::unique_ptr<ingest::FastParser> sambam_;
    bool isFastq_;
    std::vector<char> buf_;
    size_t pos_ = 0, len_ = 0;
};

// ---- varlen batch: byte bases stay on the host for record output; what crosses PCIe is the 2-bit
// packed stream (pinned) + Phred bytes (pinned) + offsets + the exception list ---------------------
struct Batch {
    std::vector<uint8_t> bases;     // concatenated, host only
    uint8_t *packed = nullptr, *quals = nullptr; // tgsf_host_alloc'ed
    size_t cap = 0, used = 0;
    std::vector<uint64_t> offsets{0};
    std::vector<string> names;
    std::vector<uint64_t> exc_pos;
    std::vector<uint8_t> exc_byte;
    bool reserve(size_t want) {
        if (want <= cap) return true;
        size_t ncap = std::max(want, cap * 2 + (1 << 20));
        uint8_t *np = nullptr, *nq = nullptr;
        if (tgsf_host_alloc((void **)&np, ncap / 4 + 64) != TGSF_OK || tgsf_host_alloc((void **)&nq, ncap) != TGSF_OK) return false;
        if (used) memcpy(nq, quals, used);
        tgsf_host_free(packed);
        tgsf_host_free(quals);
        packed = np; quals = nq; cap = ncap;
        return true;
    }
    bool add(const string &name, const string &seq, const string &qual, bool has_qual) {
        if (!reserve(used + seq.size() + 64)) return false;
        bases.insert(bases.end(), seq.begin(), seq.end());
        if (has_qual) memcpy(quals + used, qual.data(), seq.size());
        used += seq.size();
        offsets.push_back(used);
        names.push_back(name);
        return true;
    }
    // 2-bit pack the whole concatenated stream (tgsf_pack_bases), growing the exception list on demand
    bool pack() {
        uint64_t ne = 0;
        exc_pos.resize(std::max<size_t>(exc_pos.size(), 1024));
        exc_byte.resize(exc_pos.size());
        int rc = tgsf_pack_bases(bases.data(), used, packed, exc_pos.data(), exc_byte.data(), exc_pos.size(), &ne);
        if (rc == TGSF_ERR_CAPACITY) {
            exc_pos.resize(ne);
            exc_byte.resize(ne);
            rc = tgsf_pack_bases(bases.data(), used, packed, exc_pos.data(), exc_byte.data(), exc_pos.size(), &ne);
        }
        n_exc = ne;
        return rc == TGSF_OK;
    }
    uint64_t n_exc = 0;
    void clear() { used = 0; bases.clear(); offsets.assign(1, 0); names.clear(); }
    void release() { tgsf_host_free(packed); tgsf_host_free(quals); packed = quals = nullptr; cap = 0; }
    uint32_t n() const { return (uint32_t)names.size(); }
};

string new_seq_name(const string &raw, int number) { // newSeqName, T.cpp:1680-1701
    string add = ":" + std::to_string(number), out;
    bool found = false;
    for (char c : raw) {
        if (std::isspace((unsigned char)c) && !found) { out += add; out += c; found = true; }
        else out += c;
    }
    if (!found) out += add;
    return out;
}

const char *kLib[TGSF_LIB_ADAPTERS] = { // adapterLib, T.cpp:2969-2991
    "ATCTCTCTCTTTTCCTCCTCCTCCGTTGTTGTTGTTGAGAGAGAT", "ATCTCTCTCAACAACAACAACGGAGGAGGAGGAAAAGAGAGAGAT",
    "AAAAAAAAAAAAAAAAAATTAACGGAGGAGGAGGA", "TCCTCCTCCTCCGTTAATTTTTTTTTTTTTTTTTT",
    "AATGTACTTCGTTCAGTTACGTATTGCT", "AGCAATACGTAACTGAACGAAGTACATT",
    "GCAATACGTAACTGAACGAAGT", "ACTTCGTTCAGTTACGTATTGC",
    "GTTTTCGCATTTATCGTGAAACGCTTTCGCGTTTTTCGTGCGCCGCTTCA", "TGAAGCGGCGCACGAAAAACGCGAAAGCGTTTCACGATAAATGCGAAAAC",
    "GGCGTCTGCTTGGGTGTTTAACCTTTTTGTCAGAGAGGTTCCAAGTCAGAGAGGTTCCT", "AGGAACCTCTCTGACTTGGAACCTCTCTGACAAAAAGGTTAAACACCCAAGCAGACGCC",
    "GGAACCTCTCTGACTTGGAACCTCTCTGACAAAAAGGTTAAACACCCAAGCAGACGCCAGCAAT", "ATTGCTGGCGTCTGCTTGGGTGTTTAACCTTTTTGTCAGAGAGGTTCCAAGTCAGAGAGGTTCC",
    "TTTTTTTTCCTGTACTTCGTTCAGTTACGTATTGCT", "AGCAATACGTAACTGAACGAAGTACAGGAAAAAAAA",
    "GCAATACGTAACTGAACGAAGTACAGG", "CCTGTACTTCGTTCAGTTACGTATTGC",
    "ACGTAACTGAACGAAGTACAGG", "CCTGTACTTCGTTCAGTTACGT",
    "CTTGCGGGCGGCGGACTCTCCTCTGAAGATAGAGCGACAGGCAAG", "CTTGCCTGTCGCTCTATCTTCAGAGGAGAGTCCGCCGCCCGCAAG"};

// decision loop of CheckBaseContent, T.cpp:1097-1134
int base_content_trim(const std::vector<int32_t> &bn, int checkLen, int seqNum, float EndBias) {
    int maxDiff = (seqNum * EndBias) / 100;
    int trimLen = 0;
    for (int i = 1; i < checkLen - 1; i++) {
        bool leftFlag = false, rightFlag = false;
        int l = std::min(i, 5), r = std::min(checkLen - i - 1, 5);
        for (int j = 0; j < 4; j++) {
            for (int x = 1; x <= l; x++)
                if (abs(bn[i * 4 + j] - bn[(i - x) * 4 + j]) > maxDiff) { leftFlag = true; break; }
            for (int x = 1; x <= r; x++)
                if (abs(bn[(i + x) * 4 + j] - bn[i * 4 + j]) > maxDiff) { rightFlag = true; break; }
        }
        if (leftFlag && rightFlag) trimLen = i + 1;
    }
    return trimLen;
}

// Downsampling (DownSampleTask, T.cpp:2164-2568): the reads are ranked by length, longest first, and
// taken until the genome-size x depth / fraction / count target is met (get_reads_name,
// T.cpp:2297-2344); the second pass then keeps the records whose NAME was selected, in file order.
// Like the reference the ranking is keyed by read name (a later record with the same name replaces
// the length of an earlier one, T.cpp:2135/2267).  Equal lengths at the cut-off are ordered by the
// reference through std::sort over an unordered_map (unspecified); here ties keep file order.
struct RecIndex {
    std::vector<string> names;               // unique names in first-seen order
    std::vector<int> lens;                   // current length per unique name
    std::unordered_map<string, size_t> pos;  // name -> slot
    void add(const string &name, int len) {
        auto it = pos.find(name);
        if (it == pos.end()) { pos.emplace(name, names.size()); names.push_back(name); lens.push_back(len); }
        else lens[it->second] = len;
    }
};

struct Selection {
    std::vector<char> keep; // per unique-name slot
    uint64_t downBases = 0, downNum = 0;
};

// total_all: the reference's `totalSize` when it is known before the ranking (-F: get_fastx_SeqLen adds EVERY record,
// also the earlier ones of a repeated name, T.cpp:2256-2269); 0 = sum over the ranked names (filter mode, T.cpp:2318-2322).
// The ranking needs no sort: a histogram of the lengths gives the cut-off length and how many reads of exactly that
// length are taken (the first ones in file order), in O(reads + longest read).
Selection select_reads(const RecIndex &idx, const Params &P, uint64_t total_all = 0) {
    Selection S;
    const size_t n = idx.names.size();
    S.keep.assign(n, 0);
    int max_len = 0;
    uint64_t totalSize = 0;
    for (int l : idx.lens) { totalSize += (uint64_t)l; max_len = std::max(max_len, l); }
    if (total_all) totalSize = total_all;
    std::vector<uint32_t> hist((size_t)max_len + 2, 0);
    for (int l : idx.lens) hist[(size_t)std::max(l, 0)]++;
    // walk the lengths from the longest: reads are taken one by one until the target is met
    uint64_t desired = 0;
    bool by_bases = true;
    if (P.GenomeSize > 0 && P.DesiredDepth > 0) desired = P.GenomeSize * (uint64_t)P.DesiredDepth;
    else if (P.DesiredFrac > 0) desired = (uint64_t)(P.DesiredFrac * totalSize);
    else if (P.DesiredNum > 0) { desired = (uint64_t)P.DesiredNum; by_bases = false; }
    else return S;
    int cut_len = -1;          // reads longer than this are all taken
    uint64_t cut_take = 0;     // ... and this many of exactly this length
    uint64_t added = 0;
    for (int l = max_len; l >= 0 && cut_len < 0; --l) {
        const uint64_t c = hist[(size_t)l];
        if (!c) continue;
        // the loop of get_reads_name takes a read, then tests `added >= desired`
        const uint64_t unit = by_bases ? (uint64_t)l : 1;
        uint64_t need;
        if (added >= desired) need = 1;                              // (only possible before the first read: desired == 0)
        else if (unit == 0) need = c + 1;                            // zero-length reads never reach the target
        else need = (desired - added + unit - 1) / unit;             // reads of this length until added >= desired
        if (need <= c) { cut_len = l; cut_take = need; }
        else added += c * unit;
    }
    if (cut_len < 0) { cut_len = -1; cut_take = 0; }                 // target never met: everything is taken
    uint64_t at_cut = 0;
    for (size_t i = 0; i < n; i++) {
        const int l = idx.lens[i];
        bool k = l > cut_len;
        if (l == cut_len && at_cut < cut_take) { k = true; ++at_cut; }
        if (k) { S.keep[i] = 1; S.downBases += (uint64_t)l; S.downNum++; }
    }
    return S;
}

Selection select_reads_sorted(const RecIndex &idx, const Params &P, uint64_t total_all = 0) { // reference form (tests: TGSF_SELECT_SORT=1)
    Selection S;
    S.keep.assign(idx.names.size(), 0);
    std::vector<size_t> order(idx.names.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return idx.lens[a] > idx.lens[b]; });
    uint64_t totalSize = 0;
    for (int l : idx.lens) totalSize += (uint64_t)l;
    if (total_all) totalSize = total_all;
    auto take = [&](size_t i) { S.keep[i] = 1; S.downBases += (uint64_t)idx.lens[i]; S.downNum++; };
    if (P.GenomeSize > 0 && P.DesiredDepth > 0) {
        uint64_t added = 0, desired = P.GenomeSize * (uint64_t)P.DesiredDepth;
        for (size_t i : order) { take(i); added += (uint64_t)idx.lens[i]; if (added >= desired) break; }
    } else if (P.DesiredFrac > 0) {
        uint64_t added = 0, desired = (uint64_t)(P.DesiredFrac * totalSize);
        for (size_t i : order) { take(i); added += (uint64_t)idx.lens[i]; if (added >= desired) break; }
    } else if (P.DesiredNum > 0) {
        int n = 0;
        for (size_t i : order) { take(i); if (++n >= P.DesiredNum) break; }
    }
    return S;
}

struct Timer { // TGSF_TIMING=1: phase timings on stderr
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double lap() { auto t1 = std::chrono::steady_clock::now(); double d = std::chrono::duration<double>(t1 - t0).count(); t0 = t1; return d; }
};
bool g_timing = false;
void tlog(const char *what, double s) { if (g_timing) cerr << "[timing] " << what << ": " << s << " s" << endl; }

void die_tgsf(const char *what) {
    cerr << "Error: " << what << ": " << tgsf_last_error() << endl;
    exit(-1);
}

}  // namespace

int main(int argc, char **argv) {
    Params P;
    g_timing = getenv("TGSF_TIMING") != nullptr;
    Timer T_all, T_ph;
    const bool clean_exit = getenv("TGSF_CLEAN_EXIT") != nullptr; // destroy contexts / free buffers before returning
    if (const char *e = getenv("TGSF_GPUS")) P.gpus = std::max(1, atoi(e));
    if (parse_cmd(argc, argv, &P) == 1) return 1;
    std::vector<uint8_t> contam_seq;
    std::vector<uint64_t> contam_offs;
    if (!P.ContamFile.empty()) {
        if (!load_contam_fasta(P.ContamFile, contam_seq, contam_offs)) { cerr << "Error: Failed to read --contam " << P.ContamFile << endl; return 1; }
        if (contam_offs.size() < 2 || contam_seq.empty()) { cerr << "Error: no sequence in --contam " << P.ContamFile << endl; return 1; }
    }
    for (int i = 0; i < 256; i++) g_comp[i] = 'N';
    const char *pairs[] = {"AT", "GC", "CG", "TA", "at", "gc", "cg", "ta", "MK", "RY", "WW", "SS", "YR", "KM",
                           "mk", "ry", "ww", "ss", "yr", "km"};
    for (const char *p : pairs) g_comp[(unsigned char)p[0]] = p[1];

    P.Infq = file_type(P.InFile);
    if (!P.OutFile.empty() && !P.OnlyQC) {
        P.Outfq = file_type(P.OutFile);
        if (file_ext(P.OutFile) == "gz") P.OUTGZ = true;
    } else {
        P.Outfq = P.FastaOut ? 0 : (P.Infq == 2 ? 1 : P.Infq);
    }
    if (P.Infq == 3 || P.Outfq == 3) {
        cerr << "Error: The file name suffix should be '.[fastq|fq|fasta|fa][.gz] or .[sam|bam]'" << endl;
        if (P.Infq == 3) cerr << "Error: Please check your input file name: " << P.InFile << endl;
        else cerr << "Error: Please check your output file name: " << P.OutFile << endl;
        return 1;
    }
    if (P.Infq == 0 && P.Outfq == 1) { cerr << "Error: Fasta format input file can't output fastq format file" << endl; return 1; }
    const bool has_qual = P.Infq == 1 || P.Infq == 2; // BAM/SAM records carry qualities (read_bam, T.cpp:1872-1916)
    const bool sambam = P.Infq == 2;
#ifndef TGSF_HAVE_HTSLIB
    if (sambam) { // CRAM is recognised by its content, as hts_open does; without htslib it cannot be decoded: fail loudly
        char magic[4] = {0, 0, 0, 0};
        if (FILE *f = fopen(P.InFile.c_str(), "rb")) {
            if (fread(magic, 1, 4, f) != 4) magic[0] = 0;
            fclose(f);
        }
        if (memcmp(magic, "CRAM", 4) == 0) {
            cerr << "Error: CRAM input needs a build with htslib (make -C src HTS_DIR=<htslib prefix>); "
                    "convert with `samtools fastq` or to BAM" << endl;
            return 1;
        }
    }
#endif

    // ---- pre-pass: read_fastx (T.cpp:949-982) + Get_qType (T.cpp:1042-1077) -----------------------
    int checkLen = std::max(std::max(P.EndLen, P.BCLen), 100);
    int minLen = std::max(P.MinLen, 2 * checkLen);
    int maxSeq = std::max(P.ADNum, P.BCNum);
    std::vector<uint8_t> e5, e3;
    int seqNum = 0, minQ = 255, maxQ = 0;
    // One pass over the input: the reader thread parses batches; the pre-pass samples read ends from
    // them as they arrive and keeps them (pageable) for the main pass, which then carries on with the
    // rest of the stream — the reference reads the head of the file twice (T.cpp:949-982, 1845-1870).
    const uint64_t batch_bases = getenv("TGSF_BATCH_MB") ? (uint64_t)atoll(getenv("TGSF_BATCH_MB")) << 20 : P.batch_bases;
    ingest::Queue<std::unique_ptr<ingest::RawBatch>> parsed(4);
    ingest::BatchPool batch_pool;
    std::deque<std::unique_ptr<ingest::RawBatch>> pending;
    bool input_done = false;
    uint64_t pending_bytes = 0;
    // pre-pass: parsed batches are held (pageable host memory) until the sample is complete; past this budget the main pass
    // re-reads the input instead (two-pass mode, like the reference).  Default: a quarter of MemAvailable, at most 24 GB.
    double prepass_mb = 24576.0;
    if (FILE *mi = fopen("/proc/meminfo", "r")) {
        char line[256];
        unsigned long long kb;
        while (fgets(line, sizeof(line), mi))
            if (sscanf(line, "MemAvailable: %llu kB", &kb) == 1) prepass_mb = std::min(prepass_mb, (double)(kb >> 10) / 4.0);
        fclose(mi);
    }
    if (getenv("TGSF_PREPASS_BUFFER_MB")) prepass_mb = atof(getenv("TGSF_PREPASS_BUFFER_MB"));
    const uint64_t prepass_budget = (uint64_t)(prepass_mb * 1048576.0);
    std::thread reader;
    std::unique_ptr<ingest::ParallelReader> preader; // plain files: parallel chunk parser
    auto next_parsed = [&]() { return preader ? preader->pop() : parsed.pop(); };
    std::atomic<bool> reader_stop{false};
    // Leaving main while the reader / writer threads are joinable would call std::terminate; every exit after this point
    // (errors, -A) therefore goes the way the normal end of main goes: flush, then _exit without tearing anything down.
    auto quit = [&](int code) -> int { std::cout.flush(); cerr.flush(); fflush(nullptr); _exit(code); return code; };
    std::function<bool()> start_readers;
    bool two_pass = false; // the pre-pass sample did not fit the buffer budget: the main pass re-reads the input
    const bool stream_input = P.Filter || P.OnlyQC;
    if (stream_input) {
        { gzFile probe = gzopen(P.InFile.c_str(), "rb"); if (!probe) { cerr << "Error: Failed to open file: " << P.InFile << endl; return quit(1); } gzclose(probe); }
        // CUDA context creation (0.4-0.7 s warm, 1.3 s+ for the first process on a box) overlaps the parsing;
        // TGSF_INIT_FIRST=1 creates it before the parser threads start (measured: no faster)
        const bool init_first = getenv("TGSF_INIT_FIRST") != nullptr;
        auto warm_up = [&]() { Timer tw; void *warm = nullptr; if (tgsf_host_alloc(&warm, 1 << 20) == TGSF_OK) tgsf_host_free(warm); tlog("  CUDA context warm-up", tw.lap()); };
        if (init_first) warm_up();
        start_readers = [&]() -> bool {
            if (!sambam && !ingest::ParallelReader::is_gzip(P.InFile) && !getenv("TGSF_SERIAL_READER")) {
                const int hw = (int)std::thread::hardware_concurrency();
                const int nthr = getenv("TGSF_PARSE_THREADS") ? atoi(getenv("TGSF_PARSE_THREADS")) : std::max(1, std::min(8, hw - 2));
                preader.reset(new ingest::ParallelReader(P.InFile, has_qual, 2 * batch_bases, nthr, &batch_pool));
                return preader->ok();
            }
            reader_stop.store(false);
            reader = std::thread(ingest::reader_main, P.InFile, has_qual, batch_bases, &parsed, &batch_pool, &reader_stop, sambam);
            return true;
        };
        if (!start_readers()) { cerr << "Error: Failed to open file: " << P.InFile << endl; return quit(1); }
        if (!init_first) warm_up();
        while (!input_done && seqNum < maxSeq) {
            std::unique_ptr<ingest::RawBatch> rb = next_parsed();
            if (!rb) { input_done = true; break; }
            for (uint32_t i = 0; i < rb->n() && seqNum < maxSeq; i++) {
                const uint64_t s0 = rb->offsets[i];
                const int L = (int)(rb->offsets[i + 1] - s0);
                if (L < minLen) continue;
                seqNum++;
                e5.insert(e5.end(), rb->bases.begin() + s0, rb->bases.begin() + s0 + checkLen);
                for (int j = 0; j < checkLen; j++) e3.push_back((uint8_t)g_comp[rb->bases[s0 + L - 1 - j]]);
                for (int j = 0; j < checkLen && has_qual; j++) {
                    char q = (char)rb->quals[s0 + j];
                    if (minQ > q) minQ = q;
                    if (maxQ < q) maxQ = q;
                }
            }
            // The sampled reads are kept for the main pass (one pass over the input) while they fit the budget;
            // beyond it the pre-pass goes on without keeping them and the input is read again, like the
            // reference does (T.cpp:949-982 then 1845-1916).
            if (!two_pass) {
                pending_bytes += rb->bases.size() + rb->quals.size();
                pending.push_back(std::move(rb));
                if (pending_bytes > prepass_budget) {
                    two_pass = true;
                    for (auto &pb : pending) batch_pool.put(std::move(pb));
                    pending.clear();
                }
            } else {
                batch_pool.put(std::move(rb));
            }
        }
        if (two_pass) { // restart the input from its beginning
            if (preader) preader.reset();
            if (reader.joinable()) {
                reader_stop.store(true);
                while (!input_done) { if (!parsed.pop()) input_done = true; }
                reader.join();
            }
            input_done = false;
            if (!start_readers()) { cerr << "Error: Failed to open file: " << P.InFile << endl; return quit(1); }
        }
    } else { // -F: only the sample is needed here; DownSampleTask reads the file itself
        FastxReader rd(P.InFile);
        if (!rd.ok()) { cerr << "Error: Failed to open file: " << P.InFile << endl; return quit(1); }
        string name, seq, qual;
        while (rd.read(name, seq, qual)) {
            int L = (int)seq.size();
            if (L < minLen) continue;
            if (seqNum >= maxSeq) break;
            seqNum++;
            for (int i = 0; i < checkLen && has_qual; i++) {
                char q = qual[i];
                if (minQ > q) minQ = q;
                if (maxQ < q) maxQ = q;
            }
        }
    }
    tlog("prepass sampling (incl. CUDA context)", T_ph.lap());
    int qType = 0;
    if (has_qual) {
        if (minQ >= 33 && minQ <= 78 && maxQ >= 33 && maxQ <= 127) qType = 33;
        else if (minQ >= 64 && minQ <= 108 && maxQ >= 64 && maxQ <= 127) qType = 64;
        else if (minQ < 55) qType = 33;
        else qType = 64;
        cerr << "INFO: base quality scoring: Phred" << qType << endl;
        minQ -= qType;
        maxQ -= qType;
        if (P.MinQ >= 0) {
            if (P.MinQ >= maxQ) {
                cerr << "Warning: max base quality score was: " << maxQ << endl;
                cerr << "INFO: Please reset -q parameter." << endl;
                exit(-1);
            }
        } else {
            if (maxQ > 10 && P.readType == "clr") P.MinQ = 10;
            else if (maxQ > 20 && P.readType == "hifi") P.MinQ = 20;
            else if (maxQ > 10 && P.readType == "ont") P.MinQ = 10;
            else P.MinQ = 0;
        }
    }

    std::vector<string> adapters; // the global `adapters` set (T.cpp:1324); the order is irrelevant for the results
    // ... but Get_adapters prints the set in std::unordered_set iteration order (T.cpp:2937-2940): the same container with the
    // same insertions (same libstdc++ hash and rehash policy) reproduces that order for the `input adapter` lines
    std::unordered_set<string> adapter_set;
    auto add_adapter = [&](const string &a) { if (adapter_set.insert(a).second) adapters.push_back(a); };
    if (P.Filter) {
        std::vector<int32_t> bn5((size_t)checkLen * 4), bn3((size_t)checkLen * 4);
        std::vector<int64_t> m5(TGSF_LIB_ADAPTERS, 0), m3(TGSF_LIB_ADAPTERS, 0);
        std::vector<const uint8_t *> lib_seq;
        std::vector<int32_t> lib_len;
        for (const char *a : kLib) { lib_seq.push_back((const uint8_t *)a); lib_len.push_back((int32_t)strlen(a)); }
        const bool search = P.AdapterFile.empty();
        const uint8_t dummy = 0;
        if (tgsf_prepass(0, seqNum ? e5.data() : &dummy, seqNum ? e3.data() : &dummy, (uint32_t)seqNum, (uint32_t)checkLen,
                         search ? lib_seq.data() : nullptr, lib_len.data(), TGSF_LIB_ADAPTERS, P.MidSim, bn5.data(),
                         bn3.data(), m5.data(), m3.data()) != TGSF_OK)
            die_tgsf("tgsf_prepass");
        // Both CheckBaseContent threads clamp trim5p to BCLen BEFORE storing their own result
        // (T.cpp:1136-1144), so the 5' trim is clamped only if the 3' thread finishes after the 5' one
        // has stored it: a race in the reference.  Resolved here in thread-creation order (5' first).
        const bool auto5 = P.HeadTrim < 0, auto3 = P.TailTrim < 0;
        if (auto5) P.HeadTrim = base_content_trim(bn5, checkLen, seqNum, P.EndBias);
        if (auto3) {
            if (auto5 && P.HeadTrim > P.BCLen) P.HeadTrim = P.BCLen;
            P.TailTrim = base_content_trim(bn3, checkLen, seqNum, P.EndBias);
        }
        cerr << "INFO: trim 5' end length: " << P.HeadTrim << endl;
        cerr << "INFO: trim 3' end length: " << P.TailTrim << endl;
        cerr << "INFO: min output reads length: " << P.MinLen << endl;
        if (has_qual) cerr << "INFO: min Phred average quality score: " << P.MinQ << endl;
        if (!search) { // Get_adapters, T.cpp:2923-2942
            FastxReader ar(P.AdapterFile);
            string name, seq, qual;
            while (ar.read(name, seq, qual)) { add_adapter(seq); add_adapter(rev_comp(seq)); }
            int num = 0;
            for (const string &a : adapter_set) cerr << "INFO: input adapter " << ++num << " :" << a << endl;
        } else { // tail of adapterSearch (T.cpp:1178-1208) + selection (T.cpp:3081-3125)
            float minSim = P.MidSim;
            if (minSim < 0.9) minSim = 0.9;
            auto pick = [&](const std::vector<int64_t> &maps, string &ad, float &dep) {
                int best = -1;
                for (int i = 0; i < TGSF_LIB_ADAPTERS; i++)
                    if (maps[i] > 0 && (best < 0 || maps[i] > maps[best])) best = i;
                ad.clear();
                dep = 0;
                if (best >= 0) {
                    float meanDep = static_cast<float>((int)maps[best]) / strlen(kLib[best]);
                    if (meanDep >= 2 * minSim) { ad = kLib[best]; dep = meanDep; }
                }
            };
            string a5, a3;
            float d5, d3;
            pick(m5, a5, d5);
            pick(m3, a3, d3);
            if (d5 > 5 * d3) { a3 = ""; d3 = 0; }
            else if (d3 > 5 * d5) { a5 = ""; d5 = 0; }
            cerr << "INFO: 5' adapter: " << a5 << endl;
            cerr << "INFO: 3' adapter: " << a3 << endl;
            cerr << "INFO: mean depth of 5' adapter: " << d5 << endl;
            cerr << "INFO: mean depth of 3' adapter: " << d3 << endl;
            if (P.ONLYAD) return quit(0);
            if (!a5.empty()) { add_adapter(a5); add_adapter(rev_comp(a5)); }
            if (!a3.empty()) { add_adapter(a3); add_adapter(rev_comp(a3)); }
            if (a5.empty() && a3.empty()) {
                if (P.readType == "hifi" || P.readType == "clr") {
                    add_adapter(kLib[0]); add_adapter(kLib[1]);
                    cerr << "INFO: set PacBio blunt adapter to trim: " << kLib[0] << endl;
                } else if (P.readType == "ont") {
                    add_adapter(kLib[8]); add_adapter(kLib[9]);
                    cerr << "INFO: set NanoPore rapid adapter to trim: " << kLib[8] << endl;
                }
            }
        }
    }

    uint64_t cleanNum = 0, cleanBases = 0, rawNum = 0, rawBases = 0;
    uint64_t contamNum = 0, contamBases = 0; // pieces discarded by the contaminant screen (--contam)
    std::vector<int> rawLens, cleanLens;       // T.cpp:1794
    report::Side rawSide, cleanSide;
    string tmpPath;
    RecIndex recIdx;
    // Filter + downsample: the filtered records are kept in host memory for the second pass (sequence / quality bytes
    // back to back + one entry per record); only past TGSF_DOWNSAMPLE_BUFFER_MB (default: a quarter of MemAvailable, at
    // most 64 GB) they are spilled to the reference's uncompressed tmp file (T.cpp:3129-3137) and the run continues there.
    struct MemRec { uint64_t off; uint32_t len; uint32_t name; };
    std::vector<MemRec> mem_recs;
    std::vector<string> mem_names;
    string mem_seq, mem_qual;
    bool mem_mode = false;
    uint64_t mem_budget = 0;
    if (P.Filter || P.OnlyQC) {
    tlog("gpu prepass + resolve", T_ph.lap());
    // ---- contexts: one per GPU ---------------------------------------------------------------------
    tgsf_params tp;
    memset(&tp, 0, sizeof(tp));
    tp.min_len = P.MinLen; tp.max_len = P.MaxLen; tp.min_q = P.MinQ; tp.max_q = P.MaxQ;
    tp.bc_len = P.BCLen; tp.head_trim = P.HeadTrim; tp.tail_trim = P.TailTrim;
    tp.end_len = P.EndLen; tp.end_match_len = P.EndMatchLen; tp.mid_match_len = P.MidMatchLen;
    tp.extra_len = P.ExtraLen; tp.end_sim = P.EndSim; tp.mid_sim = P.MidSim;
    tp.kmer = P.Kmer; tp.min_repeat = P.MinRepeat; tp.qtype = qType;
    tp.flags = (P.Filter ? TGSF_FLAG_FILTER : 0) | (P.OnlyQC ? TGSF_FLAG_ONLY_QC : 0) | (P.discard ? TGSF_FLAG_DISCARD_MID : 0);
    // .gz output: the deflate blocks of every record are produced on the GPU (TGSF_GZ_HOST=1: host zlib instead)
    const bool gz_gpu = P.OUTGZ && !P.Downsample && !P.OnlyQC && !getenv("TGSF_GZ_HOST");
    if (gz_gpu) tp.flags |= TGSF_FLAG_GZ_BLOCKS | (P.Outfq == 1 ? 0u : TGSF_FLAG_GZ_FASTA);
    std::vector<const uint8_t *> aseq;
    std::vector<int32_t> alen;
    for (const string &a : adapters) { aseq.push_back((const uint8_t *)a.data()); alen.push_back((int32_t)a.size()); }
    tp.n_adapters = (int32_t)aseq.size();
    tp.adapter_seq = aseq.data();
    tp.adapter_len = alen.data();
    tp.n_slots = 2;
    std::vector<tgsf_ctx *> ctx((size_t)P.gpus, nullptr);
    int n_dev = 0;
    if (tgsf_device_count(&n_dev) != TGSF_OK || n_dev < 1) die_tgsf("tgsf_device_count");
    // TGSF_SHARE_DEVICES=1: more contexts than devices are placed round-robin (context g on device g % devices), so
    // the multi-GPU path (batch dealing, per-context counters, tgsf_allreduce) can run on a single-GPU box
    const bool share_dev = getenv("TGSF_SHARE_DEVICES") != nullptr;
    if (P.gpus > n_dev && !share_dev) {
        cerr << "Error: --gpus " << P.gpus << " but only " << n_dev << " CUDA device(s) are visible" << endl;
        return quit(1);
    }
    for (int g = 0; g < P.gpus; g++)
        if (tgsf_create(g % n_dev, &tp, &ctx[(size_t)g]) != TGSF_OK) die_tgsf("tgsf_create");
    if (!P.ContamFile.empty()) {
        uint64_t n_kmers = 0;
        for (int g = 0; g < P.gpus; g++)
            if (tgsf_set_contaminants(ctx[(size_t)g], contam_seq.data(), contam_offs.data(), (uint32_t)(contam_offs.size() - 1),
                                      P.ContamK, P.ContamFrac, &n_kmers) != TGSF_OK)
                die_tgsf("tgsf_set_contaminants");
        cerr << "INFO: " << n_kmers << " distinct " << P.ContamK << "-mers loaded from " << P.ContamFile << "." << endl;
        std::vector<uint8_t>().swap(contam_seq);
    }

    tlog("tgsf_create", T_ph.lap());
    // ---- main pass -----------------------------------------------------------------------------------
    FILE *out = stdout;
    auto open_tmp = [&]() -> bool { // uncompressed tmp file like T.cpp:3129-3137
        string prefix = P.InFile;
        tmpPath = prefix + ".tmp." + std::to_string((long)getpid()) + (P.Outfq == 0 ? ".fa" : ".fq");
        out = fopen(tmpPath.c_str(), "wb");
        if (!out) { cerr << "Error: Failed to open file: " << tmpPath << endl; return false; }
        return true;
    };
    if (P.Downsample) {
        uint64_t avail_mb = 0;
        if (FILE *mi = fopen("/proc/meminfo", "r")) {
            char line[256];
            while (fgets(line, sizeof(line), mi)) { unsigned long long kb; if (sscanf(line, "MemAvailable: %llu kB", &kb) == 1) avail_mb = kb >> 10; }
            fclose(mi);
        }
        uint64_t mb = std::min<uint64_t>(avail_mb / 4, 65536);
        if (const char *e = getenv("TGSF_DOWNSAMPLE_BUFFER_MB")) mb = strtoull(e, nullptr, 10);
        mem_budget = mb << 20;
        mem_mode = mem_budget > 0;
        if (!mem_mode && !open_tmp()) return quit(1);
    } else if (!P.OnlyQC && !P.OutFile.empty()) {
        out = fopen(P.OutFile.c_str(), "w+b"); // read-write: the plain writer maps the file
        if (!out) { cerr << "Error: Failed to open file: " << P.OutFile << endl; return quit(1); }
    }
    const bool gz_now = P.OUTGZ && !P.Downsample; // T.cpp:2022
    // pinned staging ring: what crosses PCIe (2-bit packed bases, Phred bytes); 2 slots per GPU
    struct PinSlot {
        uint8_t *packed = nullptr, *quals = nullptr;
        size_t cap = 0;
        std::vector<uint64_t> exc_pos;
        std::vector<uint8_t> exc_byte;
        std::unique_ptr<ingest::RawBatch> rb;
        bool reserve(size_t bases) {
            if (bases <= cap) return true;
            tgsf_host_free(packed);
            tgsf_host_free(quals);
            cap = bases + bases / 4 + (1 << 20);
            return tgsf_host_alloc((void **)&packed, cap / 4 + 64) == TGSF_OK && tgsf_host_alloc((void **)&quals, cap) == TGSF_OK;
        }
    };
    const int slots = 2 * P.gpus;
    std::vector<PinSlot> ring((size_t)slots);
    std::deque<int> inflight; // ring indices in submission order; slot i runs on GPU (i % gpus)

    // writer thread (T.cpp:2011-2053): numbers the emitted pieces of a retired batch, then
    //  * plain output: gathers name/bases/qualities straight out of the batch with (p)writev, no
    //    formatting copy; a regular file is written by several threads at precomputed offsets;
    //  * gzip output: one member per record like DeflateCompress (T.cpp:786-812), the records of a
    //    batch spread over -t compressor threads, written in order;
    //  * downsampling: the serial path (uncompressed tmp file + record index).
    struct WriteJob {
        std::unique_ptr<ingest::RawBatch> rb;
        std::vector<tgsf_piece> pieces;
        uint8_t *gz_blob = nullptr;        // GPU deflate blocks of the batch (gz_gpu): pinned, recycled through gz_pool
        size_t gz_cap = 0;
        std::vector<tgsf_gz_span> gz_spans; // per piece
        bool gz_ok = false;
    };
    struct PinnedPool { // pinned host buffers for the deflate blobs (a pageable target costs page faults + a staged copy)
        std::mutex m;
        std::vector<std::pair<uint8_t *, size_t>> free_;
        std::pair<uint8_t *, size_t> get(size_t need) {
            {
                std::lock_guard<std::mutex> lk(m);
                for (size_t i = 0; i < free_.size(); ++i)
                    if (free_[i].second >= need) { auto r = free_[i]; free_.erase(free_.begin() + (long)i); return r; }
                if (!free_.empty()) { tgsf_host_free(free_.back().first); free_.pop_back(); }
            }
            void *p = nullptr;
            const size_t cap = need + need / 4;
            if (tgsf_host_alloc(&p, cap) != TGSF_OK) return {nullptr, 0};
            return {(uint8_t *)p, cap};
        }
        void put(uint8_t *p, size_t cap) {
            if (!p) return;
            std::lock_guard<std::mutex> lk(m);
            free_.emplace_back(p, cap);
        }
    } gz_pool;
    struct Emit { uint32_t read, start, len; int pass; uint32_t piece; };
    ingest::Queue<std::unique_ptr<WriteJob>> to_write(4);
    const int out_threads = std::max(1, std::min(P.n_thread, (int)std::thread::hardware_concurrency()));
    fflush(out);
    const int out_fd = fileno(out);
    struct stat out_st;
    // positioned parallel writes only into a file this process created (stdout may be in append mode)
    const bool out_regular = out != stdout && fstat(out_fd, &out_st) == 0 && S_ISREG(out_st.st_mode) && !getenv("TGSF_SERIAL_WRITER");
    uint64_t out_off = 0; // regular file: bytes written so far
    bool out_mmap = !getenv("TGSF_NO_MMAP_OUT");
    std::thread writer([&]() {
        string obuf, rec, gz;
        std::vector<Emit> emits;
        std::vector<string> renamed; // names with a :N suffix, alive until the batch is written
        std::vector<string> bufs;
        int gz_strategy = Z_DEFAULT_STRATEGY;
        unsigned gz_batches = 0;
        while (true) {
            std::unique_ptr<WriteJob> job = to_write.pop();
            if (!job) break;
            const ingest::RawBatch &b = *job->rb;
            emits.clear();
            renamed.clear();
            uint32_t last = UINT32_MAX;
            int pass = 1;
            for (size_t pi = 0; pi < job->pieces.size(); ++pi) { // T.cpp:1976-2059
                const tgsf_piece &p = job->pieces[pi];
                if ((uint32_t)p.read != last) { last = (uint32_t)p.read; pass = 1; }
                if (p.status == TGSF_PIECE_CONTAM) { contamNum++; contamBases += (uint64_t)p.len; }
                if (p.status != TGSF_PIECE_EMIT) continue;
                emits.push_back(Emit{last, (uint32_t)p.start, (uint32_t)p.len, pass, (uint32_t)pi});
                pass++;
                cleanNum++;
                cleanBases += (uint64_t)p.len;
                cleanLens.push_back(p.len);
            }
            // names: pass 1 keeps the raw name, later pieces get ":N" before the first blank
            std::vector<const string *> nm(emits.size());
            {
                size_t nren = 0;
                for (const Emit &e : emits) nren += e.pass >= 2;
                renamed.reserve(nren);
                for (size_t i = 0; i < emits.size(); ++i) {
                    if (emits[i].pass >= 2) { renamed.push_back(new_seq_name(b.names[emits[i].read], emits[i].pass)); nm[i] = &renamed.back(); }
                    else nm[i] = &b.names[emits[i].read];
                }
            }
            auto format_rec = [&](size_t i, string &dst) {
                const Emit &e = emits[i];
                const char *sq = (const char *)b.bases.data() + b.offsets[e.read] + e.start;
                if (P.Outfq == 1) {
                    const char *q = (const char *)b.quals.data() + b.offsets[e.read] + e.start;
                    dst += '@'; dst += *nm[i]; dst += '\n'; dst.append(sq, e.len); dst += "\n+\n"; dst.append(q, e.len); dst += '\n';
                } else {
                    dst += '>'; dst += *nm[i]; dst += '\n'; dst.append(sq, e.len); dst += '\n';
                }
            };
            if (P.Downsample && mem_mode) {
                for (size_t i = 0; i < emits.size(); ++i) {
                    const Emit &e = emits[i];
                    const char *sq = (const char *)b.bases.data() + b.offsets[e.read] + e.start;
                    mem_recs.push_back(MemRec{(uint64_t)mem_seq.size(), (uint32_t)e.len, (uint32_t)mem_names.size()});
                    mem_names.push_back(*nm[i]);
                    mem_seq.append(sq, e.len);
                    if (P.Outfq == 1) mem_qual.append((const char *)b.quals.data() + b.offsets[e.read] + e.start, e.len);
                    recIdx.add(*nm[i], (int)e.len);
                }
                if (mem_seq.size() + mem_qual.size() > mem_budget) { // over budget: spill what is buffered, continue on the file
                    if (!open_tmp()) { cerr.flush(); fflush(nullptr); _exit(1); } // (writer thread: leave like quit())
                    {
                        string rec;
                        for (const MemRec &r : mem_recs) {
                            rec.clear();
                            if (P.Outfq == 1) { rec += '@'; rec += mem_names[r.name]; rec += '\n'; rec.append(mem_seq, r.off, r.len); rec += "\n+\n"; rec.append(mem_qual, r.off, r.len); rec += '\n'; }
                            else { rec += '>'; rec += mem_names[r.name]; rec += '\n'; rec.append(mem_seq, r.off, r.len); rec += '\n'; }
                            fwrite(rec.data(), 1, rec.size(), out);
                        }
                    }
                    mem_mode = false;
                    mem_recs.clear(); mem_recs.shrink_to_fit();
                    mem_names.clear(); mem_names.shrink_to_fit();
                    string().swap(mem_seq); string().swap(mem_qual);
                }
            } else if (P.Downsample) {
                for (size_t i = 0; i < emits.size(); ++i) {
                    format_rec(i, obuf);
                    recIdx.add(*nm[i], (int)emits[i].len);
                    if (obuf.size() >= (8u << 20)) { fwrite(obuf.data(), 1, obuf.size(), out); obuf.clear(); }
                }
                if (!obuf.empty()) { fwrite(obuf.data(), 1, obuf.size(), out); obuf.clear(); }
            } else if (!emits.empty()) {
                // split the records into contiguous ranges of about equal payload
                const int K = gz_now ? out_threads : (out_regular ? std::min(out_threads, 8) : 1);
                std::vector<size_t> cut((size_t)K + 1, emits.size());
                std::vector<uint64_t> bytes_before((size_t)K + 1, 0);
                {
                    uint64_t total = 0;
                    for (const Emit &e : emits) total += e.len;
                    uint64_t acc = 0, raw = 0;
                    int k = 0;
                    cut[0] = 0;
                    for (size_t i = 0; i < emits.size(); ++i) {
                        while (k + 1 < K && acc >= total * (uint64_t)(k + 1) / (uint64_t)K) { cut[(size_t)++k] = i; bytes_before[(size_t)k] = raw; }
                        acc += emits[i].len;
                        const uint64_t nl = nm[i]->size();
                        raw += P.Outfq == 1 ? 1 + nl + 1 + emits[i].len + 3 + emits[i].len + 1 : 1 + nl + 1 + emits[i].len + 1;
                    }
                    while (k + 1 < K) { cut[(size_t)++k] = emits.size(); bytes_before[(size_t)k] = raw; }
                    bytes_before[(size_t)K] = raw;
                }
                if (gz_now && job->gz_ok) {
                    // members around the GPU's deflate blocks: gzip header | stored block with the header line |
                    // blocks | CRC-32, ISIZE (include/tgsf.h, tgsf_collect_gz); CRC and copies spread over -t threads
                    bufs.resize((size_t)K);
                    auto assemble_range = [&](int k) {
                        string &dst = bufs[(size_t)k];
                        dst.clear();
                        static const unsigned char kHdr[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff};
                        for (size_t i = cut[(size_t)k]; i < cut[(size_t)k + 1]; ++i) {
                            const Emit &e = emits[i];
                            const tgsf_gz_span &sp = job->gz_spans[e.piece];
                            const Bytef *sq = (const Bytef *)b.bases.data() + b.offsets[e.read] + e.start;
                            const size_t hl = nm[i]->size() + 2;
                            string head;
                            head += P.Outfq == 1 ? '@' : '>';
                            head += *nm[i];
                            head += '\n';
                            uLong crc = crc32(0L, (const Bytef *)head.data(), (uInt)hl);
                            crc = crc32(crc, sq, (uInt)e.len);
                            uint64_t isize = hl + e.len + 1;
                            if (P.Outfq == 1) {
                                crc = crc32(crc, (const Bytef *)"\n+\n", 3);
                                crc = crc32(crc, (const Bytef *)b.quals.data() + b.offsets[e.read] + e.start, (uInt)e.len);
                                isize += 2 + e.len + 1;
                            }
                            crc = crc32(crc, (const Bytef *)"\n", 1);
                            dst.append((const char *)kHdr, 10);
                            // stored blocks hold at most 65535 bytes: header lines are far shorter, but stay correct
                            size_t done = 0;
                            while (done < hl) {
                                const size_t n = std::min<size_t>(hl - done, 65535);
                                const unsigned char sb[5] = {0, (unsigned char)n, (unsigned char)(n >> 8), (unsigned char)~n, (unsigned char)(~n >> 8)};
                                dst.append((const char *)sb, 5);
                                dst.append(head.data() + done, n);
                                done += n;
                            }
                            dst.append((const char *)job->gz_blob + sp.offset, sp.bytes);
                            const uint32_t tr[2] = {(uint32_t)crc, (uint32_t)isize};
                            dst.append((const char *)tr, 8);
                        }
                    };
                    std::vector<std::thread> th;
                    for (int k = 1; k < K; ++k) th.emplace_back(assemble_range, k);
                    assemble_range(0);
                    for (auto &t : th) t.join();
                    for (int k = 0; k < K; ++k) {
                        const string &d = bufs[(size_t)k];
                        size_t done = 0;
                        while (done < d.size()) {
                            const ssize_t w = write(out_fd, d.data() + done, d.size() - done);
                            if (w <= 0) { cerr << "Error: write failed" << endl; exit(-1); }
                            done += (size_t)w;
                        }
                    }
                } else if (gz_now) {
                    bufs.resize((size_t)K);
                    // Per-record members hold no cross-record matches, and on noisy long reads zlib's match
                    // search at the default strategy yields files no smaller than run-length + Huffman coding
                    // (Z_RLE), at 6-9x the time.  Sampled every 16th batch: Z_RLE is used while it stays
                    // within 1 % of the size the requested level gives on the sample.
                    if ((gz_batches++ & 15) == 0 && !getenv("TGSF_GZ_DEFAULT_STRATEGY")) {
                        const size_t ns = std::min<size_t>(16, emits.size());
                        std::vector<uint64_t> sz_def(ns, 0), sz_rle(ns, 0);
                        auto probe = [&](size_t a) {
                            string r, o;
                            format_rec(a * emits.size() / ns, r);
                            for (int which = 0; which < 2; ++which) {
                                z_stream zs;
                                memset(&zs, 0, sizeof(zs));
                                if (deflateInit2(&zs, P.compLevel, Z_DEFLATED, 15 + 16, 8, which ? Z_RLE : Z_DEFAULT_STRATEGY) != Z_OK) return;
                                o.resize(deflateBound(&zs, r.size()) + 32);
                                zs.next_in = (Bytef *)r.data();
                                zs.avail_in = (uInt)r.size();
                                zs.next_out = (Bytef *)&o[0];
                                zs.avail_out = (uInt)o.size();
                                deflate(&zs, Z_FINISH);
                                (which ? sz_rle : sz_def)[a] = zs.total_out;
                                deflateEnd(&zs);
                            }
                        };
                        std::vector<std::thread> pth;
                        for (size_t a = 1; a < ns; ++a) pth.emplace_back(probe, a);
                        probe(0);
                        for (auto &t : pth) t.join();
                        uint64_t sd = 0, sr = 0;
                        for (size_t a = 0; a < ns; ++a) { sd += sz_def[a]; sr += sz_rle[a]; }
                        gz_strategy = (sr * 100 <= sd * 101) ? Z_RLE : Z_DEFAULT_STRATEGY;
                    }
                    const int strategy = gz_strategy;
                    auto compress_range = [&](int k) {
                        string &dst = bufs[(size_t)k];
                        dst.clear();
                        string r;
                        z_stream zs;
                        memset(&zs, 0, sizeof(zs));
                        if (deflateInit2(&zs, P.compLevel, Z_DEFLATED, 15 + 16, 8, strategy) != Z_OK) return;
                        for (size_t i = cut[(size_t)k]; i < cut[(size_t)k + 1]; ++i) {
                            r.clear();
                            format_rec(i, r);
                            deflateReset(&zs);
                            const size_t at = dst.size(), bound = deflateBound(&zs, r.size()) + 32;
                            dst.resize(at + bound);
                            zs.next_in = (Bytef *)r.data();
                            zs.avail_in = (uInt)r.size();
                            zs.next_out = (Bytef *)&dst[at];
                            zs.avail_out = (uInt)bound;
                            deflate(&zs, Z_FINISH);
                            dst.resize(at + zs.total_out);
                        }
                        deflateEnd(&zs);
                    };
                    std::vector<std::thread> th;
                    for (int k = 1; k < K; ++k) th.emplace_back(compress_range, k);
                    compress_range(0);
                    for (auto &t : th) t.join();
                    for (int k = 0; k < K; ++k) {
                        const string &d = bufs[(size_t)k];
                        size_t done = 0;
                        while (done < d.size()) {
                            const ssize_t w = write(out_fd, d.data() + done, d.size() - done);
                            if (w <= 0) { cerr << "Error: write failed" << endl; exit(-1); }
                            done += (size_t)w;
                        }
                    }
                } else {
                    static const char kAt = '@', kGt = '>', kNl = '\n';
                    static const char kPlus[] = "\n+\n";
                    auto write_range = [&](int k) {
                        std::vector<struct iovec> iov;
                        iov.reserve(1024);
                        uint64_t off = out_off + bytes_before[(size_t)k];
                        auto flush = [&]() {
                            size_t first = 0;
                            while (first < iov.size()) {
                                const int cnt = (int)std::min<size_t>(iov.size() - first, 1024);
                                ssize_t w = out_regular ? pwritev(out_fd, iov.data() + first, cnt, (off_t)off) : writev(out_fd, iov.data() + first, cnt);
                                if (w <= 0) { cerr << "Error: write failed" << endl; exit(-1); }
                                off += (uint64_t)w;
                                while (w > 0 && first < iov.size()) { // advance over what was written
                                    if ((size_t)w >= iov[first].iov_len) { w -= (ssize_t)iov[first].iov_len; ++first; }
                                    else { iov[first].iov_base = (char *)iov[first].iov_base + w; iov[first].iov_len -= (size_t)w; w = 0; }
                                }
                            }
                            iov.clear();
                        };
                        auto add = [&](const void *ptr, size_t n) { iov.push_back({(void *)ptr, n}); };
                        for (size_t i = cut[(size_t)k]; i < cut[(size_t)k + 1]; ++i) {
                            const Emit &e = emits[i];
                            const uint8_t *sq = b.bases.data() + b.offsets[e.read] + e.start;
                            if (iov.size() + 7 > 1024) flush();
                            add(P.Outfq == 1 ? &kAt : &kGt, 1);
                            add(nm[i]->data(), nm[i]->size());
                            add(&kNl, 1);
                            add(sq, e.len);
                            if (P.Outfq == 1) {
                                add(kPlus, 3);
                                add(b.quals.data() + b.offsets[e.read] + e.start, e.len);
                            }
                            add(&kNl, 1);
                        }
                        flush();
                    };
                    // A regular file takes its inode lock for every buffered write, so positioned writes from
                    // several threads serialise.  Preferred path: reserve the batch's byte range (fallocate, so a
                    // full disk is an error here and not a SIGBUS later), map it and let the threads copy their
                    // records into the mapping; the pwritev path stays as the fallback (pipes, odd filesystems).
                    bool mapped = false;
                    const uint64_t nbytes = bytes_before[(size_t)K];
                    if (out_regular && out_mmap && nbytes) {
                        const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE);
                        const uint64_t map_off = out_off & ~(page - 1), delta = out_off - map_off;
                        if (fallocate(out_fd, 0, (off_t)out_off, (off_t)nbytes) == 0) {
                            void *m = mmap(nullptr, (size_t)(nbytes + delta), PROT_READ | PROT_WRITE, MAP_SHARED, out_fd, (off_t)map_off);
                            if (m != MAP_FAILED) {
                                auto copy_range = [&](int k) {
                                    char *dst = (char *)m + delta + bytes_before[(size_t)k];
                                    for (size_t i = cut[(size_t)k]; i < cut[(size_t)k + 1]; ++i) {
                                        const Emit &e = emits[i];
                                        *dst++ = P.Outfq == 1 ? '@' : '>';
                                        memcpy(dst, nm[i]->data(), nm[i]->size()); dst += nm[i]->size();
                                        *dst++ = '\n';
                                        memcpy(dst, b.bases.data() + b.offsets[e.read] + e.start, e.len); dst += e.len;
                                        if (P.Outfq == 1) {
                                            memcpy(dst, kPlus, 3); dst += 3;
                                            memcpy(dst, b.quals.data() + b.offsets[e.read] + e.start, e.len); dst += e.len;
                                        }
                                        *dst++ = '\n';
                                    }
                                };
                                std::vector<std::thread> th;
                                for (int k = 1; k < K; ++k) th.emplace_back(copy_range, k);
                                copy_range(0);
                                for (auto &t : th) t.join();
                                munmap(m, (size_t)(nbytes + delta));
                                mapped = true;
                            }
                        } else {
                            out_mmap = false; // filesystem without fallocate: keep to pwritev
                        }
                    }
                    if (!mapped) {
                        std::vector<std::thread> th;
                        for (int k = 1; k < K; ++k) th.emplace_back(write_range, k);
                        write_range(0);
                        for (auto &t : th) t.join();
                    }
                    out_off += nbytes;
                }
            }
            batch_pool.put(std::move(job->rb));
            gz_pool.put(job->gz_blob, job->gz_cap);
        }
    });

    std::vector<tgsf_read_result> rr;
    auto retire = [&]() {
        const int bi = inflight.front();
        inflight.pop_front();
        PinSlot &sl = ring[(size_t)bi];
        tgsf_ctx *c = ctx[(size_t)(bi % P.gpus)];
        const uint32_t n = sl.rb->n();
        std::unique_ptr<WriteJob> job(new WriteJob());
        rr.resize(n);
        job->pieces.resize((size_t)n + 4096);
        uint32_t np = 0;
        if (gz_gpu) { // before tgsf_collect, which retires the batch
            uint64_t nb = 0;
            uint32_t ns = 0;
            auto pb = gz_pool.get((size_t)(sl.rb->bases.size() * (has_qual && P.Outfq == 1 ? 1.0 : 0.5) + (1u << 20)));
            job->gz_blob = pb.first;
            job->gz_cap = pb.second;
            job->gz_spans.resize((size_t)n + 4096);
            int grc = job->gz_blob ? tgsf_collect_gz(c, job->gz_blob, job->gz_cap, &nb, job->gz_spans.data(), (uint32_t)job->gz_spans.size(), &ns)
                                   : TGSF_ERR_NOMEM;
            if (grc == TGSF_ERR_CAPACITY) {
                gz_pool.put(job->gz_blob, job->gz_cap);
                pb = gz_pool.get((size_t)nb + 16);
                job->gz_blob = pb.first;
                job->gz_cap = pb.second;
                job->gz_spans.resize((size_t)ns + 16);
                grc = job->gz_blob ? tgsf_collect_gz(c, job->gz_blob, job->gz_cap, &nb, job->gz_spans.data(), (uint32_t)job->gz_spans.size(), &ns)
                                   : TGSF_ERR_NOMEM;
            }
            job->gz_ok = grc == TGSF_OK; // otherwise (region-pool re-run, no pinned memory) the host compresses this batch
        }
        int rc = tgsf_collect(c, rr.data(), n, job->pieces.data(), (uint32_t)job->pieces.size(), &np);
        if (rc == TGSF_ERR_CAPACITY && np > job->pieces.size()) {
            job->pieces.resize(np);
            rc = tgsf_collect(c, rr.data(), n, job->pieces.data(), (uint32_t)job->pieces.size(), &np);
        }
        if (rc != TGSF_OK) die_tgsf("tgsf_collect");
        job->pieces.resize(np);
        job->rb = std::move(sl.rb);
        to_write.push(std::move(job));
    };
    const int stage_threads = getenv("TGSF_STAGE_THREADS") ? std::max(1, atoi(getenv("TGSF_STAGE_THREADS"))) : 4;
    const int stage_shift = getenv("TGSF_STAGE_MIN_SHIFT") ? std::max(6, atoi(getenv("TGSF_STAGE_MIN_SHIFT"))) : 22; // >= 4 Mbases per thread
    int cur = 0;
    double t_wait_in = 0, t_pack = 0, t_copy = 0, t_submit = 0, t_retire = 0;
    Timer T_loop;
    while (true) {
        std::unique_ptr<ingest::RawBatch> rb;
        T_loop.lap();
        if (!pending.empty()) { rb = std::move(pending.front()); pending.pop_front(); }
        else if (!input_done) { rb = next_parsed(); if (!rb) input_done = true; }
        if (!rb) break;
        t_wait_in += T_loop.lap();
        const uint32_t n = rb->n();
        const uint64_t nb = rb->bases.size();
        rawNum += n;
        rawBases += nb;
        for (uint32_t i = 0; i < n; i++) rawLens.push_back((int)(rb->offsets[i + 1] - rb->offsets[i]));
        T_loop.lap();
        if ((int)inflight.size() == slots) retire(); // ring slot `cur` is the oldest one in flight
        t_retire += T_loop.lap();
        PinSlot &sl = ring[(size_t)cur];
        if (!sl.reserve((size_t)nb + 64)) { cerr << "Error: out of pinned host memory" << endl; return quit(1); }
        // pack the bases (2 bits) and copy the qualities into the pinned slot on a few threads: the ranges are
        // multiples of 32 bases, their exception lists are concatenated with the range offset added
        uint64_t ne = 0;
        {
            const int T = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)stage_threads, nb >> stage_shift));
            const uint64_t chunk = ((nb / (uint64_t)T + 31) / 32) * 32;
            std::vector<std::vector<uint64_t>> xp((size_t)T);
            std::vector<std::vector<uint8_t>> xb((size_t)T);
            std::vector<int> rcs((size_t)T, TGSF_OK);
            auto stage = [&](int t) {
                const uint64_t lo = std::min<uint64_t>(nb, (uint64_t)t * chunk), hi = t == T - 1 ? nb : std::min<uint64_t>(nb, lo + chunk);
                if (hi > lo) {
                    uint64_t k = 0;
                    xp[(size_t)t].resize(1024);
                    xb[(size_t)t].resize(1024);
                    int r = tgsf_pack_bases(rb->bases.data() + lo, hi - lo, sl.packed + lo / 4, xp[(size_t)t].data(), xb[(size_t)t].data(), 1024, &k);
                    if (r == TGSF_ERR_CAPACITY) {
                        xp[(size_t)t].resize((size_t)k);
                        xb[(size_t)t].resize((size_t)k);
                        r = tgsf_pack_bases(rb->bases.data() + lo, hi - lo, sl.packed + lo / 4, xp[(size_t)t].data(), xb[(size_t)t].data(), k, &k);
                    }
                    xp[(size_t)t].resize((size_t)k);
                    xb[(size_t)t].resize((size_t)k);
                    for (uint64_t &q : xp[(size_t)t]) q += lo;
                    rcs[(size_t)t] = r;
                    if (has_qual) memcpy(sl.quals + lo, rb->quals.data() + lo, (size_t)(hi - lo));
                } else {
                    xp[(size_t)t].clear();
                    xb[(size_t)t].clear();
                }
            };
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) th.emplace_back(stage, t);
            stage(0);
            for (auto &x : th) x.join();
            sl.exc_pos.clear();
            sl.exc_byte.clear();
            for (int t = 0; t < T; ++t) {
                if (rcs[(size_t)t] != TGSF_OK) die_tgsf("tgsf_pack_bases");
                sl.exc_pos.insert(sl.exc_pos.end(), xp[(size_t)t].begin(), xp[(size_t)t].end());
                sl.exc_byte.insert(sl.exc_byte.end(), xb[(size_t)t].begin(), xb[(size_t)t].end());
            }
            ne = sl.exc_pos.size();
        }
        t_pack += T_loop.lap();
        t_copy += T_loop.lap();
        if (tgsf_submit_packed(ctx[(size_t)(cur % P.gpus)], sl.packed, has_qual ? sl.quals : nullptr, rb->offsets.data(), n,
                               sl.exc_pos.data(), sl.exc_byte.data(), ne) != TGSF_OK)
            die_tgsf("tgsf_submit_packed");
        t_submit += T_loop.lap();
        sl.rb = std::move(rb);
        inflight.push_back(cur);
        cur = (cur + 1) % slots;
    }
    T_loop.lap();
    while (!inflight.empty()) retire();
    t_retire += T_loop.lap();
    to_write.push(nullptr);
    writer.join();
    tlog("main loop: wait for parsed input", t_wait_in); tlog("main loop: reserve+pack", t_pack); tlog("main loop: quals memcpy", t_copy);
    tlog("main loop: submit", t_submit); tlog("main loop: collect/retire", t_retire); tlog("writer join", T_loop.lap());
    tlog("main pass total", T_ph.lap());
    if (reader.joinable()) {
        while (!input_done) { if (!next_parsed()) input_done = true; } // drain (only after an early error)
        reader.join();
    }
    if (clean_exit) for (PinSlot &sl : ring) { tgsf_host_free(sl.packed); tgsf_host_free(sl.quals); }
    if (out != stdout) fclose(out);

    // ---- counters: merge over GPUs (T.cpp:3208-3213) and the INFO lines (T.cpp:3214-3235) ----------
    tgsf_counter_layout L;
    tgsf_counter_layout_get(ctx[0], &L);
    std::vector<uint64_t> C(L.n_u64, 0);
    if (tgsf_allreduce(ctx.data(), (int)ctx.size()) != TGSF_OK) die_tgsf("tgsf_allreduce");
    if (tgsf_counters(ctx[0], C.data(), L.n_u64) != TGSF_OK) die_tgsf("tgsf_counters");
    const uint64_t *D = C.data() + L.drop_info;
    cerr << "INFO: " << rawNum << " reads with a total of " << rawBases << " bases were input." << endl;
    if (!P.OnlyQC) {
        cerr << "INFO: " << D[0] << " reads were discarded with " << D[1] << " bases due to low quality." << endl;
        cerr << "INFO: " << D[2] << " reads have adapter at 5', 3' and middle." << endl;
        cerr << "INFO: " << D[3] << " reads have adapter at 5' and middle." << endl;
        cerr << "INFO: " << D[4] << " reads have adapter at 3' and middle." << endl;
        cerr << "INFO: " << D[5] << " reads have adapter at 5' and 3' end." << endl;
        cerr << "INFO: " << D[6] << " reads only have adapter at middle." << endl;
        cerr << "INFO: " << D[7] << " reads only have adapter at 5' end." << endl;
        cerr << "INFO: " << D[8] << " reads only have adapter at 3' end." << endl;
        cerr << "INFO: " << D[9] << " reads didn't have any adapter." << endl;
        cerr << "INFO: " << D[10] << " bases were trimmed due to the adapter or base content bias." << endl;
        cerr << "INFO: " << D[11] << " reads were discarded with " << D[12] << " bases due to the short length." << endl;
        cerr << "INFO: " << D[13] << " reads were discarded with " << D[14] << " bases due to low quality after split." << endl;
        if (P.MinRepeat > 0)
            cerr << "INFO: " << D[15] << " reads were discarded with " << D[16] << " bases due to short repeat length." << endl;
        if (!P.ContamFile.empty())
            cerr << "INFO: " << contamNum << " reads were discarded with " << contamBases << " bases as contaminant." << endl;
        cerr << "INFO: " << cleanNum << " reads with a total of " << cleanBases << " bases after filtering." << endl;
        if (!P.Downsample && !P.OutFile.empty()) cerr << "INFO: Filtered reads were written to: " << P.OutFile << "." << endl;
    }
    // report columns (T.cpp:3146-3206)
    report::build_side(rawLens, rawBases, P.BCLen, has_qual, C.data(), L, false, 3, rawSide);
    if (!P.OnlyQC && !P.Downsample && cleanNum)
        report::build_side(cleanLens, cleanBases, P.BCLen, has_qual, C.data(), L, true, 3, cleanSide);
    if (const char *dump = getenv("TGSF_DUMP_COUNTERS")) { // raw counter block for report tooling / tests
        FILE *f = fopen(dump, "wb");
        if (f) {
            fwrite(&L, sizeof(L), 1, f);
            fwrite(C.data(), sizeof(uint64_t), C.size(), f);
            fclose(f);
        }
    }
    if (clean_exit) for (tgsf_ctx *c : ctx) tgsf_destroy(c);
    }

    // ---- downsampling: DownSampleTask (T.cpp:2164-2568) -------------------------------------------
    if (P.Downsample) {
        FILE *fout = stdout;
        if (!P.OutFile.empty()) {
            fout = fopen(P.OutFile.c_str(), "wb");
            if (!fout) { cerr << "Error: Failed to open file: " << P.OutFile << endl; return quit(1); }
        }
        // .gz: one member per record, compressed in chunks of ~64 MB by -t threads (same strategy rule as the main pass)
        std::vector<string> gz_pend;
        size_t gz_pend_bytes = 0;
        int gz_strategy = -1;
        auto deflate_one = [&](z_stream &zs, const string &r, string &dst) {
            deflateReset(&zs);
            const size_t at = dst.size(), bound = deflateBound(&zs, r.size()) + 32;
            dst.resize(at + bound);
            zs.next_in = (Bytef *)r.data();
            zs.avail_in = (uInt)r.size();
            zs.next_out = (Bytef *)&dst[at];
            zs.avail_out = (uInt)bound;
            deflate(&zs, Z_FINISH);
            dst.resize(at + zs.total_out);
        };
        auto flush_gz = [&]() {
            if (gz_pend.empty()) return;
            if (gz_strategy < 0) { // 16 evenly spaced records, both strategies
                uint64_t sd = 0, sr = 0;
                const size_t ns = std::min<size_t>(16, gz_pend.size());
                for (int which = 0; which < 2; ++which) {
                    z_stream zs;
                    memset(&zs, 0, sizeof(zs));
                    if (deflateInit2(&zs, P.compLevel, Z_DEFLATED, 15 + 16, 8, which ? Z_RLE : Z_DEFAULT_STRATEGY) != Z_OK) continue;
                    string tmp;
                    for (size_t a = 0; a < ns; ++a) { tmp.clear(); deflate_one(zs, gz_pend[a * gz_pend.size() / ns], tmp); (which ? sr : sd) += tmp.size(); }
                    deflateEnd(&zs);
                }
                gz_strategy = (!getenv("TGSF_GZ_DEFAULT_STRATEGY") && sr * 100 <= sd * 101) ? Z_RLE : Z_DEFAULT_STRATEGY;
            }
            const int K = std::max(1, std::min(P.n_thread, (int)std::thread::hardware_concurrency()));
            std::vector<string> bufs((size_t)K);
            auto work = [&](int k) {
                z_stream zs;
                memset(&zs, 0, sizeof(zs));
                if (deflateInit2(&zs, P.compLevel, Z_DEFLATED, 15 + 16, 8, gz_strategy) != Z_OK) return;
                for (size_t i = gz_pend.size() * (size_t)k / (size_t)K; i < gz_pend.size() * (size_t)(k + 1) / (size_t)K; ++i)
                    deflate_one(zs, gz_pend[i], bufs[(size_t)k]);
                deflateEnd(&zs);
            };
            std::vector<std::thread> th;
            for (int k = 1; k < K; ++k) th.emplace_back(work, k);
            work(0);
            for (auto &t : th) t.join();
            for (const string &d : bufs) fwrite(d.data(), 1, d.size(), fout);
            gz_pend.clear();
            gz_pend_bytes = 0;
        };
        auto emit = [&](const char *data, size_t n) {
            if (P.OUTGZ) {
                gz_pend.emplace_back(data, n);
                gz_pend_bytes += n;
                if (gz_pend_bytes >= (64u << 20)) flush_gz();
            } else {
                fwrite(data, 1, n, fout);
            }
        };
        Selection S;
        uint64_t downInNum = 0, downInBases = 0;
        const bool from_memory = P.Filter && mem_mode; // the filtered records never left host memory
        const string downInput = P.Filter ? tmpPath : P.InFile;
        if (!P.Filter) { // get_fastx_SeqLen, T.cpp:2256-2269
            FastxReader rd(P.InFile);
            string name, seq, qual;
            while (rd.read(name, seq, qual)) { recIdx.add(name, (int)seq.size()); downInNum++; downInBases += seq.size(); }
        }
        S = getenv("TGSF_SELECT_SORT") ? select_reads_sorted(recIdx, P, P.Filter ? 0 : downInBases)
                                       : select_reads(recIdx, P, P.Filter ? 0 : downInBases);
        // second pass (T.cpp:2346-2568): keep the selected names in file order and recompute the QC
        // tables of the kept reads on the GPU (a QC-only context: its "raw" tables are the report's
        // "after" column)
        tgsf_params qp;
        memset(&qp, 0, sizeof(qp));
        qp.bc_len = P.BCLen; qp.qtype = qType; qp.flags = TGSF_FLAG_ONLY_QC; qp.max_q = 255; qp.min_q = -1; qp.n_slots = 1;
        tgsf_ctx *qctx = nullptr;
        if (tgsf_create(0, &qp, &qctx) != TGSF_OK) die_tgsf("tgsf_create (downsample QC)");
        Batch qb;
        const bool dqual = from_memory ? P.Outfq == 1 : (file_type(downInput) == 1 || file_type(downInput) == 2);
        auto flush = [&]() {
            if (!qb.n()) return;
            if (!qb.pack()) die_tgsf("tgsf_pack_bases");
            if (tgsf_submit_packed(qctx, qb.packed, dqual ? qb.quals : nullptr, qb.offsets.data(), qb.n(), qb.exc_pos.data(),
                                   qb.exc_byte.data(), qb.n_exc) != TGSF_OK)
                die_tgsf("tgsf_submit_packed");
            if (tgsf_collect(qctx, nullptr, 0, nullptr, 0, nullptr) != TGSF_OK) die_tgsf("tgsf_collect");
            qb.clear();
        };
        std::vector<int> downLens;
        uint64_t downBases = 0;
        {
            string name, seq, qual, rec;
            auto take = [&]() -> bool { // one candidate record in name / seq / qual
                auto it = recIdx.pos.find(name);
                if (it == recIdx.pos.end() || !S.keep[it->second]) return true;
                rec.clear();
                if (P.Outfq == 1) { rec += '@'; rec += name; rec += '\n'; rec += seq; rec += "\n+\n"; rec += qual; rec += '\n'; }
                else { rec += '>'; rec += name; rec += '\n'; rec += seq; rec += '\n'; }
                emit(rec.data(), rec.size());
                if (!qb.add(name, seq, qual, dqual)) { cerr << "Error: out of pinned host memory" << endl; return false; }
                if (qb.used >= P.batch_bases) flush();
                return true;
            };
            if (from_memory) {
                for (const MemRec &r : mem_recs) {
                    name = mem_names[r.name];
                    seq.assign(mem_seq, r.off, r.len);
                    if (dqual) qual.assign(mem_qual, r.off, r.len);
                    if (!take()) return quit(1);
                }
            } else {
                FastxReader rd(downInput);
                while (rd.read(name, seq, qual))
                    if (!take()) return quit(1);
            }
            flush();
        }
        // the reference's table / length plots use the selection list (T.cpp:3244-3256)
        for (size_t i = 0; i < recIdx.names.size(); i++)
            if (S.keep[i]) { downLens.push_back(recIdx.lens[i]); downBases += (uint64_t)recIdx.lens[i]; }
        {
            tgsf_counter_layout QL;
            tgsf_counter_layout_get(qctx, &QL);
            std::vector<uint64_t> QC(QL.n_u64);
            if (tgsf_counters(qctx, QC.data(), QL.n_u64) != TGSF_OK) die_tgsf("tgsf_counters");
            report::build_side(downLens, downBases, P.BCLen, dqual, QC.data(), QL, false, 2, cleanSide);
        }
        qb.release();
        tgsf_destroy(qctx);
        if (!P.Filter) cerr << "INFO: " << downInNum << " reads with a total of " << downInBases << " bases were input." << endl;
        flush_gz();
        if (fout != stdout) fclose(fout);
        cerr << "INFO: " << S.downNum << " reads with a total of " << S.downBases << " bases after downsampling." << endl;
        if (!P.OutFile.empty()) cerr << "INFO: Downsampled reads were written to: " << P.OutFile << "." << endl;
        if (!tmpPath.empty()) remove(tmpPath.c_str());
    }

    tlog("counters/info/downsample", T_ph.lap());
    // ---- QC report (T.cpp:3285-3328) -----------------------------------------------------------------
    {
        auto prefix_of = [](const string &path) { // GetFilePreifx, T.cpp:824-837
            string ext = file_ext(path), prefix = path;
            if (ext == "gz") { prefix = path.substr(0, path.rfind('.')); ext = file_ext(prefix); }
            if (ext == "fq" || ext == "fastq" || ext == "fa" || ext == "fasta" || ext == "bam" || ext == "sam" || ext == "BAM" || ext == "SAM")
                prefix = prefix.substr(0, prefix.rfind('.'));
            return prefix;
        };
        string html = prefix_of(P.InFile) + ".html";
        if (!P.OutFile.empty() && !P.OnlyQC) html = prefix_of(P.OutFile) + ".html";
        string qcType = P.Infq == 0 ? "0" : "1";
        if (P.OnlyQC) qcType += "0";
        else if (!P.Filter && P.Downsample) qcType += "1";
        else qcType += "2";
        report::write_html(html, qcType, rawSide, cleanSide);
        cerr << "INFO: Quality control report was written to: " << html << "." << endl;
    }
    tlog("report", T_ph.lap());
    tlog("total", T_all.lap());
    if (clean_exit) return 0;
    // everything is written: leave without tearing down GBs of device, pinned and batch memory piece by piece
    std::cout.flush();
    cerr.flush();
    fflush(nullptr);
    _exit(0);
}
