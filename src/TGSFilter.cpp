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
#include <iostream>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
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
    string ContamReport;          // --contam-report: TSV of the contaminant pieces per --contam record
    bool Foldback = false;        // --foldback (extension): cut pieces at a fold-back junction, keep the longer arm
    bool Dust = false;            // --dust (extension): drop pieces dominated by low-complexity sequence
    int DustLevel = 7;            // --dust-level
    float DustFrac = 0.5f;        // --dust-frac
    bool Denovo = false;          // --adapter-denovo (extension): assemble an end's adapter when the library has none
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
                 "   --adapter-denovo  assemble an end's adapter from its sampled reads when no library adapter is found\n"
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
                 "   --contam-report <str> write the discarded reads and bases per --contam record to this TSV file\n"
                 " Fold-back screen:\n"
                 "   --foldback            cut reads that fold back onto their own reverse complement, keep the longer arm\n"
                 " Low-complexity screen:\n"
                 "   --dust                discard reads dominated by homopolymer or short tandem repeat (windowed DUST)\n"
                 "   --dust-level <int>    DUST score above which a 64-base window is masked, 1-30 [7]\n"
                 "   --dust-frac <float>   min fraction of a read's bases in masked windows to discard it [0.5]\n"
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
        else if (flag == "contamreport") { if (!need()) return 1; P->ContamReport = argv[i]; }
        else if (flag == "adapterdenovo") { P->Denovo = true; }
        else if (flag == "foldback") { P->Foldback = true; }
        else if (flag == "dust") { P->Dust = true; }
        else if (flag == "dustlevel") { if (!need()) return 1; P->DustLevel = atoi(argv[i]); }
        else if (flag == "dustfrac") { if (!need()) return 1; P->DustFrac = (float)atof(argv[i]); }
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
    if (!P->ContamReport.empty() && P->ContamFile.empty()) { cerr << "Error: --contam-report requires --contam" << endl; exit(-1); }
    if (!P->ContamFile.empty()) {
        if (P->OnlyQC || P->ONLYAD || !P->Filter) {
            cerr << "Error: --contam screens filtered reads and cannot be combined with --qc, -A or -F" << endl;
            exit(-1);
        }
        if (access(P->ContamFile.c_str(), R_OK) != 0) { cerr << "Error: Can't find this file for --contam " << P->ContamFile << endl; exit(-1); }
    }
    if (P->Foldback && (P->OnlyQC || P->ONLYAD || !P->Filter)) {
        cerr << "Error: --foldback screens filtered reads and cannot be combined with --qc, -A or -F" << endl;
        exit(-1);
    }
    if (P->DustLevel < 1 || P->DustLevel > 30) { cerr << "Error: --dust-level must be in [1,30]" << endl; exit(-1); }
    const long long dust_ppm = llround((double)P->DustFrac * 1e6); // as tgsf_set_dust computes it
    if (!(P->DustFrac == P->DustFrac) || dust_ppm < 1 || dust_ppm > 1000000) {
        cerr << "Error: --dust-frac must be in (0,1]" << endl;
        exit(-1);
    }
    if (P->Dust && (P->OnlyQC || P->ONLYAD || !P->Filter)) {
        cerr << "Error: --dust screens filtered reads and cannot be combined with --qc, -A or -F" << endl;
        exit(-1);
    }
    if (P->Denovo && (!P->AdapterFile.empty() || P->OnlyQC || !P->Filter)) {
        cerr << "Error: --adapter-denovo searches the sampled reads for adapters and cannot be combined with -a, --qc or -F"
             << endl;
        exit(-1);
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

// Contaminant FASTA (multi-line, plain or gzip): records back to back in seq, offs[i]..offs[i+1]; names[i] is record
// i's header up to the first space, tab or '\r' (empty for a sequence before the first '>').
bool load_contam_fasta(const string &path, std::vector<uint8_t> &seq, std::vector<uint64_t> &offs,
                       std::vector<string> &names) {
    gzFile f = gzopen(path.c_str(), "rb");
    if (!f) return false;
    gzbuffer(f, 1 << 20);
    seq.clear();
    offs.assign(1, 0);
    names.clear();
    std::vector<char> line(1 << 16);
    bool in_rec = false, at_bol = true, header = false, in_name = false;
    int n;
    while ((n = gzread(f, line.data(), (unsigned)line.size())) > 0) {
        for (int i = 0; i < n; ++i) {
            const char ch = line[(size_t)i];
            if (ch == '\n') { at_bol = true; header = false; continue; }
            if (at_bol && ch == '>') {
                if (in_rec) offs.push_back(seq.size());
                in_rec = true;
                header = true;
                in_name = true;
                names.emplace_back();
            } else if (header) {
                if (ch == ' ' || ch == '\t' || ch == '\r') in_name = false;
                else if (in_name) names.back().push_back(ch);
            } else if (ch != '\r' && ch != ' ' && ch != '\t') {
                if (!in_rec) names.emplace_back(); // a sequence before the first '>': a record without a name

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

// Leaving main while the reader / writer threads are joinable would call std::terminate; every exit after they start
// (errors, -A) therefore goes the way the normal end of main goes: flush, then _exit without tearing anything down.
[[noreturn]] void quit(int code) { std::cout.flush(); cerr.flush(); fflush(nullptr); _exit(code); }
[[noreturn]] void fail_open(const string &path) { cerr << "Error: Failed to open file: " << path << endl; quit(1); }

// Runs f(1) .. f(K-1) on new threads and f(0) on this one, and returns when all are done.
template <class F>
void run_parallel(int K, const F &f) {
    std::vector<std::thread> th;
    for (int k = 1; k < K; ++k) th.emplace_back(f, k);
    f(0);
    for (auto &t : th) t.join();
}

// Appends one gzip member holding rec to dst; zs is a gzip deflate stream (reset here).
void gz_member(z_stream &zs, const string &rec, string &dst) {
    deflateReset(&zs);
    const size_t at = dst.size(), bound = deflateBound(&zs, rec.size()) + 32;
    dst.resize(at + bound);
    zs.next_in = (Bytef *)rec.data();
    zs.avail_in = (uInt)rec.size();
    zs.next_out = (Bytef *)&dst[at];
    zs.avail_out = (uInt)bound;
    deflate(&zs, Z_FINISH);
    dst.resize(at + zs.total_out);
}

// Per-record members hold no cross-record matches, and on noisy long reads zlib's match search at the default
// strategy yields files no smaller than run-length + Huffman coding (Z_RLE), at 6-9x the time.  Z_RLE is used when
// it stays within 1 % of the size the requested level gives on the sample records (one thread per record).
int pick_gz_strategy(int level, const std::vector<string> &records) {
    const size_t ns = records.size();
    std::vector<uint64_t> sz_def(ns, 0), sz_rle(ns, 0);
    run_parallel((int)ns, [level, &records, &sz_def, &sz_rle](int a) {
        for (int which = 0; which < 2; ++which) {
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (deflateInit2(&zs, level, Z_DEFLATED, 15 + 16, 8, which ? Z_RLE : Z_DEFAULT_STRATEGY) != Z_OK) continue;
            string o;
            gz_member(zs, records[(size_t)a], o);
            (which ? sz_rle : sz_def)[(size_t)a] = o.size();
            deflateEnd(&zs);
        }
    });
    uint64_t sd = 0, sr = 0;
    for (size_t a = 0; a < ns; ++a) { sd += sz_def[a]; sr += sz_rle[a]; }
    return sr * 100 <= sd * 101 ? Z_RLE : Z_DEFAULT_STRATEGY;
}

// One FASTQ (qual: len bytes) or FASTA (qual unused) record.
void append_record(string &dst, bool fastq, const string &name, const char *seq, const char *qual, size_t len) {
    if (fastq) {
        dst += '@'; dst += name; dst += '\n'; dst.append(seq, len); dst += "\n+\n"; dst.append(qual, len); dst += '\n';
    } else {
        dst += '>'; dst += name; dst += '\n'; dst.append(seq, len); dst += '\n';
    }
}

void write_all(int fd, const char *data, size_t n) {
    size_t done = 0;
    while (done < n) {
        const ssize_t w = write(fd, data + done, n - done);
        if (w <= 0) { cerr << "Error: write failed" << endl; exit(-1); }
        done += (size_t)w;
    }
}

// MemAvailable of /proc/meminfo in MB, -1 when it cannot be read.
int64_t mem_available_mb() {
    int64_t mb = -1;
    if (FILE *mi = fopen("/proc/meminfo", "r")) {
        char line[256];
        unsigned long long kb;
        while (fgets(line, sizeof(line), mi))
            if (sscanf(line, "MemAvailable: %llu kB", &kb) == 1) mb = (int64_t)(kb >> 10);
        fclose(mi);
    }
    return mb;
}

int out_threads(const Params &P) { return std::max(1, std::min(P.n_thread, (int)std::thread::hardware_concurrency())); }

// ---- I/O types (GetFileType, T.cpp:839-857) -------------------------------------------------------------
bool check_io_types(Params &P) {
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
        return false;
    }
    if (P.Infq == 0 && P.Outfq == 1) { cerr << "Error: Fasta format input file can't output fastq format file" << endl; return false; }
#ifndef TGSF_HAVE_HTSLIB
    if (P.Infq == 2) { // CRAM is recognised by its content, as hts_open does; without htslib it cannot be decoded: fail loudly
        char magic[4] = {0, 0, 0, 0};
        if (FILE *f = fopen(P.InFile.c_str(), "rb")) {
            if (fread(magic, 1, 4, f) != 4) magic[0] = 0;
            fclose(f);
        }
        if (memcmp(magic, "CRAM", 4) == 0) {
            cerr << "Error: CRAM input needs a build with htslib (make -C src HTS_DIR=<htslib prefix>); "
                    "convert with `samtools fastq` or to BAM" << endl;
            return false;
        }
    }
#endif
    return true;
}

// ---- streamed input ---------------------------------------------------------------------------------
// The parsed batches in file order: plain files go through the parallel chunk parser, gzip and SAM/BAM through one
// reader thread.  The batches the pre-pass keeps (pageable) are handed to the main pass first; when they outgrow
// TGSF_PREPASS_BUFFER_MB (default: a quarter of MemAvailable, at most 24 GB) they are dropped and the main pass
// reads the input again from its beginning (two-pass mode, like the reference: T.cpp:949-982 then 1845-1916).
class Input {
public:
    ingest::BatchPool pool; // recycled batches: the writer returns them here
    Input(const Params &P, bool has_qual, bool sambam)
        : path_(P.InFile), has_qual_(has_qual), sambam_(sambam),
          batch_bases_(getenv("TGSF_BATCH_MB") ? (uint64_t)atoll(getenv("TGSF_BATCH_MB")) << 20 : P.batch_bases) {
        double mb = 24576.0;
        if (const int64_t avail = mem_available_mb(); avail >= 0) mb = std::min(mb, (double)avail / 4.0);
        if (getenv("TGSF_PREPASS_BUFFER_MB")) mb = atof(getenv("TGSF_PREPASS_BUFFER_MB"));
        budget_ = (uint64_t)(mb * 1048576.0);
    }
    // Starts the readers at the beginning of the input; false if it cannot be opened.
    bool start() {
        done_ = false;
        if (!sambam_ && !ingest::ParallelReader::is_gzip(path_)) {
            const int hw = (int)std::thread::hardware_concurrency();
            const int nthr = getenv("TGSF_PARSE_THREADS") ? atoi(getenv("TGSF_PARSE_THREADS")) : std::max(1, std::min(8, hw - 2));
            preader_.reset(new ingest::ParallelReader(path_, has_qual_, 2 * batch_bases_, nthr, &pool));
            return preader_->ok();
        }
        stop_.store(false);
        reader_ = std::thread(ingest::reader_main, path_, has_qual_, batch_bases_, &parsed_, &pool, &stop_, sambam_);
        return true;
    }
    std::unique_ptr<ingest::RawBatch> read() {
        if (done_) return nullptr;
        std::unique_ptr<ingest::RawBatch> rb = preader_ ? preader_->pop() : parsed_.pop();
        if (!rb) done_ = true;
        return rb;
    }
    // Pre-pass: keeps a sampled batch for the main pass, or drops it (and all kept ones) past the budget.
    void keep(std::unique_ptr<ingest::RawBatch> rb) {
        if (two_pass_) { pool.put(std::move(rb)); return; }
        kept_bytes_ += rb->bases.size() + rb->quals.size();
        kept_.push_back(std::move(rb));
        if (kept_bytes_ > budget_) {
            two_pass_ = true;
            for (auto &b : kept_) pool.put(std::move(b));
            kept_.clear();
        }
    }
    // End of the pre-pass: in two-pass mode the input starts again from its beginning.
    bool rewind() {
        if (!two_pass_) return true;
        preader_.reset();
        if (reader_.joinable()) {
            stop_.store(true);
            while (read()) {}
            reader_.join();
        }
        return start();
    }
    // Main pass: the kept batches, then the rest of the input.
    std::unique_ptr<ingest::RawBatch> next() {
        if (kept_.empty()) return read();
        std::unique_ptr<ingest::RawBatch> rb = std::move(kept_.front());
        kept_.pop_front();
        return rb;
    }
    void close() { if (reader_.joinable()) reader_.join(); } // after the main pass read the input to its end

private:
    const string path_;
    const bool has_qual_, sambam_;
    const uint64_t batch_bases_;
    uint64_t budget_ = 0, kept_bytes_ = 0;
    ingest::Queue<std::unique_ptr<ingest::RawBatch>> parsed_{4};
    std::unique_ptr<ingest::ParallelReader> preader_;
    std::thread reader_;
    std::atomic<bool> stop_{false};
    std::deque<std::unique_ptr<ingest::RawBatch>> kept_;
    bool done_ = false, two_pass_ = false;
};

// ---- pre-pass: read_fastx (T.cpp:949-982) + Get_qType (T.cpp:1042-1077) -----------------------------
struct Sample {
    const int checkLen, minLen, maxSeq;
    int seqNum = 0, minQ = 255, maxQ = 0;
    std::vector<uint8_t> e5, e3; // per sampled read: checkLen bases of the 5' end / of the reverse complement of the 3' end
    explicit Sample(const Params &P)
        : checkLen(std::max(std::max(P.EndLen, P.BCLen), 100)), minLen(std::max(P.MinLen, 2 * checkLen)),
          maxSeq(std::max(P.ADNum, P.BCNum)) {}
    void quals(const char *q) {
        for (int j = 0; j < checkLen; j++) {
            if (minQ > q[j]) minQ = q[j];
            if (maxQ < q[j]) maxQ = q[j];
        }
    }
};

// Starts the streamed input and samples the read ends from its first batches as they arrive (one pass over the
// input, Input::keep); the CUDA context is created meanwhile.
std::unique_ptr<Input> sample_stream(const Params &P, bool has_qual, bool sambam, Sample &S) {
    { gzFile probe = gzopen(P.InFile.c_str(), "rb"); if (!probe) fail_open(P.InFile); gzclose(probe); }
    std::unique_ptr<Input> in(new Input(P, has_qual, sambam));
    if (!in->start()) fail_open(P.InFile);
    // CUDA context creation (0.4-0.7 s warm, 1.3 s+ for the first process on a box) overlaps the parsing
    { Timer tw; void *warm = nullptr; if (tgsf_host_alloc(&warm, 1 << 20) == TGSF_OK) tgsf_host_free(warm); tlog("  CUDA context warm-up", tw.lap()); }
    std::unique_ptr<ingest::RawBatch> rb;
    while (S.seqNum < S.maxSeq && (rb = in->read())) {
        for (uint32_t i = 0; i < rb->n() && S.seqNum < S.maxSeq; i++) {
            const uint64_t s0 = rb->offsets[i];
            const int L = (int)(rb->offsets[i + 1] - s0);
            if (L < S.minLen) continue;
            S.seqNum++;
            S.e5.insert(S.e5.end(), rb->bases.begin() + s0, rb->bases.begin() + s0 + S.checkLen);
            for (int j = 0; j < S.checkLen; j++) S.e3.push_back((uint8_t)g_comp[rb->bases[s0 + L - 1 - j]]);
            if (has_qual) S.quals((const char *)rb->quals.data() + s0);
        }
        in->keep(std::move(rb));
    }
    if (!in->rewind()) fail_open(P.InFile);
    return in;
}

// -F: only the sample is needed here; DownSampleTask reads the file itself.
void sample_file(const Params &P, bool has_qual, Sample &S) {
    FastxReader rd(P.InFile);
    if (!rd.ok()) fail_open(P.InFile);
    string name, seq, qual;
    while (rd.read(name, seq, qual)) {
        if ((int)seq.size() < S.minLen) continue;
        if (S.seqNum >= S.maxSeq) break;
        S.seqNum++;
        if (has_qual) S.quals(qual.data());
    }
}

// Phred offset of the qualities (0 without) and the -q default.
int resolve_quality(Params &P, bool has_qual, Sample &S) {
    if (!has_qual) return 0;
    int qType;
    if (S.minQ >= 33 && S.minQ <= 78 && S.maxQ >= 33 && S.maxQ <= 127) qType = 33;
    else if (S.minQ >= 64 && S.minQ <= 108 && S.maxQ >= 64 && S.maxQ <= 127) qType = 64;
    else if (S.minQ < 55) qType = 33;
    else qType = 64;
    cerr << "INFO: base quality scoring: Phred" << qType << endl;
    S.minQ -= qType;
    S.maxQ -= qType;
    if (P.MinQ >= 0) {
        if (P.MinQ >= S.maxQ) {
            cerr << "Warning: max base quality score was: " << S.maxQ << endl;
            cerr << "INFO: Please reset -q parameter." << endl;
            exit(-1);
        }
    } else {
        if (S.maxQ > 10 && P.readType == "clr") P.MinQ = 10;
        else if (S.maxQ > 20 && P.readType == "hifi") P.MinQ = 20;
        else if (S.maxQ > 10 && P.readType == "ont") P.MinQ = 10;
        else P.MinQ = 0;
    }
    return qType;
}

// ---- de novo adapter assembly (--adapter-denovo, an extension; tgsfilter_b200/prepass.py mirrors it) ----------------
// The constants are chosen for synthetic reads with one planted adapter per end; they have not been checked on real kits.
constexpr int kDenovoK = 12;          // k-mer size of the counts
constexpr int kDenovoSupport = 100;   // a seed occurs in at least 1/100 of the rows ...
constexpr uint32_t kDenovoMinSeed = 20; // ... and at least 20 times
constexpr uint64_t kDenovoEnrich = 4; // outer-half count >= 4 x (inner-half count + 1): adapters sit at the outer end
constexpr int kDenovoMaxRun = 4;      // longest run of one base in a seed
constexpr size_t kDenovoMinLen = 20, kDenovoMaxLen = 100; // candidate length bounds

// Seed and extension over the outer / inner k-mer counts O, I of n rows (tgsf_end_kmer_counts with the split at
// (row_len - k + 1) / 2).  The seed is the k-mer with the largest O that has >= 3 distinct bases, no run longer than
// kDenovoMaxRun, O >= max(20, ceil(n/100)) and O >= 4 (I + 1); ties go to the smallest code.  The path grows to the
// right, then to the left, by the neighbour with the largest O + I (A, C, G, T order breaks ties) until that total is
// below half the seed's, the k-mer is already in the path, or the path has kDenovoMaxLen bases.  Returns "" when no
// seed qualifies or the path is shorter than kDenovoMinLen.
string assemble_adapter(const std::vector<uint32_t> &O, const std::vector<uint32_t> &I, uint32_t n) {
    const int k = kDenovoK;
    const uint32_t mask = (1u << (2 * k)) - 1;
    const uint32_t support = std::max(kDenovoMinSeed, (n + kDenovoSupport - 1) / kDenovoSupport);
    auto base = [&](uint32_t code, int i) { return (int)((code >> (2 * (k - 1 - i))) & 3); };
    auto complex_enough = [&](uint32_t code) {
        int seen = 0, run = 1, longest = 1;
        for (int i = 0; i < k; i++) {
            seen |= 1 << base(code, i);
            if (i) { run = base(code, i) == base(code, i - 1) ? run + 1 : 1; longest = std::max(longest, run); }
        }
        return __builtin_popcount(seen) >= 3 && longest <= kDenovoMaxRun;
    };
    int64_t seed = -1;
    for (uint32_t x = 0; x <= mask; x++)
        if (O[x] >= support && O[x] >= kDenovoEnrich * ((uint64_t)I[x] + 1) && (seed < 0 || O[x] > O[(size_t)seed]) &&
            complex_enough(x))
            seed = x;
    if (seed < 0) return "";
    auto total = [&](uint32_t x) { return (uint64_t)O[x] + I[x]; };
    const uint64_t cut = total((uint32_t)seed);
    std::deque<int> path;
    for (int i = 0; i < k; i++) path.push_back(base((uint32_t)seed, i));
    std::unordered_set<uint32_t> in_path{(uint32_t)seed};
    for (int right = 1; right >= 0; right--) {
        while (path.size() < kDenovoMaxLen) {
            uint32_t end = 0; // the last (right) or first (left) k - 1 bases
            for (int i = 0; i < k - 1; i++) end = (end << 2) | (uint32_t)path[right ? path.size() - (k - 1) + i : i];
            int best = 0;
            uint32_t y = 0;
            for (int b = 0; b < 4; b++) {
                const uint32_t z = right ? ((end << 2) | b) & mask : ((uint32_t)b << (2 * (k - 1))) | end;
                if (b == 0 || total(z) > total(y)) { best = b; y = z; }
            }
            if (2 * total(y) < cut || !in_path.insert(y).second) break;
            if (right) path.push_back(best);
            else path.push_front(best);
        }
    }
    if (path.size() < kDenovoMinLen) return "";
    string s;
    for (int v : path) s += "ACGT"[v];
    return s;
}

// --adapter-denovo for each end without a library pick (empty a5 / a3): assembles a candidate from that end's sampled
// rows and scores the candidates with the library search.  A candidate is accepted as the end's adapter when its mean
// depth (as `pick` computes it) reaches 2 x minSim and n / 100: the first rule alone accepts about two matching rows.
void denovo_adapters(const Sample &S, float minSim, string &a5, float &d5, string &a3, float &d3) {
    const uint32_t n = (uint32_t)S.seqNum, len = (uint32_t)S.checkLen;
    const bool run[2] = {a5.empty(), a3.empty()};
    const std::vector<uint8_t> *rows[2] = {&S.e5, &S.e3};
    string cand[2];
    if (n && (run[0] || run[1])) {
        std::vector<uint32_t> O((size_t)1 << (2 * kDenovoK)), I(O.size());
        const uint32_t split = (len - kDenovoK + 1) / 2; // checkLen >= 100 > k
        for (int e = 0; e < 2; e++) {
            if (!run[e]) continue;
            if (tgsf_end_kmer_counts(0, rows[e]->data(), n, len, kDenovoK, split, O.data(), I.data()) != TGSF_OK)
                die_tgsf("tgsf_end_kmer_counts");
            cand[e] = assemble_adapter(O, I, n);
        }
    }
    std::vector<const uint8_t *> lib_seq;
    std::vector<int32_t> lib_len;
    int slot[2] = {-1, -1};
    for (int e = 0; e < 2; e++)
        if (!cand[e].empty()) {
            slot[e] = (int)lib_seq.size();
            lib_seq.push_back((const uint8_t *)cand[e].data());
            lib_len.push_back((int32_t)cand[e].size());
        }
    float dep[2] = {0, 0};
    if (!lib_seq.empty()) {
        std::vector<int32_t> bn((size_t)len * 4 * 2);
        std::vector<int64_t> m5(lib_seq.size()), m3(lib_seq.size());
        if (tgsf_prepass(0, S.e5.data(), S.e3.data(), n, len, lib_seq.data(), lib_len.data(), (int32_t)lib_seq.size(),
                         minSim, bn.data(), bn.data() + (size_t)len * 4, m5.data(), m3.data()) != TGSF_OK)
            die_tgsf("tgsf_prepass");
        const std::vector<int64_t> *maps[2] = {&m5, &m3};
        for (int e = 0; e < 2; e++) {
            if (slot[e] < 0) continue;
            const float meanDep = static_cast<float>((int)(*maps[e])[(size_t)slot[e]]) / cand[e].size();
            if (meanDep >= 2 * minSim && meanDep >= n / 100.0f) dep[e] = meanDep;
            else cand[e].clear();
        }
    }
    const char *name[2] = {"5'", "3'"};
    for (int e = 0; e < 2; e++)
        if (run[e]) {
            cerr << "INFO: de novo " << name[e] << " adapter: " << cand[e] << endl;
            cerr << "INFO: mean depth of de novo " << name[e] << " adapter: " << dep[e] << endl;
        }
    if (run[0]) { a5 = cand[0]; d5 = dep[0]; }
    if (run[1]) { a3 = cand[1]; d3 = dep[1]; }
}

// End trims from the base content of the sample and the adapter set (the global `adapters`, T.cpp:1324): from -a, or
// searched for in the sample.  -A ends the run here.
std::vector<string> resolve_adapters(Params &P, bool has_qual, const Sample &S) {
    std::vector<string> adapters; // the order is irrelevant for the results ...
    // ... but Get_adapters prints the set in std::unordered_set iteration order (T.cpp:2937-2940): the same container with the
    // same insertions (same libstdc++ hash and rehash policy) reproduces that order for the `input adapter` lines
    std::unordered_set<string> adapter_set;
    auto add_adapter = [&](const string &a) { if (adapter_set.insert(a).second) adapters.push_back(a); };
    const int checkLen = S.checkLen, seqNum = S.seqNum;
    std::vector<int32_t> bn5((size_t)checkLen * 4), bn3((size_t)checkLen * 4);
    std::vector<int64_t> m5(TGSF_LIB_ADAPTERS, 0), m3(TGSF_LIB_ADAPTERS, 0);
    std::vector<const uint8_t *> lib_seq;
    std::vector<int32_t> lib_len;
    for (const char *a : kLib) { lib_seq.push_back((const uint8_t *)a); lib_len.push_back((int32_t)strlen(a)); }
    const bool search = P.AdapterFile.empty();
    const uint8_t dummy = 0;
    if (tgsf_prepass(0, seqNum ? S.e5.data() : &dummy, seqNum ? S.e3.data() : &dummy, (uint32_t)seqNum, (uint32_t)checkLen,
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
        return adapters;
    }
    // tail of adapterSearch (T.cpp:1178-1208) + selection (T.cpp:3081-3125)
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
    if (P.Denovo) denovo_adapters(S, minSim, a5, d5, a3, d3);
    if (d5 > 5 * d3) { a3 = ""; d3 = 0; }
    else if (d3 > 5 * d5) { a5 = ""; d5 = 0; }
    cerr << "INFO: 5' adapter: " << a5 << endl;
    cerr << "INFO: 3' adapter: " << a3 << endl;
    cerr << "INFO: mean depth of 5' adapter: " << d5 << endl;
    cerr << "INFO: mean depth of 3' adapter: " << d3 << endl;
    if (P.ONLYAD) quit(0);
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
    return adapters;
}

// ---- contexts: one per GPU, with the contaminant set (--contam), the fold-back screen (--foldback) and the DUST screen (--dust) on each
// --contam-report: the set is installed with labels and record_kmers receives the keys per record (shared keys last).
std::vector<tgsf_ctx *> create_contexts(const Params &P, int qType, const std::vector<string> &adapters, bool gz_gpu,
                                        std::vector<uint8_t> &contam_seq, const std::vector<uint64_t> &contam_offs,
                                        std::vector<uint64_t> &record_kmers) {
    tgsf_params tp;
    memset(&tp, 0, sizeof(tp));
    tp.min_len = P.MinLen; tp.max_len = P.MaxLen; tp.min_q = P.MinQ; tp.max_q = P.MaxQ;
    tp.bc_len = P.BCLen; tp.head_trim = P.HeadTrim; tp.tail_trim = P.TailTrim;
    tp.end_len = P.EndLen; tp.end_match_len = P.EndMatchLen; tp.mid_match_len = P.MidMatchLen;
    tp.extra_len = P.ExtraLen; tp.end_sim = P.EndSim; tp.mid_sim = P.MidSim;
    tp.kmer = P.Kmer; tp.min_repeat = P.MinRepeat; tp.qtype = qType;
    tp.flags = (P.Filter ? TGSF_FLAG_FILTER : 0) | (P.OnlyQC ? TGSF_FLAG_ONLY_QC : 0) | (P.discard ? TGSF_FLAG_DISCARD_MID : 0);
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
        quit(1);
    }
    for (int g = 0; g < P.gpus; g++)
        if (tgsf_create(g % n_dev, &tp, &ctx[(size_t)g]) != TGSF_OK) die_tgsf("tgsf_create");
    if (!P.ContamFile.empty()) {
        uint64_t n_kmers = 0;
        const uint32_t n_seqs = (uint32_t)(contam_offs.size() - 1);
        if (!P.ContamReport.empty()) record_kmers.assign((size_t)n_seqs + 1, 0);
        for (int g = 0; g < P.gpus; g++) {
            if (P.ContamReport.empty()) {
                if (tgsf_set_contaminants(ctx[(size_t)g], contam_seq.data(), contam_offs.data(), n_seqs, P.ContamK,
                                          P.ContamFrac, &n_kmers) != TGSF_OK)
                    die_tgsf("tgsf_set_contaminants");
            } else if (tgsf_set_contaminants_labelled(ctx[(size_t)g], contam_seq.data(), contam_offs.data(), n_seqs,
                                                      P.ContamK, P.ContamFrac, &n_kmers, record_kmers.data()) != TGSF_OK) {
                die_tgsf("tgsf_set_contaminants_labelled");
            }
        }
        cerr << "INFO: " << n_kmers << " distinct " << P.ContamK << "-mers loaded from " << P.ContamFile << "." << endl;
        std::vector<uint8_t>().swap(contam_seq);
    }
    if (P.Foldback)
        for (int g = 0; g < P.gpus; g++)
            if (tgsf_set_foldback(ctx[(size_t)g], 1) != TGSF_OK) die_tgsf("tgsf_set_foldback");
    if (P.Dust)
        for (int g = 0; g < P.gpus; g++)
            if (tgsf_set_dust(ctx[(size_t)g], P.DustLevel, P.DustFrac) != TGSF_OK) die_tgsf("tgsf_set_dust");
    return ctx;
}

// ---- writer (T.cpp:2011-2053) -----------------------------------------------------------------------
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
};

// Filter + downsample: the filtered records are kept for the downsampling pass, in host memory (sequence / quality bytes
// back to back + one entry per record); only past TGSF_DOWNSAMPLE_BUFFER_MB (default: a quarter of MemAvailable, at most
// 64 GB) they are spilled to the reference's uncompressed tmp file (T.cpp:3129-3137) and the run continues there.
struct Filtered {
    ingest::RawBatch mem; // qualities for FASTQ output only
    bool in_memory = false;
    string tmp_path;
    RecIndex idx; // every filtered record's name and length
};

// The writer thread numbers the emitted pieces of each retired batch, then
//  * plain output: gathers name/bases/qualities straight out of the batch, no formatting copy; a regular file is
//    written by several threads at precomputed offsets;
//  * gzip output: one member per record like DeflateCompress (T.cpp:786-812), the records of a batch spread over -t
//    threads, written in order;
//  * downsampling: keeps the records (Filtered).
// The counters, cleanLens and `kept` belong to the writer thread until join().
class Writer {
public:
    PinnedPool gz_pool;
    uint64_t cleanNum = 0, cleanBases = 0;
    uint64_t contamNum = 0, contamBases = 0; // pieces discarded by the contaminant screen (--contam)
    uint64_t dustNum = 0, dustBases = 0;     // pieces discarded by the DUST screen (--dust)
    std::vector<int> cleanLens;              // T.cpp:1794
    Filtered kept;
    // Opens the output (stdout, -o, or with downsampling the buffer / tmp file) and starts the thread.
    Writer(const Params &P, ingest::BatchPool &batches)
        : P_(P), fq_(P.Outfq == 1), gz_(P.OUTGZ && !P.Downsample), threads_(out_threads(P)), batches_(batches) {
        if (P.Downsample) {
            uint64_t mb = std::min<uint64_t>((uint64_t)std::max<int64_t>(mem_available_mb(), 0) / 4, 65536);
            if (const char *e = getenv("TGSF_DOWNSAMPLE_BUFFER_MB")) mb = strtoull(e, nullptr, 10);
            mem_budget_ = mb << 20;
            kept.in_memory = mem_budget_ > 0;
            if (!kept.in_memory) open_tmp();
        } else if (!P.OnlyQC && !P.OutFile.empty()) {
            out_ = fopen(P.OutFile.c_str(), "w+b"); // read-write: the plain writer maps the file
            if (!out_) fail_open(P.OutFile);
        }
        fflush(out_);
        out_fd_ = fileno(out_);
        struct stat st;
        // positioned parallel writes only into a file this process created (stdout may be in append mode)
        out_regular_ = out_ != stdout && fstat(out_fd_, &st) == 0 && S_ISREG(st.st_mode);
        th_ = std::thread(&Writer::run, this);
    }
    void push(std::unique_ptr<WriteJob> job) { jobs_.push(std::move(job)); }
    // After the last batch: waits until everything is written, then closes the output.
    void join() {
        jobs_.push(nullptr);
        th_.join();
        if (out_ != stdout) fclose(out_);
    }

private:
    struct Emit { uint32_t read, start, len; int pass; uint32_t piece; };
    void run() {
        while (std::unique_ptr<WriteJob> job = jobs_.pop()) {
            const ingest::RawBatch &b = *job->rb;
            number(*job);
            if (P_.Downsample) keep(b);
            else if (!emits_.empty() && gz_) write_gz(*job);
            else if (!emits_.empty()) write_plain(b);
            batches_.put(std::move(job->rb));
            gz_pool.put(job->gz_blob, job->gz_cap);
        }
    }
    // T.cpp:1976-2059: pass 1 keeps the raw name, later pieces of a read get ":N" before the first blank
    void number(const WriteJob &job) {
        const ingest::RawBatch &b = *job.rb;
        emits_.clear();
        renamed_.clear();
        uint32_t last = UINT32_MAX;
        int pass = 1;
        for (size_t pi = 0; pi < job.pieces.size(); ++pi) {
            const tgsf_piece &p = job.pieces[pi];
            if ((uint32_t)p.read != last) { last = (uint32_t)p.read; pass = 1; }
            if (p.status == TGSF_PIECE_CONTAM) { contamNum++; contamBases += (uint64_t)p.len; }
            if (p.status == TGSF_PIECE_LOWCOMPLEX) { dustNum++; dustBases += (uint64_t)p.len; }
            if (p.status != TGSF_PIECE_EMIT) continue;
            emits_.push_back(Emit{last, (uint32_t)p.start, (uint32_t)p.len, pass, (uint32_t)pi});
            pass++;
            cleanNum++;
            cleanBases += (uint64_t)p.len;
            cleanLens.push_back(p.len);
        }
        renamed_.reserve(emits_.size()); // nm_ points into it
        nm_.resize(emits_.size());
        for (size_t i = 0; i < emits_.size(); ++i) {
            if (emits_[i].pass >= 2) { renamed_.push_back(new_seq_name(b.names[emits_[i].read], emits_[i].pass)); nm_[i] = &renamed_.back(); }
            else nm_[i] = &b.names[emits_[i].read];
        }
    }
    void format(const ingest::RawBatch &b, size_t i, string &dst) const {
        const Emit &e = emits_[i];
        const uint64_t at = b.offsets[e.read] + e.start;
        append_record(dst, fq_, *nm_[i], (const char *)b.bases.data() + at, fq_ ? (const char *)b.quals.data() + at : nullptr, e.len);
    }
    void open_tmp() { // uncompressed tmp file like T.cpp:3129-3137
        kept.tmp_path = P_.InFile + ".tmp." + std::to_string((long)getpid()) + (P_.Outfq == 0 ? ".fa" : ".fq");
        out_ = fopen(kept.tmp_path.c_str(), "wb");
        if (!out_) fail_open(kept.tmp_path);
    }
    void keep(const ingest::RawBatch &b) {
        if (!kept.in_memory) {
            for (size_t i = 0; i < emits_.size(); ++i) {
                format(b, i, obuf_);
                kept.idx.add(*nm_[i], (int)emits_[i].len);
                if (obuf_.size() >= (8u << 20)) { fwrite(obuf_.data(), 1, obuf_.size(), out_); obuf_.clear(); }
            }
            if (!obuf_.empty()) { fwrite(obuf_.data(), 1, obuf_.size(), out_); obuf_.clear(); }
            return;
        }
        ingest::RawBatch &m = kept.mem;
        for (size_t i = 0; i < emits_.size(); ++i) {
            const Emit &e = emits_[i];
            const uint64_t at = b.offsets[e.read] + e.start;
            m.names.push_back(*nm_[i]);
            m.bases.insert(m.bases.end(), b.bases.data() + at, b.bases.data() + at + e.len);
            if (fq_) m.quals.insert(m.quals.end(), b.quals.data() + at, b.quals.data() + at + e.len);
            m.offsets.push_back(m.bases.size());
            kept.idx.add(*nm_[i], (int)e.len);
        }
        if (m.bases.size() + m.quals.size() > mem_budget_) { // over budget: spill what is buffered, continue on the file
            open_tmp();
            string rec;
            for (uint32_t r = 0; r < m.n(); ++r) {
                rec.clear();
                append_record(rec, fq_, m.names[r], (const char *)m.bases.data() + m.offsets[r],
                              fq_ ? (const char *)m.quals.data() + m.offsets[r] : nullptr, m.offsets[r + 1] - m.offsets[r]);
                fwrite(rec.data(), 1, rec.size(), out_);
            }
            kept.in_memory = false;
            m = ingest::RawBatch();
        }
    }
    // Splits the records into K contiguous ranges of about equal payload.
    void split(int K) {
        cut_.assign((size_t)K + 1, emits_.size());
        bytes_before_.assign((size_t)K + 1, 0);
        uint64_t total = 0;
        for (const Emit &e : emits_) total += e.len;
        uint64_t acc = 0, raw = 0;
        int k = 0;
        cut_[0] = 0;
        for (size_t i = 0; i < emits_.size(); ++i) {
            while (k + 1 < K && acc >= total * (uint64_t)(k + 1) / (uint64_t)K) { cut_[(size_t)++k] = i; bytes_before_[(size_t)k] = raw; }
            acc += emits_[i].len;
            const uint64_t nl = nm_[i]->size();
            raw += fq_ ? 1 + nl + 1 + emits_[i].len + 3 + emits_[i].len + 1 : 1 + nl + 1 + emits_[i].len + 1;
        }
        while (k + 1 < K) { cut_[(size_t)++k] = emits_.size(); bytes_before_[(size_t)k] = raw; }
        bytes_before_[(size_t)K] = raw;
    }
    // gzip: one member per record, spread over -t threads, from the GPU's deflate blocks when the batch has them, else by
    // host zlib (TGSF_GZ_HOST=1, or a batch whose blocks could not be collected)
    void write_gz(const WriteJob &job) {
        const int K = threads_;
        split(K);
        bufs_.resize((size_t)K);
        if (!job.gz_ok && (gz_batches_++ & 15) == 0) { // zlib strategy: every 16th batch, 16 evenly spaced records of it
            const size_t ns = std::min<size_t>(16, emits_.size());
            std::vector<string> sample(ns);
            for (size_t a = 0; a < ns; ++a) format(*job.rb, a * emits_.size() / ns, sample[a]);
            gz_strategy_ = pick_gz_strategy(P_.compLevel, sample);
        }
        run_parallel(K, [this, &job](int k) {
            bufs_[(size_t)k].clear();
            if (job.gz_ok) wrap_gz_blocks(job, k);
            else deflate_range(*job.rb, k);
        });
        for (int k = 0; k < K; ++k) write_all(out_fd_, bufs_[(size_t)k].data(), bufs_[(size_t)k].size());
    }
    // members around the GPU's deflate blocks: gzip header | stored block with the header line | blocks | CRC-32, ISIZE
    // (include/tgsf.h, tgsf_collect_gz)
    void wrap_gz_blocks(const WriteJob &job, int k) {
        const ingest::RawBatch &b = *job.rb;
        string &dst = bufs_[(size_t)k];
        static const unsigned char kHdr[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff};
        for (size_t i = cut_[(size_t)k]; i < cut_[(size_t)k + 1]; ++i) {
            const Emit &e = emits_[i];
            const tgsf_gz_span &sp = job.gz_spans[e.piece];
            const Bytef *sq = (const Bytef *)b.bases.data() + b.offsets[e.read] + e.start;
            const size_t hl = nm_[i]->size() + 2;
            string head;
            head += fq_ ? '@' : '>';
            head += *nm_[i];
            head += '\n';
            uLong crc = crc32(0L, (const Bytef *)head.data(), (uInt)hl);
            crc = crc32(crc, sq, (uInt)e.len);
            uint64_t isize = hl + e.len + 1;
            if (fq_) {
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
            dst.append((const char *)job.gz_blob + sp.offset, sp.bytes);
            const uint32_t tr[2] = {(uint32_t)crc, (uint32_t)isize};
            dst.append((const char *)tr, 8);
        }
    }
    void deflate_range(const ingest::RawBatch &b, int k) {
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (deflateInit2(&zs, P_.compLevel, Z_DEFLATED, 15 + 16, 8, gz_strategy_) != Z_OK) return;
        string r;
        for (size_t i = cut_[(size_t)k]; i < cut_[(size_t)k + 1]; ++i) {
            r.clear();
            format(b, i, r);
            gz_member(zs, r, bufs_[(size_t)k]);
        }
        deflateEnd(&zs);
    }
    void write_plain(const ingest::RawBatch &b) {
        const int K = out_regular_ ? std::min(threads_, 8) : 1;
        split(K);
        static const char kAt = '@', kGt = '>', kNl = '\n';
        static const char kPlus[] = "\n+\n";
        // A regular file takes its inode lock for every buffered write, so positioned writes from
        // several threads serialise.  Preferred path: reserve the batch's byte range (fallocate, so a
        // full disk is an error here and not a SIGBUS later), map it and let the threads copy their
        // records into the mapping; the pwritev path stays as the fallback (pipes, odd filesystems).
        bool mapped = false;
        const uint64_t nbytes = bytes_before_[(size_t)K];
        if (out_regular_ && out_mmap_ && nbytes) {
            const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE);
            const uint64_t map_off = out_off_ & ~(page - 1), delta = out_off_ - map_off;
            if (fallocate(out_fd_, 0, (off_t)out_off_, (off_t)nbytes) == 0) {
                void *m = mmap(nullptr, (size_t)(nbytes + delta), PROT_READ | PROT_WRITE, MAP_SHARED, out_fd_, (off_t)map_off);
                if (m != MAP_FAILED) {
                    run_parallel(K, [this, &b, m, delta](int k) {
                        char *dst = (char *)m + delta + bytes_before_[(size_t)k];
                        for (size_t i = cut_[(size_t)k]; i < cut_[(size_t)k + 1]; ++i) {
                            const Emit &e = emits_[i];
                            *dst++ = fq_ ? '@' : '>';
                            memcpy(dst, nm_[i]->data(), nm_[i]->size()); dst += nm_[i]->size();
                            *dst++ = '\n';
                            memcpy(dst, b.bases.data() + b.offsets[e.read] + e.start, e.len); dst += e.len;
                            if (fq_) {
                                memcpy(dst, kPlus, 3); dst += 3;
                                memcpy(dst, b.quals.data() + b.offsets[e.read] + e.start, e.len); dst += e.len;
                            }
                            *dst++ = '\n';
                        }
                    });
                    munmap(m, (size_t)(nbytes + delta));
                    mapped = true;
                }
            } else {
                out_mmap_ = false; // filesystem without fallocate: keep to pwritev
            }
        }
        if (!mapped) {
            run_parallel(K, [this, &b](int k) {
                std::vector<struct iovec> iov;
                iov.reserve(1024);
                uint64_t off = out_off_ + bytes_before_[(size_t)k];
                auto flush = [&]() {
                    size_t first = 0;
                    while (first < iov.size()) {
                        const int cnt = (int)std::min<size_t>(iov.size() - first, 1024);
                        ssize_t w = out_regular_ ? pwritev(out_fd_, iov.data() + first, cnt, (off_t)off) : writev(out_fd_, iov.data() + first, cnt);
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
                for (size_t i = cut_[(size_t)k]; i < cut_[(size_t)k + 1]; ++i) {
                    const Emit &e = emits_[i];
                    const uint8_t *sq = b.bases.data() + b.offsets[e.read] + e.start;
                    if (iov.size() + 7 > 1024) flush();
                    add(fq_ ? &kAt : &kGt, 1);
                    add(nm_[i]->data(), nm_[i]->size());
                    add(&kNl, 1);
                    add(sq, e.len);
                    if (fq_) {
                        add(kPlus, 3);
                        add(b.quals.data() + b.offsets[e.read] + e.start, e.len);
                    }
                    add(&kNl, 1);
                }
                flush();
            });
        }
        out_off_ += nbytes;
    }
    const Params &P_;
    const bool fq_, gz_; // FASTQ records; gzip output (T.cpp:2022)
    const int threads_;  // -t
    ingest::BatchPool &batches_;
    ingest::Queue<std::unique_ptr<WriteJob>> jobs_{4};
    FILE *out_ = stdout;
    int out_fd_ = -1;
    bool out_regular_ = false, out_mmap_ = true;
    uint64_t out_off_ = 0, mem_budget_ = 0; // out_off_: bytes written so far to a regular file
    int gz_strategy_ = Z_DEFAULT_STRATEGY;
    unsigned gz_batches_ = 0;
    std::vector<Emit> emits_;
    std::vector<string> renamed_;          // names with a :N suffix, alive until the batch is written
    std::vector<const string *> nm_;       // name of each emitted piece
    std::vector<size_t> cut_;              // thread k writes records [cut_[k], cut_[k + 1])
    std::vector<uint64_t> bytes_before_;   // ... starting this many bytes into the batch's output
    std::vector<string> bufs_;             // gzip: thread k's members
    string obuf_;
    std::thread th_;
};

// ---- main pass: parse -> pinned ring -> tgsf_submit_packed -> tgsf_collect -> writer ------------------------
// pinned staging slot: what crosses PCIe (2-bit packed bases, Phred bytes); 2 slots per GPU
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
    // pack the bases (2 bits) and copy the qualities into the slot on T threads: the ranges are multiples of 32
    // bases, their exception lists are concatenated with the range offset added
    void stage(const ingest::RawBatch &b, bool has_qual, int T) {
        const uint64_t nb = b.bases.size();
        if (!reserve((size_t)nb + 64)) { cerr << "Error: out of pinned host memory" << endl; quit(1); }
        const uint64_t chunk = ((nb / (uint64_t)T + 31) / 32) * 32;
        std::vector<std::vector<uint64_t>> xp((size_t)T);
        std::vector<std::vector<uint8_t>> xb((size_t)T);
        std::vector<int> rcs((size_t)T, TGSF_OK);
        run_parallel(T, [this, &b, has_qual, T, nb, chunk, &xp, &xb, &rcs](int t) {
            const uint64_t lo = std::min<uint64_t>(nb, (uint64_t)t * chunk), hi = t == T - 1 ? nb : std::min<uint64_t>(nb, lo + chunk);
            if (hi <= lo) return;
            uint64_t k = 0;
            xp[(size_t)t].resize(1024);
            xb[(size_t)t].resize(1024);
            int r = tgsf_pack_bases(b.bases.data() + lo, hi - lo, packed + lo / 4, xp[(size_t)t].data(), xb[(size_t)t].data(), 1024, &k);
            if (r == TGSF_ERR_CAPACITY) {
                xp[(size_t)t].resize((size_t)k);
                xb[(size_t)t].resize((size_t)k);
                r = tgsf_pack_bases(b.bases.data() + lo, hi - lo, packed + lo / 4, xp[(size_t)t].data(), xb[(size_t)t].data(), k, &k);
            }
            xp[(size_t)t].resize((size_t)k);
            xb[(size_t)t].resize((size_t)k);
            for (uint64_t &q : xp[(size_t)t]) q += lo;
            rcs[(size_t)t] = r;
            if (has_qual) memcpy(quals + lo, b.quals.data() + lo, (size_t)(hi - lo));
        });
        exc_pos.clear();
        exc_byte.clear();
        for (int t = 0; t < T; ++t) {
            if (rcs[(size_t)t] != TGSF_OK) die_tgsf("tgsf_pack_bases");
            exc_pos.insert(exc_pos.end(), xp[(size_t)t].begin(), xp[(size_t)t].end());
            exc_byte.insert(exc_byte.end(), xb[(size_t)t].begin(), xb[(size_t)t].end());
        }
    }
    void submit(tgsf_ctx *c, const ingest::RawBatch &b, bool has_qual) {
        if (tgsf_submit_packed(c, packed, has_qual ? quals : nullptr, b.offsets.data(), b.n(), exc_pos.data(), exc_byte.data(),
                               exc_pos.size()) != TGSF_OK)
            die_tgsf("tgsf_submit_packed");
    }
};

// Collects the results of the slot's batch into a write job; with gz_pool (GPU deflate blocks) the blocks first.
std::unique_ptr<WriteJob> collect(tgsf_ctx *c, PinSlot &sl, PinnedPool *gz_pool, double blob_per_base,
                                  std::vector<tgsf_read_result> &rr) {
    const uint32_t n = sl.rb->n();
    std::unique_ptr<WriteJob> job(new WriteJob());
    rr.resize(n);
    job->pieces.resize((size_t)n + 4096);
    uint32_t np = 0;
    if (gz_pool) { // before tgsf_collect, which retires the batch; a second try with the sizes the first one reported
        uint64_t nb = 0;
        uint32_t ns = 0;
        size_t want = (size_t)(sl.rb->bases.size() * blob_per_base + (1u << 20)), spans = (size_t)n + 4096;
        int grc = TGSF_ERR_CAPACITY;
        for (int attempt = 0; attempt < 2 && grc == TGSF_ERR_CAPACITY; ++attempt) {
            if (attempt) { gz_pool->put(job->gz_blob, job->gz_cap); want = (size_t)nb + 16; spans = (size_t)ns + 16; }
            std::tie(job->gz_blob, job->gz_cap) = gz_pool->get(want);
            job->gz_spans.resize(spans);
            grc = job->gz_blob ? tgsf_collect_gz(c, job->gz_blob, job->gz_cap, &nb, job->gz_spans.data(), (uint32_t)spans, &ns) : TGSF_ERR_NOMEM;
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
    return job;
}

struct MainPass {
    uint64_t rawNum = 0, rawBases = 0;
    std::vector<int> rawLens; // T.cpp:1794
    double t_wait_in = 0, t_pack = 0, t_copy = 0, t_submit = 0, t_retire = 0;
};

// Feeds every batch of the input to the GPUs (two in flight per GPU, dealt round-robin) and hands the results, in
// input order, to the writer.
MainPass feed(Input &in, const std::vector<tgsf_ctx *> &ctx, Writer &w, bool has_qual, bool gz_gpu, double blob_per_base,
              bool clean_exit) {
    MainPass M;
    const int gpus = (int)ctx.size(), slots = 2 * gpus;
    std::vector<PinSlot> ring((size_t)slots);
    std::deque<int> inflight; // ring indices in submission order; slot i runs on GPU (i % gpus)
    std::vector<tgsf_read_result> rr;
    auto retire = [&]() {
        const int bi = inflight.front();
        inflight.pop_front();
        w.push(collect(ctx[(size_t)(bi % gpus)], ring[(size_t)bi], gz_gpu ? &w.gz_pool : nullptr, blob_per_base, rr));
    };
    const int stage_threads = getenv("TGSF_STAGE_THREADS") ? std::max(1, atoi(getenv("TGSF_STAGE_THREADS"))) : 4;
    const int stage_shift = getenv("TGSF_STAGE_MIN_SHIFT") ? std::max(6, atoi(getenv("TGSF_STAGE_MIN_SHIFT"))) : 22; // >= 4 Mbases per thread
    int cur = 0;
    Timer T_loop;
    while (true) {
        T_loop.lap();
        std::unique_ptr<ingest::RawBatch> rb = in.next();
        if (!rb) break;
        M.t_wait_in += T_loop.lap();
        const uint32_t n = rb->n();
        const uint64_t nb = rb->bases.size();
        M.rawNum += n;
        M.rawBases += nb;
        for (uint32_t i = 0; i < n; i++) M.rawLens.push_back((int)(rb->offsets[i + 1] - rb->offsets[i]));
        T_loop.lap();
        if ((int)inflight.size() == slots) retire(); // ring slot `cur` is the oldest one in flight
        M.t_retire += T_loop.lap();
        PinSlot &sl = ring[(size_t)cur];
        sl.stage(*rb, has_qual, (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)stage_threads, nb >> stage_shift)));
        M.t_pack += T_loop.lap();
        M.t_copy += T_loop.lap();
        sl.submit(ctx[(size_t)(cur % gpus)], *rb, has_qual);
        M.t_submit += T_loop.lap();
        sl.rb = std::move(rb);
        inflight.push_back(cur);
        cur = (cur + 1) % slots;
    }
    T_loop.lap();
    while (!inflight.empty()) retire();
    M.t_retire += T_loop.lap();
    if (clean_exit) for (PinSlot &sl : ring) { tgsf_host_free(sl.packed); tgsf_host_free(sl.quals); }
    return M;
}

// ---- counters: merge over GPUs (T.cpp:3208-3213), INFO lines (T.cpp:3214-3235), report columns (T.cpp:3146-3206) ----
void report_filter(const Params &P, std::vector<tgsf_ctx *> &ctx, const MainPass &M, const Writer &w, bool has_qual,
                   report::Side &rawSide, report::Side &cleanSide) {
    tgsf_counter_layout L;
    tgsf_counter_layout_get(ctx[0], &L);
    std::vector<uint64_t> C(L.n_u64, 0);
    if (tgsf_allreduce(ctx.data(), (int)ctx.size()) != TGSF_OK) die_tgsf("tgsf_allreduce");
    if (tgsf_counters(ctx[0], C.data(), L.n_u64) != TGSF_OK) die_tgsf("tgsf_counters");
    const uint64_t *D = C.data() + L.drop_info;
    cerr << "INFO: " << M.rawNum << " reads with a total of " << M.rawBases << " bases were input." << endl;
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
            cerr << "INFO: " << w.contamNum << " reads were discarded with " << w.contamBases << " bases as contaminant." << endl;
        if (P.Dust)
            cerr << "INFO: " << w.dustNum << " reads were discarded with " << w.dustBases << " bases as low complexity." << endl;
        if (P.Foldback) {
            uint64_t F[4] = {0, 0, 0, 0};
            for (tgsf_ctx *c : ctx) {
                uint64_t f[4];
                if (tgsf_foldback_stats(c, f) != TGSF_OK) die_tgsf("tgsf_foldback_stats");
                for (int i = 0; i < 4; i++) F[i] += f[i];
            }
            cerr << "INFO: " << F[0] << " reads were cut at a fold-back junction, removing " << F[1] << " bases." << endl;
            cerr << "INFO: " << F[2] << " reads were discarded with " << F[3] << " bases as too short after a fold-back cut."
                 << endl;
        }
        cerr << "INFO: " << w.cleanNum << " reads with a total of " << w.cleanBases << " bases after filtering." << endl;
        if (!P.Downsample && !P.OutFile.empty()) cerr << "INFO: Filtered reads were written to: " << P.OutFile << "." << endl;
    }
    report::build_side(M.rawLens, M.rawBases, P.BCLen, has_qual, C.data(), L, false, 3, rawSide);
    if (!P.OnlyQC && !P.Downsample && w.cleanNum)
        report::build_side(w.cleanLens, w.cleanBases, P.BCLen, has_qual, C.data(), L, true, 3, cleanSide);
    if (const char *dump = getenv("TGSF_DUMP_COUNTERS")) { // raw counter block for report tooling / tests
        if (FILE *f = fopen(dump, "wb")) {
            fwrite(&L, sizeof(L), 1, f);
            fwrite(C.data(), sizeof(uint64_t), C.size(), f);
            fclose(f);
        }
    }
}

// ---- --contam-report: the contaminant pieces per record, summed over the contexts --------------------------------------
void write_contam_report(FILE *f, const string &path, std::vector<tgsf_ctx *> &ctx, const std::vector<string> &names,
                         const std::vector<uint64_t> &offs, const std::vector<uint64_t> &record_kmers) {
    const uint32_t rows = (uint32_t)names.size() + 1;
    std::vector<uint64_t> reads(rows, 0), bases(rows, 0), r(rows), b(rows);
    for (tgsf_ctx *c : ctx) {
        if (tgsf_contam_record_stats(c, r.data(), b.data(), rows) != TGSF_OK) die_tgsf("tgsf_contam_record_stats");
        for (uint32_t i = 0; i < rows; ++i) { reads[i] += r[i]; bases[i] += b[i]; }
    }
    string out = "#record\tname\tlength\tunique_kmers\treads\tbases\n";
    for (uint32_t i = 0; i + 1 < rows; ++i)
        out += std::to_string(i) + "\t" + names[i] + "\t" + std::to_string(offs[i + 1] - offs[i]) + "\t" +
               std::to_string(record_kmers[i]) + "\t" + std::to_string(reads[i]) + "\t" + std::to_string(bases[i]) + "\n";
    out += "*\tshared\t.\t" + std::to_string(record_kmers[rows - 1]) + "\t" + std::to_string(reads[rows - 1]) + "\t" +
           std::to_string(bases[rows - 1]) + "\n";
    if (fwrite(out.data(), 1, out.size(), f) != out.size() || fclose(f) != 0) {
        cerr << "Error: Failed to write --contam-report " << path << endl;
        quit(1);
    }
}

// ---- downsampling: DownSampleTask (T.cpp:2164-2568) ----------------------------------------------------
// Selects the reads, writes them in file order from the filtered records (-F: the input) and recomputes the QC tables
// of the kept reads on the GPU (a QC-only context: its "raw" tables are the report's "after" column).
void downsample(const Params &P, int qType, Filtered kept, report::Side &cleanSide) {
    FILE *fout = stdout;
    if (!P.OutFile.empty()) {
        fout = fopen(P.OutFile.c_str(), "wb");
        if (!fout) fail_open(P.OutFile);
    }
    // .gz: one member per record, compressed in chunks of ~64 MB by -t threads; the zlib strategy is picked once, on 16
    // evenly spaced records of the first chunk
    std::vector<string> gz_pend;
    size_t gz_pend_bytes = 0;
    int gz_strategy = -1;
    auto flush_gz = [&]() {
        if (gz_pend.empty()) return;
        if (gz_strategy < 0) {
            const size_t ns = std::min<size_t>(16, gz_pend.size());
            std::vector<string> sample(ns);
            for (size_t a = 0; a < ns; ++a) sample[a] = gz_pend[a * gz_pend.size() / ns];
            gz_strategy = pick_gz_strategy(P.compLevel, sample);
        }
        const int K = out_threads(P);
        std::vector<string> bufs((size_t)K);
        run_parallel(K, [&P, K, &gz_pend, gz_strategy, &bufs](int k) {
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (deflateInit2(&zs, P.compLevel, Z_DEFLATED, 15 + 16, 8, gz_strategy) != Z_OK) return;
            for (size_t i = gz_pend.size() * (size_t)k / (size_t)K; i < gz_pend.size() * (size_t)(k + 1) / (size_t)K; ++i)
                gz_member(zs, gz_pend[i], bufs[(size_t)k]);
            deflateEnd(&zs);
        });
        for (const string &d : bufs) fwrite(d.data(), 1, d.size(), fout);
        gz_pend.clear();
        gz_pend_bytes = 0;
    };
    RecIndex &recIdx = kept.idx;
    uint64_t downInNum = 0, downInBases = 0;
    const bool from_memory = P.Filter && kept.in_memory; // the filtered records never left host memory
    const string downInput = P.Filter ? kept.tmp_path : P.InFile;
    if (!P.Filter) { // get_fastx_SeqLen, T.cpp:2256-2269
        FastxReader rd(P.InFile);
        string name, seq, qual;
        while (rd.read(name, seq, qual)) { recIdx.add(name, (int)seq.size()); downInNum++; downInBases += seq.size(); }
    }
    const Selection S = getenv("TGSF_SELECT_SORT") ? select_reads_sorted(recIdx, P, P.Filter ? 0 : downInBases)
                                                   : select_reads(recIdx, P, P.Filter ? 0 : downInBases);
    // second pass (T.cpp:2346-2568): keep the selected names in file order
    tgsf_params qp;
    memset(&qp, 0, sizeof(qp));
    qp.bc_len = P.BCLen; qp.qtype = qType; qp.flags = TGSF_FLAG_ONLY_QC; qp.max_q = 255; qp.min_q = -1; qp.n_slots = 1;
    tgsf_ctx *qctx = nullptr;
    if (tgsf_create(0, &qp, &qctx) != TGSF_OK) die_tgsf("tgsf_create (downsample QC)");
    const bool dqual = from_memory ? P.Outfq == 1 : (file_type(downInput) == 1 || file_type(downInput) == 2);
    ingest::RawBatch qb;
    PinSlot qs;
    auto flush = [&]() {
        if (!qb.n()) return;
        qs.stage(qb, dqual, 1);
        qs.submit(qctx, qb, dqual);
        if (tgsf_collect(qctx, nullptr, 0, nullptr, 0, nullptr) != TGSF_OK) die_tgsf("tgsf_collect");
        qb.bases.clear(); qb.quals.clear(); qb.offsets.assign(1, 0); qb.names.clear();
    };
    string name, seq, qual, rec;
    auto take = [&]() { // one candidate record in name / seq / qual
        auto it = recIdx.pos.find(name);
        if (it == recIdx.pos.end() || !S.keep[it->second]) return;
        rec.clear();
        append_record(rec, P.Outfq == 1, name, seq.data(), qual.data(), seq.size());
        if (!P.OUTGZ) fwrite(rec.data(), 1, rec.size(), fout);
        else { gz_pend.push_back(rec); gz_pend_bytes += rec.size(); if (gz_pend_bytes >= (64u << 20)) flush_gz(); }
        qb.names.push_back(name);
        qb.bases.insert(qb.bases.end(), seq.begin(), seq.end());
        if (dqual) qb.quals.insert(qb.quals.end(), qual.begin(), qual.begin() + (long)seq.size());
        qb.offsets.push_back(qb.bases.size());
        if (qb.bases.size() >= P.batch_bases) flush();
    };
    if (from_memory) {
        const ingest::RawBatch &m = kept.mem;
        for (uint32_t r = 0; r < m.n(); ++r) {
            name = m.names[r];
            seq.assign(m.bases.begin() + (long)m.offsets[r], m.bases.begin() + (long)m.offsets[r + 1]);
            if (dqual) qual.assign(m.quals.begin() + (long)m.offsets[r], m.quals.begin() + (long)m.offsets[r + 1]);
            take();
        }
    } else {
        FastxReader rd(downInput);
        while (rd.read(name, seq, qual)) take();
    }
    flush();
    // the reference's table / length plots use the selection list (T.cpp:3244-3256)
    std::vector<int> downLens;
    uint64_t downBases = 0;
    for (size_t i = 0; i < recIdx.names.size(); i++)
        if (S.keep[i]) { downLens.push_back(recIdx.lens[i]); downBases += (uint64_t)recIdx.lens[i]; }
    tgsf_counter_layout QL;
    tgsf_counter_layout_get(qctx, &QL);
    std::vector<uint64_t> QC(QL.n_u64);
    if (tgsf_counters(qctx, QC.data(), QL.n_u64) != TGSF_OK) die_tgsf("tgsf_counters");
    report::build_side(downLens, downBases, P.BCLen, dqual, QC.data(), QL, false, 2, cleanSide);
    tgsf_host_free(qs.packed); tgsf_host_free(qs.quals);
    tgsf_destroy(qctx);
    if (!P.Filter) cerr << "INFO: " << downInNum << " reads with a total of " << downInBases << " bases were input." << endl;
    flush_gz();
    if (fout != stdout) fclose(fout);
    cerr << "INFO: " << S.downNum << " reads with a total of " << S.downBases << " bases after downsampling." << endl;
    if (!P.OutFile.empty()) cerr << "INFO: Downsampled reads were written to: " << P.OutFile << "." << endl;
    if (!kept.tmp_path.empty()) remove(kept.tmp_path.c_str());
}

// ---- QC report (T.cpp:3285-3328) -------------------------------------------------------------------------
string file_prefix(const string &path) { // GetFilePreifx, T.cpp:824-837
    string ext = file_ext(path), prefix = path;
    if (ext == "gz") { prefix = path.substr(0, path.rfind('.')); ext = file_ext(prefix); }
    if (ext == "fq" || ext == "fastq" || ext == "fa" || ext == "fasta" || ext == "bam" || ext == "sam" || ext == "BAM" || ext == "SAM")
        prefix = prefix.substr(0, prefix.rfind('.'));
    return prefix;
}

void write_report(const Params &P, const report::Side &rawSide, const report::Side &cleanSide) {
    string html = file_prefix(P.InFile) + ".html";
    if (!P.OutFile.empty() && !P.OnlyQC) html = file_prefix(P.OutFile) + ".html";
    string qcType = P.Infq == 0 ? "0" : "1";
    if (P.OnlyQC) qcType += "0";
    else if (!P.Filter && P.Downsample) qcType += "1";
    else qcType += "2";
    report::write_html(html, qcType, rawSide, cleanSide);
    cerr << "INFO: Quality control report was written to: " << html << "." << endl;
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
    std::vector<uint64_t> contam_offs, record_kmers;
    std::vector<string> contam_names;
    FILE *contam_report = nullptr;
    if (!P.ContamFile.empty()) {
        if (!load_contam_fasta(P.ContamFile, contam_seq, contam_offs, contam_names)) { cerr << "Error: Failed to read --contam " << P.ContamFile << endl; return 1; }
        if (contam_offs.size() < 2 || contam_seq.empty()) { cerr << "Error: no sequence in --contam " << P.ContamFile << endl; return 1; }
        if (!P.ContamReport.empty() && !(contam_report = fopen(P.ContamReport.c_str(), "w"))) {
            cerr << "Error: Failed to open file for --contam-report " << P.ContamReport << endl;
            return 1;
        }
    }
    for (int i = 0; i < 256; i++) g_comp[i] = 'N';
    const char *pairs[] = {"AT", "GC", "CG", "TA", "at", "gc", "cg", "ta", "MK", "RY", "WW", "SS", "YR", "KM",
                           "mk", "ry", "ww", "ss", "yr", "km"};
    for (const char *p : pairs) g_comp[(unsigned char)p[0]] = p[1];
    if (!check_io_types(P)) return 1;
    const bool has_qual = P.Infq == 1 || P.Infq == 2; // BAM/SAM records carry qualities (read_bam, T.cpp:1872-1916)

    Sample S(P);
    std::unique_ptr<Input> in; // from here on, leave through quit()
    if (P.Filter || P.OnlyQC) in = sample_stream(P, has_qual, P.Infq == 2, S);
    else sample_file(P, has_qual, S);
    tlog("prepass sampling (incl. CUDA context)", T_ph.lap());
    const int qType = resolve_quality(P, has_qual, S);
    std::vector<string> adapters;
    if (P.Filter) adapters = resolve_adapters(P, has_qual, S);

    report::Side rawSide, cleanSide;
    std::unique_ptr<Writer> w;
    if (in) {
        tlog("gpu prepass + resolve", T_ph.lap());
        // .gz output: the deflate blocks of every record are produced on the GPU (TGSF_GZ_HOST=1: host zlib instead)
        const bool gz_gpu = P.OUTGZ && !P.Downsample && !P.OnlyQC && !getenv("TGSF_GZ_HOST");
        std::vector<tgsf_ctx *> ctx = create_contexts(P, qType, adapters, gz_gpu, contam_seq, contam_offs, record_kmers);
        tlog("tgsf_create", T_ph.lap());
        w.reset(new Writer(P, in->pool));
        const MainPass M = feed(*in, ctx, *w, has_qual, gz_gpu, has_qual && P.Outfq == 1 ? 1.0 : 0.5, clean_exit);
        Timer T_join;
        w->join();
        tlog("main loop: wait for parsed input", M.t_wait_in); tlog("main loop: reserve+pack", M.t_pack); tlog("main loop: quals memcpy", M.t_copy);
        tlog("main loop: submit", M.t_submit); tlog("main loop: collect/retire", M.t_retire); tlog("writer join", T_join.lap());
        tlog("main pass total", T_ph.lap());
        in->close();
        report_filter(P, ctx, M, *w, has_qual, rawSide, cleanSide);
        if (contam_report) write_contam_report(contam_report, P.ContamReport, ctx, contam_names, contam_offs, record_kmers);
        if (clean_exit) for (tgsf_ctx *c : ctx) tgsf_destroy(c);
    }
    if (P.Downsample) downsample(P, qType, w ? std::move(w->kept) : Filtered(), cleanSide);
    tlog("counters/info/downsample", T_ph.lap());
    write_report(P, rawSide, cleanSide);
    tlog("report", T_ph.lap());
    tlog("total", T_all.lap());
    if (clean_exit) return 0;
    quit(0); // everything is written: leave without tearing down GBs of device, pinned and batch memory piece by piece
}
