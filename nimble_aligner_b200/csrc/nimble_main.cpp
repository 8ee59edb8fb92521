// nimble_main.cpp — `nimble` CLI with the arguments of /root/reference/src/bin/cli.yml:5-50 and the dispatch of
// src/bin/main.rs:12-162, on top of the C ABI (include/nimble_b200.h).
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

static void die(const std::string& m) { fprintf(stderr, "%s\n", m.c_str()); exit(101); }  // a Rust panic exits 101

// SIZE = decimal bytes with an optional K, M or G suffix (powers of 1024); 0 when malformed, zero or too large
static uint64_t parse_size(const std::string& t) {
  size_t n = 0; uint64_t v = 0;
  while (n < t.size() && t[n] >= '0' && t[n] <= '9') { if (v > (UINT64_MAX - 9) / 10) return 0; v = v * 10 + (uint64_t)(t[n] - '0'); n++; }
  if (n == 0) return 0;
  int shift = 0;
  if (n + 1 == t.size()) { const char c = t[n]; shift = c == 'K' ? 10 : c == 'M' ? 20 : c == 'G' ? 30 : -1; if (shift < 0) return 0; }
  else if (n != t.size()) return 0;
  if (v > (UINT64_MAX >> shift)) return 0;
  return v << shift;
}

int main(int argc, char** argv) {
  std::vector<std::string> refs, outs, ins, mats; bool have_mats = false, no_rows = false, any_order = false; uint64_t device_budget = 0; bool have_budget = false; std::string cores = "1", strand = "unstranded", trim, devs = getenv("NB_DEVICES") ? getenv("NB_DEVICES") : "0"; bool have_trim = false, force_paired = false;
  std::vector<std::string>* cur = nullptr;
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    auto val = [&](const char* name) -> std::string { if (i + 1 >= argc) die(std::string("error: The argument '") + name + "' requires a value but none was supplied"); return argv[++i]; };
    if (a == "-r" || a == "--reference") { cur = &refs; continue; }
    if (a == "-o" || a == "--output") { cur = &outs; continue; }
    if (a == "-i" || a == "--input") { cur = &ins; continue; }
    if (a == "-c" || a == "--cores") { cores = val("--cores"); cur = nullptr; continue; }
    if (a == "-f" || a == "--strand_filter") { strand = val("--strand_filter"); cur = nullptr; continue; }
    if (a == "-t" || a == "--trim") { trim = val("--trim"); have_trim = true; cur = nullptr; continue; }
    if (a == "-p" || a == "--force_bam_paired") { force_paired = true; cur = nullptr; continue; }
    if (a == "-d" || a == "--devices") { devs = val("--devices"); cur = nullptr; continue; }   // not in cli.yml: which GPUs to use, "0,1,..." (default: NB_DEVICES or 0)
    if (a == "--index-cache") { const std::string dir = val("--index-cache"); setenv("NB_INDEX_CACHE", dir.c_str(), 1); cur = nullptr; continue; }   // not in cli.yml: keep each library's index in <dir>/<key>.nbix (default: NB_INDEX_CACHE, else rebuilt per run like the reference)
    if (a == "--cell-matrix") { cur = &mats; have_mats = true; continue; }   // not in cli.yml: BAM mode, one directory per -r for a cell x feature matrix (10x v3 layout)
    if (a == "--no-rows") { no_rows = true; cur = nullptr; continue; }          // not in cli.yml: BAM mode, no TSV.gz rows (with --cell-matrix, without -o)
    if (a == "--any-order") { any_order = true; cur = nullptr; continue; }      // not in cli.yml: BAM mode, scopes from the tags of a BAM in any record order (-o rows, or --cell-matrix --no-rows)
    if (a == "--device-budget") { const std::string v = val("--device-budget"); device_budget = parse_size(v); have_budget = true; if (!device_budget) die("error: --device-budget needs a positive number of bytes with an optional K, M or G suffix, not '" + v + "'"); cur = nullptr; continue; }   // not in cli.yml: with --any-order, the device memory it may allocate
    if (a == "-h" || a == "--help") {
      printf("nimble 0.8.0 (B200)\nUSAGE: nimble [FLAGS] [OPTIONS] --input <input>... --output <output>... --reference <reference>...\n"
             "  -d, --devices <list>          GPUs to use, \"0,1,...\" (default: NB_DEVICES, else 0)\n"
             "      --index-cache <dir>       keep each library's index in <dir> (default: NB_INDEX_CACHE)\n"
             "      --cell-matrix <dir>...    BAM input: also write a cell x feature matrix per reference library into <dir>\n"
             "                                (matrix.mtx.gz UMIs, reads.mtx.gz reads, features.tsv.gz, barcodes.tsv.gz)\n"
             "      --no-rows                 BAM input with --cell-matrix: skip the TSV.gz rows (no --output)\n"
             "      --any-order               BAM input in any record order (e.g. position-sorted), no sort by UB needed (no -p):\n"
             "                                with --output, the TSV.gz rows in any order (assembled on the GPU); with\n"
             "                                --cell-matrix --no-rows, the matrices; (UMI, CB) scopes are formed on the GPU\n"
             "      --device-budget <size>    with --any-order: device memory it may allocate, bytes or with a K/M/G suffix\n"
             "                                (powers of 1024); records that do not fit take more passes over the file\n");
      return 0;
    }
    if (a == "-V" || a == "--version") { printf("nimble 0.8.0\n"); return 0; }
    if (!cur) die("error: Found argument '" + a + "' which wasn't expected, or isn't valid in this context");
    cur->push_back(a);
  }
  if (have_budget && !any_order) die("error: --device-budget needs --any-order");
  if (any_order && have_mats && !no_rows) die("error: --any-order writes either the TSV rows (--output) or the cell matrices (--cell-matrix --no-rows), not both: run the two modes separately");
  if (any_order && force_paired) die("error: --any-order cannot pair mates (-p): the mates of a position-sorted file are not neighbours");
  if (no_rows && !outs.empty()) die("error: --no-rows writes no TSV: leave out --output");
  if (no_rows && !have_mats) die("error: --no-rows needs --cell-matrix (there would be nothing to write)");
  if (have_mats && mats.size() != refs.size()) die("error: --cell-matrix needs one directory per reference library");
  if (refs.empty() || (outs.empty() && !no_rows) || ins.empty()) die("error: The following required arguments were not provided: --reference/--output/--input");
  char* end = nullptr; long ncores = strtol(cores.c_str(), &end, 10);
  if (*end || ncores < 0) die("Error -- please provide an integer value for the number of cores");
  int chem;
  if (strand == "unstranded") chem = NB_CHEM_UNSTRANDED; else if (strand == "fiveprime") chem = NB_CHEM_FIVEPRIME; else if (strand == "threeprime") chem = NB_CHEM_THREEPRIME; else if (strand == "none") chem = NB_CHEM_NONE; else die("Could not parse strand_filter option.");
  if (have_trim) {  // src/bin/main.rs:74-93
    size_t n = 1 + std::count(trim.begin(), trim.end(), ',');
    size_t p = 0;
    while (p <= trim.size()) { size_t e = trim.find(',', p); if (e == std::string::npos) e = trim.size(); std::string t = trim.substr(p, e - p); size_t c = t.find(':'); if (c == std::string::npos) die("Invalid strictness"); char* e1; strtoul(t.substr(0, c).c_str(), &e1, 10); if (*e1) die("Invalid length"); char* e2; strtod(t.substr(c + 1).c_str(), &e2); if (*e2) die("Invalid strictness"); p = e + 1; }
    if (n != refs.size()) die("The number of trim options does not match the number of reference libraries");
  }
  std::vector<int> devices;
  { size_t p = 0; while (p <= devs.size()) { size_t e = devs.find(',', p); if (e == std::string::npos) e = devs.size(); std::string t = devs.substr(p, e - p); char* e1; long v = strtol(t.c_str(), &e1, 10); if (t.empty() || *e1 || v < 0) die("Error -- please provide a comma-separated list of GPU ordinals for --devices"); devices.push_back((int)v); p = e + 1; } }
  std::string first = ins[0]; std::string lower = first; std::transform(lower.begin(), lower.end(), lower.begin(), ::tolower);
  auto ends = [](const std::string& s, const char* suf) { size_t n = strlen(suf); return s.size() >= n && s.compare(s.size() - n, n, suf) == 0; };
  std::vector<const char*> r, o, in;
  for (auto& s : refs) { printf("Loading and preprocessing reference data for %s\n", s.c_str()); r.push_back(s.c_str()); }
  for (auto& s : outs) o.push_back(s.c_str());
  for (auto& s : ins) in.push_back(s.c_str());
  if (!no_rows && outs.size() < refs.size()) die("index out of bounds: one output path per reference library is required");
  printf("Loading read sequences and aligning\n");
  std::vector<const char*> m; for (auto& s : mats) m.push_back(s.c_str());
  if (ends(first, ".fastq.gz") || ends(lower, ".fastq")) {
    if (have_mats || no_rows || any_order) die("error: --cell-matrix, --no-rows and --any-order need a BAM input (FASTQ reads have no cells)");
    printf("Processing as FASTQ file\n");
    int rc = nb_process_fastq_devices(in.data(), (uint32_t)std::min<size_t>(in.size(), 2), r.data(), o.data(), (uint32_t)r.size(), chem, (int)ncores, devices.data(), (uint32_t)devices.size());
    if (rc != NB_OK) die(nb_last_error());
  } else if (ends(lower, ".bam")) {
    printf("Processing as BAM file\n");
    int rc = (any_order && !have_mats) ? nb_process_bam_rows_any_order(in[0], r.data(), o.data(), (uint32_t)r.size(), chem, have_trim ? trim.c_str() : nullptr, (int)ncores, devices[0], have_budget ? device_budget : 0)
           : any_order ? (have_budget ? nb_process_bam_cells_any_order_budget(in[0], r.data(), m.data(), (uint32_t)r.size(), chem, have_trim ? trim.c_str() : nullptr, (int)ncores, devices[0], device_budget)
                                      : nb_process_bam_cells_any_order(in[0], r.data(), m.data(), (uint32_t)r.size(), chem, have_trim ? trim.c_str() : nullptr, (int)ncores, devices[0]))
                       : nb_process_bam_cells(in[0], r.data(), no_rows ? nullptr : o.data(), have_mats ? m.data() : nullptr, (uint32_t)r.size(), chem, have_trim ? trim.c_str() : nullptr, (int)ncores, force_paired ? 1 : 0, devices[0]);   // (BAM mode is bound by BGZF inflate and row formatting on the host: one GPU)
    if (rc != NB_OK) die(nb_last_error());
  } else die("Unsupported file format: " + (lower.find('.') == std::string::npos ? std::string("") : lower.substr(lower.rfind('.') + 1)));
  printf("Alignment successful, terminating.\n");
  return 0;
}
