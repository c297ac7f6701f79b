// sqy — command line front end over the C ABI of libsqeazy.so (B200 build).
//
// Mirrors the reference's `sqy` tool for the verbs of the volume-pipeline hot path (src/sqy.cpp:182-396,
// verbs/compress.hpp:225-338, verbs/decompress.hpp:30-233, verbs/bench.hpp:60-131,383-526, verbs/compare.hpp):
//   compress|enc|encode|comp   <tiff ..>   -p/--pipeline  -o/--output_name  -e/--output_suffix  -n/--nthreads  -v  -h
//   decompress|dec|decode|rec  <sqy ..>    -o/--output_name  -e/--output_suffix (default .tif)  --roi lo:hi[:step],.. (a box or strided slice only)
//   bench|ben                  <tiff ..>   + -c/--as-csv  --noheader  -r/--repetitions  --comment
//   compare|cmp                <a.tif> <b.tif>     (exit 0 when both stacks hold the same voxels)
// The reference CLI instantiates the C++ pipeline templates; this one only calls the exported SQY_* functions, i.e. it is
// also the smallest complete client of the drop-in boundary. TIFF I/O: tiff_min.hpp (no libtiff in this image). HDF5
// targets (.h5) are refused: there is no libhdf5 here (SQY_h5_* return 1).
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <map>
#include <numeric>
#include <sstream>
#include <string>
#include <vector>

#include "../../../include/sqeazy.h"
#include "../../../include/sqeazy_b200.h"
#include "tiff_min.hpp"

namespace {

struct Options {
  std::map<std::string, std::string> kv;   // long name -> value ("" for flags)
  std::vector<std::string> files;
  bool has(const std::string& k) const { return kv.count(k) != 0; }
  std::string get(const std::string& k, const std::string& d) const { auto f = kv.find(k); return f == kv.end() ? d : f->second; }
};

struct OptSpec { const char* longname; char shortname; bool takes_value; const char* help; };

const OptSpec kGeneral[] = {
    {"help", 'h', false, "produce help message"},
    {"verbose", 'v', false, "enable verbose output"},
    {"nthreads", 'n', true, "number of host threads to use (they stage the stack for the PCIe hop; <= 0: all cores)"},
};
const OptSpec kCompress[] = {
    {"pipeline", 'p', true, "compression pipeline to be used (default bitswap1->lz4)"},
    {"dataset_name", 'd', true, "name of the HDF5 dataset (ignored: no HDF5 in this build)"},
    {"output_name", 'o', true, "file location to write output to (if only 1 is given)"},
    {"output_suffix", 'e', true, "file extension to be used (must include period)"},
};
const OptSpec kDecompress[] = {
    {"roi", 0, true, "decompress only the slice lo:hi[:step],lo:hi[:step],.. (half-open, step >= 1, one range per dimension, in the order of the shape)"},
};
const OptSpec kBench[] = {
    {"as-csv", 'c', false, "print results as comma-separated table"},
    {"noheader", 0, false, "print results without header"},
    {"repetitions", 'r', true, "how many times to repeat the benchmark run (default 10)"},
    {"comment", 0, true, "comment value to fill in for every benchmark measurement"},
};

void print_specs(const OptSpec* s, size_t n) {
  for (size_t i = 0; i < n; ++i) {
    std::ostringstream name;
    if (s[i].shortname) name << "-" << s[i].shortname << " [ --" << s[i].longname << " ]";
    else name << "--" << s[i].longname;
    if (s[i].takes_value) name << " arg";
    std::cout << "  " << std::left << std::setw(32) << name.str() << s[i].help << "\n";
  }
}

// boost::program_options style: "--name value", "--name=value", "-n value", "-nvalue"; unknown words are input files
bool parse(int argc, char** argv, int first, const std::vector<const OptSpec*>& tables, const std::vector<size_t>& sizes, Options& out) {
  auto find_long = [&](const std::string& n) -> const OptSpec* {
    for (size_t t = 0; t < tables.size(); ++t)
      for (size_t i = 0; i < sizes[t]; ++i)
        if (n == tables[t][i].longname) return &tables[t][i];
    return nullptr;
  };
  auto find_short = [&](char c) -> const OptSpec* {
    for (size_t t = 0; t < tables.size(); ++t)
      for (size_t i = 0; i < sizes[t]; ++i)
        if (tables[t][i].shortname == c) return &tables[t][i];
    return nullptr;
  };
  for (int i = first; i < argc; ++i) {
    const std::string a = argv[i];
    if (a.size() > 2 && a[0] == '-' && a[1] == '-') {
      const size_t eq = a.find('=');
      const std::string name = a.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
      const OptSpec* s = find_long(name);
      if (!s) { out.files.push_back(a); continue; }   // allow_unregistered(): collected with the positionals
      if (!s->takes_value) out.kv[name] = "";
      else if (eq != std::string::npos) out.kv[name] = a.substr(eq + 1);
      else if (i + 1 < argc) out.kv[name] = argv[++i];
      else { std::cerr << "[sqy] option --" << name << " needs a value\n"; return false; }
    } else if (a.size() >= 2 && a[0] == '-' && a[1] != '-') {
      const OptSpec* s = find_short(a[1]);
      if (!s) { out.files.push_back(a); continue; }
      if (!s->takes_value) out.kv[s->longname] = "";
      else if (a.size() > 2) out.kv[s->longname] = a.substr(2);
      else if (i + 1 < argc) out.kv[s->longname] = argv[++i];
      else { std::cerr << "[sqy] option -" << a[1] << " needs a value\n"; return false; }
    } else {
      out.files.push_back(a);
    }
  }
  return true;
}

bool matches(const std::string& verb, std::initializer_list<const char*> aliases) {
  for (const char* a : aliases)
    if (verb == a) return true;
  return false;
}

std::string extension_of(const std::string& p) {
  const size_t slash = p.find_last_of('/');
  const size_t dot = p.find_last_of('.');
  if (dot == std::string::npos || (slash != std::string::npos && dot < slash)) return "";
  return p.substr(dot);
}
std::string replace_extension(const std::string& p, const std::string& ext) {
  const std::string e = extension_of(p);
  return p.substr(0, p.size() - e.size()) + ext;
}
std::string stem_of(const std::string& p) {
  const size_t slash = p.find_last_of('/');
  const std::string base = slash == std::string::npos ? p : p.substr(slash + 1);
  const std::string e = extension_of(base);
  return base.substr(0, base.size() - e.size());
}
bool file_exists(const std::string& p) { std::ifstream f(p, std::ios::binary); return f.good(); }

// verbs/compress.hpp:268-283, verbs/decompress.hpp:198-209: suffix with a period replaces the extension, one without is
// appended to the stem; --output_name wins when a single input is given
std::string target_name(const std::string& input, const Options& o, const std::string& default_suffix) {
  std::string out = replace_extension(input, default_suffix);
  const std::string suffix = o.get("output_suffix", default_suffix);
  if (!suffix.empty() && suffix.front() == '.') out = replace_extension(input, suffix);
  else out = stem_of(input) + suffix;
  if (o.has("output_name") && o.files.size() == 1) out = o.get("output_name", out);
  return out;
}

int brief_help() {
  std::cout << "usage: sqy <-h|optional> <verb> <files|..>\n\n"
            << "available verbs (their description and aliases):\n"
            << "    bench              benchmark the compression to native sqy format                 (ben|bench)\n"
            << "    compare            compare two tiff stacks and see if they are equal              (compare|cmp)\n"
            << "    compress           compress a tiff stack to native sqy format                     (compress|enc|encode|comp)\n"
            << "    decompress         decompress a .sqy file to tiff                                 (decompress|dec|decode|rec)\n"
            << "    help               print a help message\n"
            << "    <verb> -h/--help   print detailed help for <verb>, e.g. sqy compress -h\n\n"
            << "available flags to sqy only:\n"
            << "  -h [ --help ]                   produce help message\n"
            << "  --fullhelp                      produce exhaustive help message with all verbs documented\n"
            << "  -v [ --version ]                print the version of this sqy build\n\n"
            << "verbs of the reference tool that are not part of this build: scan, diff, convert (.yuv/.y4m), HDF5 targets\n";
  return 0;
}

void pipeline_help() {
  std::cout << "pipeline builder\n----------------\n"
            << "  stages are joined by '->', parameters go in parentheses: remove_background(threshold=110)->bitswap1->lz4\n"
            << "available filters (before sink), 16-bit stacks: bitswap1 bitswap2 bitswap4 bitswap8 remove_background rmestbkrd\n"
            << "available filters (before sink),  8-bit stacks: bitswap1 bitswap2 bitswap4 remove_background\n"
            << "available sinks: lz4 quantiser(16-bit only) pass_through\n"
            << "available filters (after sink): lz4\n\n";
}

bool read_file(const std::string& path, std::vector<char>& buf) {
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  if (!f.good()) return false;
  const std::streamsize n = f.tellg();
  f.seekg(0);
  buf.resize((size_t)n);
  return n == 0 || (bool)f.read(buf.data(), n);
}

// one encode through the C ABI; returns blob bytes or 0
long encode_stack(const sqycli::TiffStack& in, const std::string& pipeline, int nthreads, std::vector<char>& blob, bool verbose) {
  std::vector<long> shape(in.shape.begin(), in.shape.end());
  long cap = (long)in.data.size();
  const int rc_len = in.bits == 16 ? SQY_Pipeline_Max_Compressed_Length_UI16(pipeline.c_str(), (long)pipeline.size(), &cap)
                                   : SQY_Pipeline_Max_Compressed_Length_UI8(pipeline.c_str(), (long)pipeline.size(), &cap);
  if (rc_len) return 0;
  if (blob.size() < (size_t)cap) blob.resize((size_t)cap);
  long n = 0;
  const int rc = in.bits == 16 ? SQY_PipelineEncode_UI16(pipeline.c_str(), in.data.data(), shape.data(), (unsigned)shape.size(), blob.data(), &n, nthreads)
                               : SQY_PipelineEncode_UI8(pipeline.c_str(), in.data.data(), shape.data(), (unsigned)shape.size(), blob.data(), &n, nthreads);
  if (rc) {
    if (verbose) std::cerr << "[SQY]\tnative compression failed! Nothing to write to disk...\n";
    return 0;
  }
  return n;
}

bool pipeline_ok(const std::string& p, int bits) { return SQY_Pipeline_Possible(p.c_str(), bits / 8); }

int compress_files(const Options& o) {
  int value = 1;
  const std::string pipeline = o.get("pipeline", "bitswap1->lz4");
  if (!pipeline_ok(pipeline, 16) && !pipeline_ok(pipeline, 8)) {
    std::cerr << "[SQY]\tunable to build pipeline from " << pipeline << "\nDoing nothing.\n";
    return value;
  }
  const int nthreads = std::atoi(o.get("nthreads", "1").c_str());
  if (o.files.size() > 1) std::cout << "[SQY]\tmultiple input files detected, ignoring --output_name flag\n";
  std::vector<char> blob;
  for (const std::string& file : o.files) {
    if (!file_exists(file)) { std::cerr << "[SQY]\tunable to open " << file << "\t skipping it\n"; continue; }
    sqycli::TiffStack in;
    const std::string err = sqycli::tiff_read(file, in);
    if (!err.empty()) { std::cerr << "[SQY]\t" << file << ": " << err << "\t skipping it\n"; continue; }
    const std::string out = target_name(file, o, ".sqy");
    size_t written = 0;
    if (extension_of(out) == ".sqy") {
      if (!pipeline_ok(pipeline, in.bits)) {
        std::cerr << "[SQY]\tunable to build pipeline from " << pipeline << " for " << in.bits << "-bit input\n";
      } else {
        const long n = encode_stack(in, pipeline, nthreads, blob, o.has("verbose"));
        if (n > 0) {
          std::ofstream f(out, std::ios::binary);
          if (!f.good()) std::cerr << "[SQY]\tunable to open " << out << "as output file. Skipping it!\n";
          else { f.write(blob.data(), n); written = f.good() ? (size_t)n : 0; }
          if (o.has("verbose") && written)
            std::cout << "[SQY]\t" << file << " -> " << out << " (" << in.data.size() << " -> " << written << " bytes, ratio "
                      << (double)in.data.size() / (double)written << ")\n";
        }
      }
    } else {
      std::cerr << "[SQY]\toutput format " << extension_of(out) << " is not available in this build (native .sqy only)\n";
    }
    if (!written) std::cerr << "[SQY]\terrors occurred while processing " << file << "\n";
    else value = 0;
  }
  return value;
}

// "lo:hi[:step],.." -> {lo_0, hi_0, step_0, lo_1, ..} (step 1 when it is left out); false when it is not of that form, a range
// is empty (lo >= hi: a TIFF has no page of zero extent) or a step is less than 1
bool parse_roi(const std::string& text, std::vector<long>& slices) {
  slices.clear();
  std::stringstream ss(text);
  std::string range;
  while (std::getline(ss, range, ',')) {
    const size_t colon = range.find(':');
    if (colon == std::string::npos) return false;
    char* end = nullptr;
    const long lo = std::strtol(range.c_str(), &end, 10);
    if (end != range.c_str() + colon) return false;
    const char* hi_text = range.c_str() + colon + 1;
    const long hi = std::strtol(hi_text, &end, 10);
    if (end == hi_text || lo >= hi) return false;
    long step = 1;
    if (*end == ':') {
      const char* step_text = end + 1;
      step = std::strtol(step_text, &end, 10);
      if (end == step_text || step < 1) return false;
    }
    if (*end != '\0') return false;
    slices.insert(slices.end(), {lo, hi, step});
  }
  return !slices.empty();
}

int decompress_files(const Options& o) {
  int value = 1;
  std::vector<long> slices;
  if (o.has("roi") && !parse_roi(o.get("roi", ""), slices)) {
    std::cerr << "[SQY]\t--roi expects lo:hi[:step],.. (one non-empty range per dimension, lo < hi, step >= 1)\n";
    return 1;
  }
  const int nthreads = std::atoi(o.get("nthreads", "1").c_str());
  if (o.files.size() > 1) std::cout << "[SQY]\tmultiple input files detected, ignoring --output_name flag\n";
  std::vector<char> blob, raw;
  for (const std::string& file : o.files) {
    if (!file_exists(file)) { std::cerr << "[SQY]\tunable to open " << file << "\t skipping it\n"; continue; }
    if (extension_of(file) != ".sqy") {
      std::cerr << "[SQY]\t" << file << ": only native .sqy files can be decompressed by this build\n";
      continue;
    }
    if (!read_file(file, blob) || blob.empty()) { std::cerr << "[SQY]\tunable to load " << file << "\n"; continue; }
    long nd = (long)blob.size(), bytes = (long)blob.size(), so = (long)blob.size();
    if (SQY_Decompressed_NDims(blob.data(), &nd) || nd <= 0 || nd > 8 || SQY_Decompressed_Length(blob.data(), &bytes) ||
        SQY_Decompressed_Sizeof(blob.data(), &so) || (so != 1 && so != 2)) {
      std::cerr << "[SQY]\t" << file << " has no usable sqy header\n";
      continue;
    }
    std::vector<long> shape((size_t)nd, 0);
    shape[0] = (long)blob.size();
    if (SQY_Decompressed_Shape(blob.data(), shape.data())) { std::cerr << "[SQY]\t" << file << " has no usable sqy header\n"; continue; }
    int rc = 0;
    if (o.has("roi")) {
      // the slice alone, in the dimension order of the shape
      if (slices.size() != 3 * shape.size()) { std::cerr << "[SQY]\t" << file << ": --roi needs " << shape.size() << " ranges\n"; continue; }
      bytes = so;
      for (size_t k = 0; k < shape.size(); ++k) {
        shape[k] = std::max((slices[3 * k + 1] - slices[3 * k] + slices[3 * k + 2] - 1) / slices[3 * k + 2], 0l);
        bytes *= shape[k];
      }
      raw.resize((size_t)bytes);
      rc = so == 2 ? sqyx_decode_slice_UI16(blob.data(), (long)blob.size(), slices.data(), (unsigned)shape.size(), raw.data(), bytes, nthreads)
                   : sqyx_decode_slice_UI8(blob.data(), (long)blob.size(), slices.data(), (unsigned)shape.size(), raw.data(), bytes, nthreads);
    } else {
      raw.resize((size_t)bytes);
      rc = so == 2 ? SQY_Decode_UI16(blob.data(), (long)blob.size(), raw.data(), nthreads)
                   : SQY_Decode_UI8(blob.data(), (long)blob.size(), raw.data(), nthreads);
    }
    if (rc) { std::cerr << "[SQY]\tdecompressing " << file << " failed! Nothing to write to disk...\n"; continue; }
    const std::string out = target_name(file, o, ".tif");
    const std::string err = sqycli::tiff_write(out, std::vector<uint64_t>(shape.begin(), shape.end()), (int)so * 8, raw.data());
    if (!err.empty()) { std::cerr << "[SQY]\t" << err << "\n"; continue; }
    if (o.has("verbose")) std::cout << "[SQY]\t" << file << " -> " << out << " (" << blob.size() << " -> " << bytes << " bytes)\n";
    value = 0;
  }
  return value;
}

// verbs/bench.hpp:60-131: one row per repetition; ingest bandwidth in MiB/s of raw input
int bench_files(const Options& o) {
  int value = 1;
  const std::string pipeline = o.get("pipeline", "bitswap1->lz4");
  if (!pipeline_ok(pipeline, 16) && !pipeline_ok(pipeline, 8)) {
    std::cerr << "[SQY]\tunable to build pipeline from " << pipeline << "\nDoing nothing.\n";
    return value;
  }
  const int nthreads = std::atoi(o.get("nthreads", "1").c_str());
  const int reps = std::max(1, std::atoi(o.get("repetitions", "10").c_str()));
  const bool csv = o.has("as-csv");
  bool header = !o.has("noheader");
  std::ostringstream cmt;
  cmt << pipeline << "|" << nthreads << "threads|" << (long)std::time(nullptr);
  const std::string comment = o.get("comment", "").empty() ? cmt.str() : o.get("comment", "");
  const std::string delim = csv ? "," : "";
  std::vector<char> blob;
  for (const std::string& file : o.files) {
    if (!file_exists(file)) { std::cerr << "[SQY]\tunable to open " << file << "\t skipping it\n"; continue; }
    sqycli::TiffStack in;
    const std::string err = sqycli::tiff_read(file, in);
    if (!err.empty() || !pipeline_ok(pipeline, in.bits)) { std::cerr << "[SQY]\t" << file << ": " << (err.empty() ? "pipeline not available for this bit depth" : err) << "\n"; continue; }
    std::ostringstream shp;
    for (size_t i = 0; i < in.shape.size(); ++i) shp << in.shape[i] << (i + 1 < in.shape.size() ? "x" : "");
    const uint64_t len = in.voxels();
    const int so = in.bits / 8;
    if (header) {
      auto w = [&](int n) { return csv ? std::setw(0) : std::setw(n); };
      std::cout << w(2) << "id" << delim << w(15) << "shape" << delim << w(15) << "time_mus" << delim << w(15) << "final_bytes" << delim << w(18)
                << "ingest_bw_mbps" << delim << w(15) << "sizeof_pixel" << delim << w(15) << "n_elements" << delim;
      if (csv) std::cout << "filename" << delim << "comment";
      else std::cout << " filename+comment";
      std::cout << "\n";
      header = false;
    }
    for (int i = 0; i < reps; ++i) {
      const auto t0 = std::chrono::high_resolution_clock::now();
      const long n = encode_stack(in, pipeline, nthreads, blob, o.has("verbose"));
      const auto t1 = std::chrono::high_resolution_clock::now();
      if (n <= 0) { std::cerr << "[SQY]\tnative benchmark of compression at iteration " << i << " failed! Exiting.\n"; return 1; }
      const double mus = std::chrono::duration<double, std::micro>(t1 - t0).count();
      const float bw = float(len * (uint64_t)so) / (1024.f * 1024.f) / float(mus * 1e-6);
      auto w = [&](int nn) { return csv ? std::setw(0) : std::setw(nn); };
      std::cout << w(2) << i << delim << w(15) << shp.str() << delim << w(15) << mus << delim << w(15) << n << delim << w(18) << bw << delim << w(15)
                << so << delim << w(15) << len << delim << (csv ? "\"" : " ") << file << (csv ? "\"" : ",") << delim << (csv ? "\"" : " ") << comment
                << (csv ? "\"" : "") << "\n";
      value = 0;
    }
  }
  return value;
}

int compare_files(const Options& o) {
  if (o.files.size() != 2) { std::cerr << "[SQY]\tcompare needs exactly two tiff files\n"; return 1; }
  sqycli::TiffStack a, b;
  std::string err = sqycli::tiff_read(o.files[0], a);
  if (!err.empty()) { std::cerr << "[SQY]\t" << o.files[0] << ": " << err << "\n"; return 1; }
  err = sqycli::tiff_read(o.files[1], b);
  if (!err.empty()) { std::cerr << "[SQY]\t" << o.files[1] << ": " << err << "\n"; return 1; }
  const bool same = a.shape == b.shape && a.bits == b.bits && a.data == b.data;
  if (o.has("verbose") || !same)
    std::cout << "[SQY]\t" << o.files[0] << (same ? " == " : " != ") << o.files[1] << "\n";
  return same ? 0 : 1;
}

}  // namespace

int main(int argc, char** argv) {
  if (argc < 2) return brief_help();
  const std::string verb = argv[1];
  std::vector<const OptSpec*> tables = {kGeneral};
  std::vector<size_t> sizes = {sizeof(kGeneral) / sizeof(OptSpec)};
  enum { None, Compress, Decompress, Bench, Compare } mode = None;
  if (matches(verb, {"compress", "enc", "encode", "comp"})) mode = Compress;
  else if (matches(verb, {"decompress", "dec", "decode", "rec"})) mode = Decompress;
  else if (matches(verb, {"bench", "ben"})) mode = Bench;
  else if (matches(verb, {"compare", "cmp"})) mode = Compare;
  if (mode == None) {
    if (verb == "-v" || verb == "--version") {
      int v[3] = {0, 0, 0};
      SQY_Version_Triple(v);
      std::cout << "sqy " << v[0] << "." << v[1] << "." << v[2] << " (b200)\n";
      return 1;   // like the reference (sqy.cpp:318-324)
    }
    if (verb == "-h" || verb == "--help" || verb == "--fullhelp") {
      brief_help();
      if (verb == "--fullhelp") pipeline_help();
      return verb == "--fullhelp" ? 1 : 0;
    }
    std::cerr << "unable to find matching verb for " << verb << "\n";
    brief_help();
    return 1;
  }
  if (mode == Compress || mode == Bench || mode == Decompress) { tables.push_back(kCompress); sizes.push_back(sizeof(kCompress) / sizeof(OptSpec)); }
  if (mode == Bench) { tables.push_back(kBench); sizes.push_back(sizeof(kBench) / sizeof(OptSpec)); }
  if (mode == Decompress) { tables.push_back(kDecompress); sizes.push_back(sizeof(kDecompress) / sizeof(OptSpec)); }
  Options o;
  if (!parse(argc, argv, 2, tables, sizes, o)) return 1;
  if (o.has("help")) {
    for (size_t t = 0; t < tables.size(); ++t) print_specs(tables[t], sizes[t]);
    std::cout << "\n";
    if (mode == Compress || mode == Bench) pipeline_help();
    return 1;
  }
  if (o.files.empty()) {
    std::cerr << "[sqy] no input files given, exiting ...\n";
    return 1;
  }
  switch (mode) {
    case Compress: return compress_files(o);
    case Decompress: return decompress_files(o);
    case Bench: return bench_files(o);
    case Compare: return compare_files(o);
    default: return 1;
  }
}
