// ecdna -- host front end over libecdna_b200.so with the reference's command line and output files.
//
// Mirrors, flag for flag, the clap definition of the reference (src/clap_app.rs:26-100) and the
// defaults that Cli::build derives (clap_app.rs:136-230); replaces the rayon loop over replicate
// indices (src/main.rs:212-225) by one call of ecdna_b200_run(); writes the same files as `save`
// (src/process.rs:31-55) with the names of src/lib.rs:27-45: one JSON histogram per triggered
// snapshot, one for the final state, one per --subsamples size.
//
// The index range runs on every visible B200 (ecdna_b200_multi_run_sparse: one host thread and context per GPU; the
// distributions come back as descriptors + occupied bins, a tenth of the dense form for the default snapshots),
// in chunks, so that host memory is O(chunk) whatever --runs is; the files of a chunk are written while the
// next one is simulated.  `ecdna abc --target FILE.json ...` is the front end of the reference's removed ABC
// binary (abc.md:10-55): prior draws over (b1, d0, d1), one run per draw, abc.csv with every draw;
// `ecdna abc --generations G` runs ABC-SMC instead (ecdna_b200_abc_smc_ex) and writes one CSV per population.
//
// The reference is Rust; no Rust toolchain exists in this image, so the host side above the C ABI is
// C++ (INTEGRATION.md shows the Rust binding a maintainer would add instead of this file).
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <future>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "ecdna_b200.h"

namespace {

constexpr uint64_t kMaxIter = 1000000000ull;   // main.rs:23
constexpr uint64_t kMaxCells = 1000000000ull;  // main.rs:25

struct Cli {
  std::string segregation = "binomial";  // clap_app.rs:35-36
  std::string growth = "exponential";    // clap_app.rs:38-39
  float b0 = 1.f, b1 = 1.f;              // clap_app.rs:41-45
  bool has_d0 = false, has_d1 = false;
  float d0 = 0.f, d1 = 0.f;              // clap_app.rs:49-55
  bool has_years = false, has_cells = false;
  uint64_t years = 0, cells = 0;         // clap_app.rs:57-61
  uint64_t seed = 26;                    // clap_app.rs:63-64
  bool debug = false, sequential = false;
  std::string path, initial;
  uint64_t runs = 12;                    // clap_app.rs:89-91
  bool has_subsamples = false, has_snapshots = false;
  std::vector<uint64_t> subsamples, snapshots;
  int verbosity = 0;
  // outputs the reference dropped after 0.19/0.23 (CHANGELOG.md:14-16, 34-40), off by default
  bool summaries = false;  // mean / frequency / entropy of the final distribution
  bool dynamics = false;   // 300 samples of (nminus, nplus, mean, variance, entropy) every 0.1 time units
  // engine knobs (not in the reference)
  std::vector<int> devices;  // empty = every visible B200
  uint64_t chunk = 0;        // replicates per library call (0 = sized for ~2 GiB of host buffers per GPU)
  uint32_t tile_width = 0, state_mode = 0;
  uint32_t bd_count_mode = 0;  // 0: --cells counts cells; 1: sosa's literal population sum (SURVEY 8c R1)
  // `ecdna abc` (abc.md:10-55)
  bool abc = false;
  std::string target;
  float b1_range[2] = {1.f, 2.f}, d0_range[2] = {0.f, 0.5f}, d1_range[2] = {0.f, 0.5f};
  float thresholds[4] = {0.05f, 0.1f, 0.1f, 0.1f};
  // `ecdna abc --generations G`: ABC-SMC (0 = rejection ABC over --runs draws)
  uint32_t generations = 0, population = 1000;
  double quantile = 0.5;
  uint64_t max_simulations = 10000000ull;
  uint32_t smc_kernel = ECDNA_B200_SMC_KERNEL_COMPONENT;
};

[[noreturn]] void die(const std::string& msg) {
  std::fprintf(stderr, "error: %s\n\nFor more information, try '--help'.\n", msg.c_str());
  std::exit(2);
}

void usage() {
  std::puts(
      "Study the effect of the random segregation and positive selection on the ecDNA dynamics using a\n"
      "stochastic simulation algorithm (SSA) aka Gillespie algorithm  [B200 backend]\n\n"
      "Usage: ecdna [OPTIONS] <DIR>\n\n"
      "Arguments:\n  <DIR>  Path to store the results of the simulations\n\n"
      "Options:\n"
      "      --segregation <SEGREGATION>  [default: binomial] [possible values: deterministic,\n"
      "                                   binomial-no-uneven, binomial, binomial-no-nminus]\n"
      "      --growth <GROWTH>            [default: exponential] [possible values: exponential, constant]\n"
      "      --b0 <RATE>                  Proliferation rate of the cells without ecDNAs [default: 1]\n"
      "      --b1 <RATE>                  Proliferation rate of the cells with ecDNAs [default: 1]\n"
      "      --d0 <RATE>                  Death rate of the cells without ecDNAs\n"
      "      --d1 <RATE>                  Death rate of the cells with ecDNAs\n"
      "  -y, --years <YEARS>              Number of years to simulate before stopping\n"
      "  -c, --cells <CELLS>              Number of cells to simulate before stopping\n"
      "      --seed <SEED>                Seed for reproducibility [default: 26]\n"
      "  -d, --debug                      max verbosity, 1 sequential simulation\n"
      "  -s, --sequential                 accepted for compatibility (replicates always run on the GPU)\n"
      "      --initial <FILE>             The JSON file used as an initial starting distribution\n"
      "  -r, --runs <RUNS>                Number of independent realisations [default: 12]\n"
      "      --subsamples[=<N>...]        Subsample the ecDNA distribution at the end of the simulation\n"
      "      --snapshots[=<N>...]         Number of cells that will trigger the saving of the distribution\n"
      "  -v, --verbosity...\n"
      "      --summaries                  also write <cells>cells/{mean,frequency,entropy}/<t>years/<name>.json\n"
      "      --dynamics                   also write <cells>cells/dynamics/<t>years/<name>.json (300 x 0.1)\n"
      "      --devices <all|N,N,...>      GPUs to use [default: all]   --chunk <N> replicates per library call\n"
      "      --tile-width <1|2|4|8|16|32>  --state <auto|smem|hbm>   (B200 engine knobs)\n"
      "      --bd-count-mode <cells|sosa-sum>  what --cells counts for the birth-death process [default: cells]\n"
      "  -h, --help\n  -V, --version\n\n"
      "ABC (abc.md): ecdna abc --target <FILE.json> [-r draws] [--b1-range lo,hi] [--d0-range lo,hi] [--d1-range lo,hi]\n"
      "              [--thresholds ks,mean,entropy,frequency] [--cells N] [--seed S] [--initial FILE] <DIR>\n"
      "              writes <DIR>/abc.csv (every draw) and <DIR>/abc_accepted.csv\n"
      "ABC-SMC:      ecdna abc --target <FILE.json> --generations <G> [--population M] [--quantile A]\n"
      "              [--max-simulations S] [--kernel K] [the ranges, thresholds and model options above] <DIR>\n"
      "              populations of M particles [default: 1000], the tolerance of generation t+1 the A-quantile\n"
      "              [default: 0.5] of generation t's distances, until the thresholds themselves are reached, G\n"
      "              generations or S draws [default: 10000000]; writes <DIR>/abc_gen<t>.csv per generation and\n"
      "              <DIR>/abc_smc.json (cannot be combined with --runs); --kernel: the perturbation kernel\n"
      "              [default: component] [possible values: component (a Gaussian per parameter), mvn (2 x the\n"
      "              population covariance), olcm (a local covariance per particle)]");
}

std::vector<uint64_t> parse_list(const std::string& v) {
  std::vector<uint64_t> out;
  std::stringstream ss(v);
  std::string tok;
  while (std::getline(ss, tok, ',')) {
    if (tok.empty()) continue;
    char* end = nullptr;
    const unsigned long long x = std::strtoull(tok.c_str(), &end, 10);
    if (*end) die("invalid value '" + tok + "': invalid digit found in string");
    out.push_back(x);
  }
  return out;
}

Cli parse(int argc, char** argv) {
  Cli c;
  bool have_path = false, runs_given = false, verb_given = false, smc_opt_given = false, generations_given = false;
  auto need = [&](int& i, const std::string& name) -> std::string {
    if (i + 1 >= argc) die("a value is required for '" + name + "' but none was supplied");
    return argv[++i];
  };
  auto number = [&](const std::string& v, const std::string& name) -> double {  // clap: "invalid value"
    char* end = nullptr;
    const double x = std::strtod(v.c_str(), &end);
    if (v.empty() || *end) die("invalid value '" + v + "' for '" + name + "': invalid number");
    return x;
  };
  auto pair_of = [&](const std::string& v, float* out) {
    const size_t comma = v.find(',');
    if (comma == std::string::npos) die("invalid range '" + v + "': expected lo,hi");
    out[0] = std::strtof(v.substr(0, comma).c_str(), nullptr);
    out[1] = std::strtof(v.substr(comma + 1).c_str(), nullptr);
  };
  int first = 1;
  if (argc > 1 && std::string(argv[1]) == "abc") { c.abc = true; first = 2; }
  for (int i = first; i < argc; ++i) {
    std::string a = argv[i], val;
    const size_t eq = a.find('=');
    bool has_eq = false;
    if (a.rfind("--", 0) == 0 && eq != std::string::npos) { val = a.substr(eq + 1); a = a.substr(0, eq); has_eq = true; }
    auto value = [&]() { return has_eq ? val : need(i, a); };
    if (a == "-h" || a == "--help") { usage(); std::exit(0); }
    else if (a == "-V" || a == "--version") { std::puts("Dynamics 0.26.0-b200"); std::exit(0); }
    else if (a == "--segregation") c.segregation = value();
    else if (a == "--growth") c.growth = value();
    else if (a == "--b0") c.b0 = std::strtof(value().c_str(), nullptr);
    else if (a == "--b1") c.b1 = std::strtof(value().c_str(), nullptr);
    else if (a == "--d0") { c.d0 = std::strtof(value().c_str(), nullptr); c.has_d0 = true; }
    else if (a == "--d1") { c.d1 = std::strtof(value().c_str(), nullptr); c.has_d1 = true; }
    else if (a == "-y" || a == "--years") { c.years = std::strtoull(value().c_str(), nullptr, 10); c.has_years = true; }
    else if (a == "-c" || a == "--cells") { c.cells = std::strtoull(value().c_str(), nullptr, 10); c.has_cells = true; }
    else if (a == "--seed") c.seed = std::strtoull(value().c_str(), nullptr, 10);
    else if (a == "-d" || a == "--debug") c.debug = true;
    else if (a == "-s" || a == "--sequential") c.sequential = true;
    else if (a == "--initial") c.initial = value();
    else if (a == "-r" || a == "--runs") { c.runs = std::strtoull(value().c_str(), nullptr, 10); runs_given = true; }
    else if (a == "--subsamples") { c.has_subsamples = true; if (has_eq) c.subsamples = parse_list(val); }  // require_equals
    else if (a == "--snapshots") { c.has_snapshots = true; if (has_eq) c.snapshots = parse_list(val); }
    else if (a == "--summaries") c.summaries = true;
    else if (a == "--dynamics") c.dynamics = true;
    else if (a == "--device" || a == "--devices") {
      const std::string v = value();
      if (v != "all") for (uint64_t d : parse_list(v)) c.devices.push_back((int)d);
    }
    else if (a == "--chunk") c.chunk = std::strtoull(value().c_str(), nullptr, 10);
    else if (a == "--bd-count-mode") {
      const std::string v = value();
      if (v != "cells" && v != "sosa-sum") die("invalid value '" + v + "' for '--bd-count-mode' [possible values: cells, sosa-sum]");
      c.bd_count_mode = v == "sosa-sum" ? 1u : 0u;
    }
    else if (c.abc && a == "--target") c.target = value();
    else if (c.abc && a == "--b1-range") pair_of(value(), c.b1_range);
    else if (c.abc && a == "--d0-range") pair_of(value(), c.d0_range);
    else if (c.abc && a == "--d1-range") pair_of(value(), c.d1_range);
    else if (c.abc && a == "--thresholds") {
      std::stringstream ss(value());
      std::string tok;
      int j = 0;
      while (std::getline(ss, tok, ',') && j < 4) c.thresholds[j++] = std::strtof(tok.c_str(), nullptr);
      if (j != 4) die("--thresholds needs four values: ks,mean,entropy,frequency");
    }
    else if (a == "--generations") {
      const double g = number(value(), "--generations <G>");
      if (!(g >= 1.0 && g <= 4294967295.0) || g != std::floor(g)) die("invalid value for '--generations <G>': must be an integer >= 1");
      c.generations = (uint32_t)g;
      generations_given = true;
    }
    else if (c.abc && a == "--population") {
      const double m = number(value(), "--population <M>");
      if (!(m >= 1.0 && m <= 4294967295.0) || m != std::floor(m)) die("invalid value for '--population <M>': must be an integer >= 1");
      c.population = (uint32_t)m;
      smc_opt_given = true;
    }
    else if (c.abc && a == "--quantile") {
      c.quantile = number(value(), "--quantile <A>");
      if (!(c.quantile > 0.0 && c.quantile < 1.0)) die("invalid value for '--quantile <A>': must lie in (0, 1)");
      smc_opt_given = true;
    }
    else if (c.abc && a == "--max-simulations") {
      const double s = number(value(), "--max-simulations <S>");
      if (!(s >= 0.0 && s < 1.8e19) || s != std::floor(s)) die("invalid value for '--max-simulations <S>': must be an integer >= 0 (0 = no limit)");
      c.max_simulations = (uint64_t)s;
      smc_opt_given = true;
    }
    else if (c.abc && a == "--kernel") {
      const std::string v = value();
      if (v == "component") c.smc_kernel = ECDNA_B200_SMC_KERNEL_COMPONENT;
      else if (v == "mvn") c.smc_kernel = ECDNA_B200_SMC_KERNEL_MVN;
      else if (v == "olcm") c.smc_kernel = ECDNA_B200_SMC_KERNEL_OLCM;
      else die("invalid value '" + v + "' for '--kernel' [possible values: component, mvn, olcm]");
      smc_opt_given = true;
    }
    else if (a == "--tile-width") c.tile_width = (uint32_t)std::atoi(value().c_str());
    else if (a == "--state") {
      const std::string s = value();
      c.state_mode = s == "smem" ? ECDNA_B200_STATE_SMEM : (s == "hbm" ? ECDNA_B200_STATE_HBM : ECDNA_B200_STATE_AUTO);
    }
    else if (a.size() >= 2 && a[0] == '-' && a[1] == 'v') { c.verbosity += (int)a.size() - 1; verb_given = true; }
    else if (a == "--verbosity") { c.verbosity += 1; verb_given = true; }
    else if (!a.empty() && a[0] == '-') die("unexpected argument '" + a + "' found");
    else if (!have_path) { c.path = a; have_path = true; }
    else die("unexpected argument '" + a + "' found");
  }
  if (!have_path) die("the following required arguments were not provided:\n  <DIR>");
  if (c.abc && c.target.empty()) die("the following required arguments were not provided:\n  --target <FILE.json>");
  if (generations_given && !c.abc) die("the argument '--generations <G>' is only valid after the 'abc' subcommand");
  if (generations_given && runs_given) die("the argument '--generations <G>' cannot be used with '--runs <RUNS>'");
  if (smc_opt_given && !generations_given)
    die("the arguments '--population', '--quantile', '--max-simulations' and '--kernel' require '--generations <G>'");
  if (c.has_years && c.has_cells) die("the argument '--years <YEARS>' cannot be used with '--cells <CELLS>'");
  if (c.debug && (c.has_years || c.has_cells || c.sequential || runs_given || verb_given))
    die("the argument '--debug' cannot be used with one or more of the other specified arguments");
  if (!c.initial.empty() && (c.initial.size() < 5 || c.initial.substr(c.initial.size() - 5) != ".json"))
    die("invalid value '" + c.initial + "' for '--initial <FILE>': Must be JSON file: extension must be .json)");
  return c;
}

// Rust's `f32::to_string`: shortest decimal that round-trips, never in exponent form
std::string rust_f32_to_string(float v) {
  if (std::isnan(v)) return "NaN";
  if (std::isinf(v)) return v > 0 ? "inf" : "-inf";
  if (v == 0.f) return std::signbit(v) ? "-0" : "0";
  char buf[64];
  int prec = 0;
  for (; prec < 9; ++prec) {
    std::snprintf(buf, sizeof buf, "%.*e", prec, (double)v);
    if (std::strtof(buf, nullptr) == v) break;
  }
  std::string digits;
  const char* p = buf;
  bool neg = false;
  if (*p == '-') { neg = true; ++p; }
  for (; *p && *p != 'e'; ++p) if (*p != '.') digits.push_back(*p);
  const int exp10 = std::atoi(p + 1);
  while (digits.size() > 1 && digits.back() == '0') digits.pop_back();
  std::string out;
  const int point = exp10 + 1;  // digits before the decimal point
  if (point <= 0) out = "0." + std::string((size_t)-point, '0') + digits;
  else if ((size_t)point >= digits.size()) out = digits + std::string((size_t)point - digits.size(), '0');
  else out = digits.substr(0, (size_t)point) + "." + digits.substr((size_t)point);
  return neg ? "-" + out : out;
}
std::string dotted(float v) {
  std::string s = rust_f32_to_string(v);
  std::string out;
  for (char ch : s) { if (ch == '.') out += "dot"; else out.push_back(ch); }
  return out;
}
// lib.rs:27-45
std::string make_filename(const Cli& c, bool birth_death, float d0, float d1, uint64_t idx) {
  if (birth_death) return dotted(c.b0) + "b0_" + dotted(c.b1) + "b1_" + dotted(d0) + "d0_" + dotted(d1) + "d1_" + std::to_string(idx) + "idx";
  return dotted(c.b0) + "b0_" + dotted(c.b1) + "b1_0d0_0d1_" + std::to_string(idx) + "idx";
}

void mkdirs(const std::string& path) {
  std::string cur;
  for (size_t i = 0; i <= path.size(); ++i) {
    if (i == path.size() || path[i] == '/') {
      if (!cur.empty()) ::mkdir(cur.c_str(), 0777);
    }
    if (i < path.size()) cur.push_back(path[i]);
  }
}

// process.rs:31-55; the distribution arrives as the library's sparse form: cells without ecDNA in the descriptor,
// the occupied copy numbers k_min .. k_min + k_len - 1 in the arena
void save(const Cli& c, const std::string& filename, const ecdna_b200_dist_t& d, const uint32_t* arena, int verbosity) {
  const uint64_t cells = d.cells;
  const float time = d.time;
  char tbuf[64];
  std::snprintf(tbuf, sizeof tbuf, "%.1f", (double)time);
  std::string tp;
  for (const char* p = tbuf; *p; ++p) { if (*p == '.') tp += "dot"; else tp.push_back(*p); }
  tp += "years";
  const std::string dir = c.path + "/" + std::to_string(cells) + "cells/ecdna/" + tp;
  mkdirs(dir);
  const std::string file = dir + "/" + filename + ".json";
  if (verbosity > 0) std::printf("saving state at time %s with %llu cells in \"%s\"\n", rust_f32_to_string(time).c_str(), (unsigned long long)cells, file.c_str());
  std::ofstream f(file);
  if (!f) { std::fprintf(stderr, "Cannot create %s\n", file.c_str()); std::exit(101); }
  f << "{";
  bool first = true;
  if (d.nminus) { f << "\"0\":" << d.nminus; first = false; }
  const uint32_t* bins = arena + d.offset;
  for (uint32_t i = 0; i < d.k_len; ++i) {
    if (!bins[i]) continue;
    if (!first) f << ",";
    f << "\"" << (d.k_min + i) << "\":" << bins[i];
    first = false;
  }
  f << "}";
}

// same directory scheme as `save`, with the measurement name in place of "ecdna"
std::string measurement_path(const Cli& c, uint64_t cells, float time, const char* what, const std::string& filename) {
  char tbuf[64];
  std::snprintf(tbuf, sizeof tbuf, "%.1f", (double)time);
  std::string tp;
  for (const char* p = tbuf; *p; ++p) { if (*p == '.') tp += "dot"; else tp.push_back(*p); }
  const std::string dir = c.path + "/" + std::to_string(cells) + "cells/" + what + "/" + tp + "years";
  mkdirs(dir);
  return dir + "/" + filename + ".json";
}

// {"0": 2, "1": 2, "10": 1} (dynamics.md:7-8)
std::map<uint32_t, uint64_t> load_json_hist(const std::string& path) {
  std::ifstream f(path);
  if (!f) die("Cannot load the ecDNA distribution from \"" + path + "\"");
  std::string s((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::map<uint32_t, uint64_t> out;
  size_t i = 0;
  while ((i = s.find('"', i)) != std::string::npos) {
    const size_t j = s.find('"', i + 1);
    if (j == std::string::npos) break;
    const unsigned long k = std::strtoul(s.substr(i + 1, j - i - 1).c_str(), nullptr, 10);
    const size_t colon = s.find(':', j);
    if (colon == std::string::npos) break;
    const unsigned long long cnt = std::strtoull(s.c_str() + colon + 1, nullptr, 10);
    if (k > 65535) die("copy number does not fit u16 in " + path);
    out[(uint32_t)k] += cnt;
    i = colon + 1;
  }
  if (out.empty()) die("empty distribution in " + path);
  return out;
}

std::string utc_now() {
  using namespace std::chrono;
  const auto now = system_clock::now();
  const std::time_t t = system_clock::to_time_t(now);
  const auto ns = duration_cast<nanoseconds>(now.time_since_epoch()).count() % 1000000000ll;
  char buf[64];
  std::tm tm{};
  gmtime_r(&t, &tm);
  std::strftime(buf, sizeof buf, "%Y-%m-%d %H:%M:%S", &tm);
  char out[96];
  std::snprintf(out, sizeof out, "%s.%09lld UTC", buf, (long long)ns);
  return out;
}

const char* kStopNames[] = {"NoIndividualsLeft", "MaxItersReached", "MaxTimeReached", "MaxIndividualsReached",
                            "AbsorbingStateReached", "CopyNumberOverflow", "HistogramOverflow", "ReplayExhausted",
                            "ReplayInconsistent"};

// `ecdna abc`: the removed ABC binary of the reference (abc.md:10-55).  One run per prior draw over
// (f1 = b1, d2 = d0, d1), the four distances to the target distribution from the kernel's fused epilogue, and
// abc.csv with EVERY draw ("save all, filter later", abc.md:57-71) in the column order of abc.md:38-55;
// abc_accepted.csv holds the draws within the thresholds.
int run_abc(const Cli& c, ecdna_b200_multi* gpus, ecdna_b200_params_t p, uint64_t idx_begin, uint64_t draws,
            const std::map<uint32_t, uint64_t>& init) {
  const std::map<uint32_t, uint64_t> tgt = load_json_hist(c.target);
  std::vector<uint64_t> target((size_t)tgt.rbegin()->first + 1, 0);
  for (auto& kv : tgt) target[kv.first] = kv.second;
  uint64_t init_cells = 0, init_copies = 0;
  for (auto& kv : init) { init_cells += kv.second; init_copies += (uint64_t)kv.first * kv.second; }
  const double init_mean = init_cells ? (double)init_copies / (double)init_cells : 0.0;
  p.abc_enabled = 1;
  p.abc_target_hist = target.data();
  p.abc_target_len = (uint32_t)target.size();
  for (int j = 0; j < 4; ++j) p.abc_thresholds[j] = c.thresholds[j];
  p.hist_stride = 64;  // (the distributions themselves are not written)
  mkdirs(c.path);
  std::ofstream all(c.path + "/abc.csv"), acc(c.path + "/abc_accepted.csv");
  if (!all || !acc) { std::fprintf(stderr, "Cannot create %s/abc.csv\n", c.path.c_str()); return 101; }
  const char* header = "parental_idx,idx,timepoint,seed,ecdna,mean,entropy,f1,f2,d1,d2,cells,tumour_cells,init_mean,init_cells,init_copies\n";
  all << header;
  acc << header;
  ecdna_b200_ctx* prior_ctx = nullptr;  // prior draws: Philox keyed (seed, draw index), on the first GPU
  if (ecdna_b200_create(c.devices.empty() ? 0 : c.devices[0], &prior_ctx) != ECDNA_B200_OK) return 101;
  const uint64_t chunk = c.chunk ? c.chunk : 262144ull * (uint64_t)ecdna_b200_multi_device_count(gpus);
  uint64_t n_acc = 0;
  for (uint64_t first = 0; first < draws; first += chunk) {
    const uint64_t n = std::min<uint64_t>(chunk, draws - first);
    std::vector<float> rates(n * 4), dist(n * 4);
    std::vector<uint8_t> accept(n);
    std::vector<uint64_t> nminus(n), nplus(n);
    std::vector<uint32_t> stop(n);
    int rc = ecdna_b200_abc_draw_priors(prior_ctx, c.seed, idx_begin + first, n, c.b0, c.b1_range, c.d0_range, c.d1_range, rates.data());
    if (rc != ECDNA_B200_OK) { std::fprintf(stderr, "prior draws: %s\n", ecdna_b200_last_error(prior_ctx)); return 101; }
    p.rates_per_run = rates.data();
    ecdna_b200_results_t r;
    std::memset(&r, 0, sizeof r);
    r.stop_reason = stop.data(); r.nminus = nminus.data(); r.nplus = nplus.data();
    r.abc_distance = dist.data(); r.abc_accept = accept.data();
    rc = ecdna_b200_multi_run(gpus, &p, idx_begin + first, n, &r);
    if (rc != ECDNA_B200_OK) { std::fprintf(stderr, "ecdna_b200_multi_run: %s\n", ecdna_b200_multi_last_error(gpus)); return 101; }
    char line[512];
    for (uint64_t i = 0; i < n; ++i) {
      const unsigned long long tumour = nminus[i] + nplus[i];
      // abc.md:44-52: f1/d1 belong to the cells WITH ecDNA, f2/d2 to the cells without
      std::snprintf(line, sizeof line, ",%llu,0,%llu,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%.9g,%llu,%llu,%.9g,%llu,%llu\n",
                    (unsigned long long)(idx_begin + first + i), (unsigned long long)c.seed, (double)dist[4 * i], (double)dist[4 * i + 1],
                    (double)dist[4 * i + 2], (double)rates[4 * i + 1], (double)rates[4 * i], (double)rates[4 * i + 3],
                    (double)rates[4 * i + 2], tumour, tumour, init_mean, (unsigned long long)init_cells, (unsigned long long)init_copies);
      all << line;
      if (accept[i]) { acc << line; ++n_acc; }
    }
  }
  ecdna_b200_destroy(prior_ctx);
  std::printf("%llu of %llu draws within the thresholds\n", (unsigned long long)n_acc, (unsigned long long)draws);
  return 0;
}

std::string g9(double v) {  // %.9g (round-trips f32); JSON spells infinity as Python's json module does
  char buf[64];
  std::snprintf(buf, sizeof buf, "%.9g", v);
  return buf;
}
std::string g17(double v) {
  char buf[64];
  std::snprintf(buf, sizeof buf, "%.17g", v);
  return buf;
}
std::string json_num(const std::string& s) { return s == "inf" ? "Infinity" : (s == "-inf" ? "-Infinity" : s); }

// `ecdna abc --generations G`: ABC-SMC over the GPUs of `gpus` (ecdna_b200_abc_smc_ex); <DIR>/abc_gen<t>.csv holds
// population t in the columns of abc.csv (parental_idx = idx of the perturbed particle) plus generation, epsilon,
// weight, and <DIR>/abc_smc.json the schedule.  Byte for byte what write_abc_smc (abc.py) writes for the same run.
int run_abc_smc(const Cli& c, ecdna_b200_multi* gpus, ecdna_b200_params_t p, uint64_t idx_begin,
                const std::map<uint32_t, uint64_t>& init) {
  const std::map<uint32_t, uint64_t> tgt = load_json_hist(c.target);
  std::vector<uint64_t> target((size_t)tgt.rbegin()->first + 1, 0);
  for (auto& kv : tgt) target[kv.first] = kv.second;
  uint64_t init_cells = 0, init_copies = 0;
  for (auto& kv : init) { init_cells += kv.second; init_copies += (uint64_t)kv.first * kv.second; }
  const double init_mean = init_cells ? (double)init_copies / (double)init_cells : 0.0;
  p.abc_enabled = 1;
  p.abc_target_hist = target.data();
  p.abc_target_len = (uint32_t)target.size();
  for (int j = 0; j < 4; ++j) p.abc_thresholds[j] = c.thresholds[j];
  ecdna_b200_smc_options_t o;
  std::memset(&o, 0, sizeof o);
  o.population = c.population; o.quantile = c.quantile; o.max_generations = c.generations;
  o.max_simulations = c.max_simulations; o.idx_begin = idx_begin; o.chunk = c.chunk;
  for (int j = 0; j < 2; ++j) { o.b1_range[j] = c.b1_range[j]; o.d0_range[j] = c.d0_range[j]; o.d1_range[j] = c.d1_range[j]; }
  const size_t G = c.generations, M = c.population;
  std::vector<uint64_t> idx(G * M), parent(G * M), cells(G * M), consumed(G), simulated(G);
  std::vector<float> rates(G * M * 4), dist(G * M * 4), eps(G);
  std::vector<double> weight(G * M), ess(G);
  ecdna_b200_smc_result_t r;
  std::memset(&r, 0, sizeof r);
  r.idx = idx.data(); r.parent_idx = parent.data(); r.rates = rates.data(); r.distance = dist.data();
  r.weight = weight.data(); r.cells = cells.data(); r.epsilon = eps.data(); r.consumed = consumed.data();
  r.simulated = simulated.data(); r.ess = ess.data();
  ecdna_b200_smc_kernel_t kernel;
  std::memset(&kernel, 0, sizeof kernel);
  kernel.kernel = c.smc_kernel;
  std::vector<uint32_t> used(G);
  const int rc = ecdna_b200_abc_smc_ex(gpus, &p, &o, &kernel, &r, used.data());
  if (rc != ECDNA_B200_OK) { std::fprintf(stderr, "ecdna_b200_abc_smc_ex: %s\n", ecdna_b200_multi_last_error(gpus)); return 101; }
  mkdirs(c.path);
  for (uint32_t t = 0; t < r.generations; ++t) {
    const std::string file = c.path + "/abc_gen" + std::to_string(t) + ".csv";
    std::ofstream f(file);
    if (!f) { std::fprintf(stderr, "Cannot create %s\n", file.c_str()); return 101; }
    f << "parental_idx,idx,timepoint,seed,ecdna,mean,entropy,f1,f2,d1,d2,cells,tumour_cells,init_mean,init_cells,init_copies,"
         "generation,epsilon,weight\n";
    const std::string e = g9(eps[t]);
    for (size_t i = t * M; i < (t + 1) * M; ++i) {
      const float* x = &rates[4 * i];
      const float* d = &dist[4 * i];
      // abc.md:44-52: f1/d1 belong to the cells WITH ecDNA, f2/d2 to the cells without
      if (t > 0) f << parent[i];
      f << "," << idx[i] << ",0," << c.seed << "," << g9(d[0]) << "," << g9(d[1]) << "," << g9(d[2]) << "," << g9(x[1]) << ","
        << g9(x[0]) << "," << g9(x[3]) << "," << g9(x[2]) << "," << cells[i] << "," << cells[i] << "," << g9(init_mean) << ","
        << init_cells << "," << init_copies << "," << t << "," << e << "," << g17(weight[i]) << "\n";
    }
  }
  const char* status[] = {"reached", "max_generations", "budget"};
  std::ofstream js(c.path + "/abc_smc.json");
  if (!js) { std::fprintf(stderr, "Cannot create %s/abc_smc.json\n", c.path.c_str()); return 101; }
  auto list = [&](auto n, auto fmt) {
    std::string out = "[";
    for (uint32_t t = 0; t < n; ++t) out += (t ? "," : "") + fmt(t);
    return out + "]";
  };
  const uint32_t n = r.generations;
  auto pair = [&](const float* v) { return "[" + g9(v[0]) + "," + g9(v[1]) + "]"; };
  js << "{\"status\":\"" << status[r.status > 2 ? 2 : r.status] << "\",\"generations\":" << n
     << ",\"epsilon\":" << list(n, [&](uint32_t t) { return json_num(g9(eps[t])); })
     << ",\"consumed\":" << list(n, [&](uint32_t t) { return std::to_string(consumed[t]); })
     << ",\"simulated\":" << list(n, [&](uint32_t t) { return std::to_string(simulated[t]); })
     << ",\"ess\":" << list(n, [&](uint32_t t) { return json_num(g17(ess[t])); });
  const char* kernels[] = {"component", "mvn", "olcm"};
  if (c.smc_kernel != ECDNA_B200_SMC_KERNEL_COMPONENT)  // (the component kernel's files stay those of a run without it)
    js << ",\"kernel\":\"" << kernels[c.smc_kernel] << "\",\"kernel_used\":" << list(n, [&](uint32_t t) {
      return used[t] > 2 ? std::string("null") : "\"" + std::string(kernels[used[t]]) + "\"";
    });
  js << ",\"options\":{\"seed\":" << c.seed << ",\"idx_begin\":" << idx_begin << ",\"population\":" << c.population
     << ",\"quantile\":" << g17(c.quantile) << ",\"max_generations\":" << c.generations
     << ",\"max_simulations\":" << c.max_simulations << ",\"b1_range\":" << pair(c.b1_range)
     << ",\"d0_range\":" << pair(c.d0_range) << ",\"d1_range\":" << pair(c.d1_range) << ",\"thresholds\":"
     << list(4u, [&](uint32_t j) { return json_num(g9(c.thresholds[j])); }) << "}}\n";
  uint64_t total = 0;
  for (uint32_t t = 0; t < n; ++t) total += simulated[t];
  std::printf("%u generations (%s), %llu draws simulated, final tolerance factor %s\n", n, status[r.status > 2 ? 2 : r.status],
              (unsigned long long)total, n ? g9(eps[n - 1]).c_str() : "-");
  return 0;
}

}  // namespace

int main(int argc, char** argv) {
  Cli c = parse(argc, argv);
  if (c.growth == "constant") { std::fprintf(stderr, "not yet implemented\n"); return 101; }  // todo!(), main.rs:49
  if (c.growth != "exponential") die("invalid value '" + c.growth + "' for '--growth <GROWTH>'");
  uint32_t seg;
  if (c.segregation == "deterministic") seg = ECDNA_B200_SEG_DETERMINISTIC;
  else if (c.segregation == "binomial-no-uneven") seg = ECDNA_B200_SEG_BINOMIAL_NO_UNEVEN;
  else if (c.segregation == "binomial") seg = ECDNA_B200_SEG_BINOMIAL;
  else if (c.segregation == "binomial-no-nminus") seg = ECDNA_B200_SEG_BINOMIAL_NO_NMINUS;
  else die("invalid value '" + c.segregation + "' for '--segregation <SEGREGATION>'");

  // clap_app.rs:140-157
  uint64_t cells, years, runs;
  int verbosity;
  if (c.debug) { cells = 300; years = 2; verbosity = 255; runs = 1; }
  else if (c.has_years) { cells = kMaxCells; years = c.years; verbosity = c.verbosity; runs = c.runs; }
  else {
    cells = c.has_cells ? c.cells : 1000;
    years = (uint64_t)(log2f((float)cells) + 4.f);
    verbosity = c.verbosity;
    runs = c.runs;
  }
  // clap_app.rs:102-134
  std::vector<uint64_t> snapshots;
  if (c.has_snapshots) snapshots = c.snapshots;
  else {
    const uint64_t dx = cells / 10;
    snapshots.assign(11, 1);
    for (int i = 1; i < 10; ++i) snapshots[i] = snapshots[i - 1] + dx;
    snapshots[10] = cells;
  }
  std::sort(snapshots.begin(), snapshots.end());
  // clap_app.rs:165-174
  const float d0 = c.has_d0 ? c.d0 : 0.f, d1 = c.has_d1 ? c.d1 : 0.f;
  const bool birth_death = (c.has_d0 && c.d0 > 0.f) || (c.has_d1 && c.d1 > 0.f);
  // clap_app.rs:177-192
  std::map<uint32_t, uint64_t> init;
  if (!c.initial.empty()) init = load_json_hist(c.initial);
  else init[1] = 1;
  std::vector<uint16_t> init_k;
  std::vector<uint64_t> init_c;
  for (auto& kv : init) { init_k.push_back((uint16_t)kv.first); init_c.push_back(kv.second); }

  std::printf("%s Starting the simulation\n", utc_now().c_str());  // main.rs:53

  ecdna_b200_multi* gpus = nullptr;
  int rc = ecdna_b200_multi_create(c.devices.empty() ? nullptr : c.devices.data(), (int)c.devices.size(), &gpus);
  if (rc != ECDNA_B200_OK) {
    std::fprintf(stderr, "ecdna_b200_multi_create failed with status %d (no B200 visible? this backend has no CPU path)\n", rc);
    return 101;
  }
  const int n_gpus = ecdna_b200_multi_device_count(gpus);
  ecdna_b200_params_t p;
  std::memset(&p, 0, sizeof p);
  p.abi_version = ECDNA_B200_ABI_VERSION;
  p.b0 = c.b0; p.b1 = c.b1; p.d0 = d0; p.d1 = d1;
  p.segregation = seg;
  p.max_cells = cells; p.max_iter = kMaxIter; p.max_time = (float)years;  // clap_app.rs:204-209
  p.seed = c.seed;
  p.bd_count_mode = c.bd_count_mode;
  p.n_init = (uint32_t)init_k.size(); p.init_k = init_k.data(); p.init_c = init_c.data();
  p.tile_width = c.tile_width; p.state_mode = c.state_mode;
  const uint64_t idx_begin = c.seed * 10;  // main.rs:214
  if (c.abc) {
    const int arc = c.generations ? run_abc_smc(c, gpus, p, idx_begin, init) : run_abc(c, gpus, p, idx_begin, runs, init);
    ecdna_b200_multi_destroy(gpus);
    if (arc == 0) std::printf("%s End simulation\n", utc_now().c_str());
    return arc;
  }
  p.n_snapshots = (uint32_t)snapshots.size(); p.snapshot_cells = snapshots.empty() ? nullptr : snapshots.data();
  if (c.has_subsamples && !c.subsamples.empty()) {  // main.rs:110-123, drawn on the device
    p.n_subsamples = (uint32_t)c.subsamples.size();
    p.subsample_cells = c.subsamples.data();
  }
  const uint32_t dyn_points = c.dynamics ? 300u : 0u;  // CHANGELOG.md:34-36
  p.dyn_points = dyn_points;
  p.dyn_dt = 0.1f;

  // The index range goes through the library in chunks (host memory is O(chunk), whatever --runs is); the
  // files of a chunk are written while the next chunk is simulated.
  uint32_t stride = 1024;  // bins per distribution ON THE DEVICE; the host receives the occupied windows only
  const size_t n_snap = snapshots.size();
  const size_t n_dist = 1 + n_snap + p.n_subsamples;  // distributions per replicate
  auto per_replicate_bytes = [&](uint32_t st) { return n_dist * st * 4 + (size_t)dyn_points * 20 + 64; };
  uint64_t chunk = c.chunk ? c.chunk : std::max<uint64_t>(1024, std::min<uint64_t>(262144, (8ull << 30) / per_replicate_bytes(stride))) * (uint64_t)n_gpus;
  struct Buffers {
    std::vector<uint32_t> stop, kmax, dyn_count, arena;
    std::vector<ecdna_b200_dist_t> final_dist, snap_dist, sub_dist;
    std::vector<uint64_t> nminus, nplus;
    std::vector<float> time, mean, freq, entropy, dyn;
    uint64_t first = 0, n = 0;
  } buf[2];
  auto simulate = [&](Buffers& b, uint64_t first, uint64_t n) -> int {
    b.first = first; b.n = n;
    b.stop.assign(n, 0); b.kmax.assign(n, 0); b.dyn_count.assign(n, 0);
    b.nminus.assign(n, 0); b.nplus.assign(n, 0); b.time.assign(n, 0.f);
    b.mean.assign(n, 0.f); b.freq.assign(n, 0.f); b.entropy.assign(n, 0.f); b.dyn.assign((size_t)n * dyn_points * 5, 0.f);
    b.final_dist.assign(n, ecdna_b200_dist_t{}); b.snap_dist.assign(n * n_snap, ecdna_b200_dist_t{});
    b.sub_dist.assign(n * p.n_subsamples, ecdna_b200_dist_t{});
    for (int attempt = 0; attempt < 2; ++attempt) {
      p.hist_stride = stride;
      ecdna_b200_results_t r;
      std::memset(&r, 0, sizeof r);
      r.stop_reason = b.stop.data(); r.nminus = b.nminus.data(); r.nplus = b.nplus.data(); r.time = b.time.data();
      r.kmax = b.kmax.data();
      if (c.summaries) { r.mean = b.mean.data(); r.frequency = b.freq.data(); r.entropy = b.entropy.data(); }
      if (c.dynamics) { r.dyn = b.dyn.data(); r.dyn_count = b.dyn_count.data(); }
      ecdna_b200_sparse_t sp;
      std::memset(&sp, 0, sizeof sp);
      sp.final_dist = b.final_dist.data();
      if (n_snap) sp.snap_dist = b.snap_dist.data();
      if (p.n_subsamples) sp.sub_dist = b.sub_dist.data();
      sp.arena = b.arena.data(); sp.arena_words = b.arena.size();
      int rc2 = ecdna_b200_multi_run_sparse(gpus, &p, idx_begin + first, n, &r, &sp);
      if (rc2 == ECDNA_B200_ERR_ARENA) {  // the two-call pattern: the packed chunk waits on the devices for a larger arena
        b.arena.resize(sp.arena_used + sp.arena_used / 4);
        sp.arena = b.arena.data(); sp.arena_words = b.arena.size();
        rc2 = ecdna_b200_multi_sparse_fetch(gpus, &sp);
      }
      if (rc2 != ECDNA_B200_OK) { std::fprintf(stderr, "ecdna_b200_multi_run_sparse: %s\n", ecdna_b200_multi_last_error(gpus)); return 101; }
      uint32_t top = 0;
      for (uint64_t i = 0; i < n; ++i) top = std::max(top, b.kmax[i]);
      if (top < stride) break;
      stride = ((top + 1 + 1023) / 1024) * 1024;  // histograms were truncated: run again with room for them
    }
    return 0;
  };
  auto write_files = [&](const Buffers& b) -> int {
    for (uint64_t i = 0; i < b.n; ++i) {
      const uint64_t idx = idx_begin + b.first + i;
      const std::string filename = make_filename(c, birth_death, d0, d1, idx);
      const uint32_t code = b.stop[i] & 0xFFu;
      if (code == ECDNA_B200_STOP_COPY_OVERFLOW) {  // proliferation.rs:63-67 panics: the reference aborts here
        std::fprintf(stderr, "Overflow while segregating DNA into two daughter cells (idx %llu)\n", (unsigned long long)idx);
        return 101;
      }
      for (size_t sidx = 0; sidx < n_snap; ++sidx) {
        const ecdna_b200_dist_t& d = b.snap_dist[(size_t)i * n_snap + sidx];
        if (!(d.flags & ECDNA_B200_DIST_TAKEN)) break;  // (sizes ascend: the first one not reached ends the list)
        if (verbosity > 0) std::printf("saving state for timepoint at time %s with cells %llu \n", rust_f32_to_string(d.time).c_str(), (unsigned long long)d.cells);
        save(c, filename, d, b.arena.data(), verbosity);
      }
      save(c, filename, b.final_dist[i], b.arena.data(), verbosity);  // main.rs:100-109
      if (c.summaries) {
        const uint64_t cells_now = b.nminus[i] + b.nplus[i];
        const std::pair<const char*, float> m[] = {{"mean", b.mean[i]}, {"frequency", b.freq[i]}, {"entropy", b.entropy[i]}};
        for (auto& kv : m) {
          std::ofstream f(measurement_path(c, cells_now, b.time[i], kv.first, filename));
          f << rust_f32_to_string(kv.second);
        }
      }
      if (c.dynamics) {
        std::ofstream f(measurement_path(c, b.nminus[i] + b.nplus[i], b.time[i], "dynamics", filename));
        const char* names[5] = {"nminus", "nplus", "mean", "variance", "entropy"};
        f << "{\"dt\":0.1";
        for (int q = 0; q < 5; ++q) {
          f << ",\"" << names[q] << "\":[";
          for (uint32_t j = 0; j < b.dyn_count[i]; ++j) {
            if (j) f << ",";
            f << rust_f32_to_string(b.dyn[((size_t)i * dyn_points + j) * 5 + q]);
          }
          f << "]";
        }
        f << "}";
      }
      for (uint32_t j = 0; j < p.n_subsamples; ++j)  // main.rs:110-123: one file per --subsamples size
        save(c, filename, b.sub_dist[(size_t)i * p.n_subsamples + j], b.arena.data(), verbosity);
      if (verbosity > 0)  // main.rs:205-210
        std::printf("stop reason: %s\nnminus, nplus: [\n    %llu,\n    %llu,\n]\ntime: %s\n", kStopNames[code > 8 ? 8 : code],
                    (unsigned long long)b.nminus[i], (unsigned long long)b.nplus[i], rust_f32_to_string(b.time[i]).c_str());
    }
    return 0;
  };
  int status = 0, cur = 0;
  std::future<int> writer;
  for (uint64_t first = 0; first < runs && status == 0; first += chunk, cur ^= 1) {
    status = simulate(buf[cur], first, std::min<uint64_t>(chunk, runs - first));
    if (writer.valid()) { const int w = writer.get(); if (status == 0) status = w; }
    if (status == 0) writer = std::async(std::launch::async, write_files, std::cref(buf[cur]));
  }
  if (writer.valid()) { const int w = writer.get(); if (status == 0) status = w; }
  ecdna_b200_multi_destroy(gpus);
  if (status) return status;
  std::printf("%s End simulation\n", utc_now().c_str());  // main.rs:226
  return 0;
}
