// sb_cli.cc -- `sigmap` command-line driver on top of the C ABI: the drop-in for the
// reference's `sigmap -i` / `sigmap -m` (flags of sigmap.cc:1331-1377, same files in and
// out).  Host-side only: parses flags, reads FASTA / .pt / BLOW5, calls smb_map_reads, writes
// the modified PAF.  Extra flags: --gpu N (device ordinal), or --gpus LIST (several devices,
// one context and one host thread each) with --shard reads (each device maps its own slice of
// the reads against a full copy of the index; default) or --shard contigs (the index is
// partitioned by contig, every device maps every read, chains merged by the library's
// collectives -- for references whose index exceeds one GPU).  `-t` is accepted for
// compatibility (the GPU path does not use host mapping threads).
//
// `-i` writes <prefix>.pt and <prefix>.si (a KD-tree in nanoflann's layout, for the reference's own
// `sigmap -m`; this program never reads it: the device index is rebuilt from the point cloud at
// load time).  The point cloud is built on the host, or on device N with an explicit --gpu N; the
// files are the same byte for byte.  `-m --index-from-ref` builds the device index(es) from -r on
// the devices instead of reading -x (with --shard contigs every device builds only its own part):
// the way to map against a reference whose point cloud would not fit in host memory.
// Difference kept on purpose and documented in DESIGN.md: FAST5 input is not supported (BLOW5 only).
#include <dirent.h>
#include <sys/stat.h>
#include <sys/time.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sigmap_b200.h"

namespace {

double now() {
  struct timeval tp;
  gettimeofday(&tp, nullptr);
  return tp.tv_sec + tp.tv_usec * 1e-6;
}

[[noreturn]] void die(const std::string &msg) {  // ExitWithMessage, utils.h:67
  fprintf(stderr, "%s\n", msg.c_str());
  exit(-1);
}

bool is_dir(const std::string &p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}

void collect_blow5(const std::string &dir, std::vector<std::string> &out, int depth = 0) {
  DIR *d = opendir(dir.c_str());
  if (!d) return;
  std::vector<std::string> names;
  while (struct dirent *e = readdir(d)) names.push_back(e->d_name);
  closedir(d);
  std::sort(names.begin(), names.end());
  for (const std::string &n : names) {
    if (n == "." || n == "..") continue;
    const std::string p = dir + "/" + n;
    if (is_dir(p)) {
      if (depth < 1) collect_blow5(p, out, depth + 1);  // signal_batch.cc:36-47: one level down
    } else if (p.find(".blow5") != std::string::npos) {
      out.push_back(p);
    } else if (p.find(".fast5") != std::string::npos) {
      fprintf(stderr, "warning: FAST5 input is not supported by this build, skipping %s\n", p.c_str());
    }
  }
}

struct Args {
  bool index = false, map = false, help = false;
  std::string ref, model, ref_index, sig_dir, output;
  int dimension = 6, max_leaf = 20, threads = 1, gpu = 0;
  bool gpu_given = false;       // --gpu N given: `-i` builds the point cloud on device N
  bool index_from_ref = false;  // --index-from-ref: `-m` builds the index from -r, no -x
  std::vector<int> gpus;       // --gpus 0,1,2,...: empty = the single device --gpu
  bool shard_contigs = false;  // --shard contigs
  smb_params prm;
};

const char *kHelp =
    "Map ONT raw signal data (B200 build)\nUsage:\n  sigmap [OPTION...]\n\n"
    " Indexing options:\n  -i, --build-index      Build spatial index for reference\n"
    "  -d, --dimension INT    Dimension of spatial index [6]\n"
    "  -l, --max-leaf INT     Max leaf of spatial index [20]\n\n"
    " Mapping options:\n  -m, --map              Map signal data\n"
    "      --step-size INT    Seeding step size in reads [2]\n"
    "  -t, --num-threads INT  # threads for mapping [1] (accepted, unused on GPU)\n"
    "      --gpu INT          CUDA device ordinal [0]; with -i: build the point cloud on it\n"
    "      --gpus LIST        several devices, e.g. 0,1,2,3 (one context per entry)\n"
    "      --shard MODE       with --gpus: reads (split the reads, index replicated; default)\n"
    "                         or contigs (split the index by contig, chains merged)\n\n"
    " Input options:\n  -r, --ref FILE         Reference file\n  -p, --pore-model FILE  Pore model file\n"
    "  -x, --ref-index FILE   Reference index file\n"
    "      --index-from-ref   with -m: build the index on the device(s) from -r instead of -x\n  -s, --sig-dir DIR      Signal data directory\n\n"
    " Output options:\n  -o, --output arg       Output file\n\n"
    " Development options:\n      --search-radius FLT            Search radius for each seed [0.08]\n"
    "      --max-num-chunks INT           Max # chunks before stop trying to map a read [30]\n"
    "      --min-num-anchors INT          Min # anchors to stop mapping [10]\n"
    "      --min-num-anchors-output INT   Min # anchors to output mappings [10]\n"
    "      --stop-mapping FLOAT           best/second-best chaining score to stop mapping [1.4]\n"
    "      --stop-mapping-output FLOAT    best/second-best chaining score to output mappings [1.2]\n"
    "      --stop-mapping-mean FLOAT      best/mean chaining score to stop mapping [5]\n"
    "      --stop-mapping-mean-output FLOAT best/mean chaining score to output mappings [5]\n"
    "  -h, --help                         Print help\n";

Args parse(int argc, char **argv) {
  Args a;
  smb_default_params(&a.prm);
  auto need = [&](int &i) -> const char * {
    if (i + 1 >= argc) die(std::string("Option ") + argv[i] + " is missing an argument");
    return argv[++i];
  };
  for (int i = 1; i < argc; ++i) {
    std::string o = argv[i], v;
    size_t eq = o.find('=');
    bool has_v = false;
    if (o.rfind("--", 0) == 0 && eq != std::string::npos) {
      v = o.substr(eq + 1);
      o = o.substr(0, eq);
      has_v = true;
    }
    auto val = [&]() -> std::string { return has_v ? v : std::string(need(i)); };
    if (o == "-i" || o == "--build-index") a.index = true;
    else if (o == "-m" || o == "--map") a.map = true;
    else if (o == "-h" || o == "--help") a.help = true;
    else if (o == "-d" || o == "--dimension") a.dimension = atoi(val().c_str());
    else if (o == "-l" || o == "--max-leaf") a.max_leaf = atoi(val().c_str());
    else if (o == "-t" || o == "--num-threads") a.threads = atoi(val().c_str());
    else if (o == "--gpu") {
      a.gpu = atoi(val().c_str());
      a.gpu_given = true;
    } else if (o == "--index-from-ref") a.index_from_ref = true;
    else if (o == "--gpus") {
      const std::string list = val();
      for (size_t at = 0; at <= list.size();) {
        size_t comma = list.find(',', at);
        if (comma == std::string::npos) comma = list.size();
        if (comma > at) a.gpus.push_back(atoi(list.substr(at, comma - at).c_str()));
        at = comma + 1;
      }
      if (a.gpus.empty()) die("--gpus needs a list of device ordinals");
    } else if (o == "--shard") {
      const std::string m = val();
      if (m == "contigs") a.shard_contigs = true;
      else if (m != "reads") die("--shard must be reads or contigs");
    }
    else if (o == "-r" || o == "--ref") a.ref = val();
    else if (o == "-p" || o == "--pore-model") a.model = val();
    else if (o == "-x" || o == "--ref-index") a.ref_index = val();
    else if (o == "-s" || o == "--sig-dir") a.sig_dir = val();
    else if (o == "-o" || o == "--output") a.output = val();
    else if (o == "--step-size") a.prm.step_size = atoi(val().c_str());
    else if (o == "--search-radius") a.prm.search_radius = (float)atof(val().c_str());
    else if (o == "--max-num-chunks") a.prm.max_num_chunks = atoi(val().c_str());
    else if (o == "--min-num-anchors") a.prm.min_num_anchors = atoi(val().c_str());
    else if (o == "--min-num-anchors-output") a.prm.min_num_anchors_output = atoi(val().c_str());
    else if (o == "--stop-mapping") a.prm.stop_mapping = (float)atof(val().c_str());
    else if (o == "--stop-mapping-output") a.prm.stop_mapping_output = (float)atof(val().c_str());
    else if (o == "--stop-mapping-mean") a.prm.stop_mapping_mean = (float)atof(val().c_str());
    else if (o == "--stop-mapping-mean-output") a.prm.stop_mapping_mean_output = (float)atof(val().c_str());
    else die("Option '" + o + "' does not exist");
  }
  return a;
}

int build_index(const Args &a) {
  if (a.ref.empty()) die("No reference file specified!");
  if (a.model.empty()) die("No pore model file specified!");
  if (a.output.empty()) die("No output file specified!");
  if (a.dimension != SMB_DIM) die("Only dimension 6 is supported by this build");
  fprintf(stderr, "Dimension: %d, max leaf: %d\nReference file: %s\nPore model file: %s\nOutput file: %s\n",
          a.dimension, a.max_leaf, a.ref.c_str(), a.model.c_str(), a.output.c_str());
  double t0 = now();
  std::vector<float> mean(4096), stdv(4096);
  if (smbh_pore_model_load(a.model.c_str(), mean.data(), stdv.data())) die("Cannot load pore model!");
  smbh_fasta fa;
  if (smbh_fasta_load(a.ref.c_str(), &fa)) die("Cannot find sequence file!");
  uint64_t *pos = nullptr;
  float *val = nullptr;
  size_t n = 0;
  if (a.gpu_given) {
    smb_ctx *ctx = nullptr;
    if (smb_create(&ctx, a.gpu)) die(std::string("smb_create: ") + smb_last_error(nullptr));
    if (smb_point_cloud_build(ctx, fa.seqs, fa.lengths, fa.n, mean.data(), &pos, &val, &n))
      die(std::string("smb_point_cloud_build: ") + smb_last_error(ctx));
    smb_destroy(ctx);
  } else if (smbh_build_point_cloud_alloc(fa.seqs, fa.lengths, fa.n, mean.data(), &pos, &val, &n)) {
    die("Out of memory while collecting points!");
  }
  fprintf(stderr, "Collected %zu points.\n", n);
  if (smbh_pt_write(a.output.c_str(), pos, val, n, a.dimension, a.max_leaf))
    die("Cannot write index file!");
  // <prefix>.si: not read by this program (the flat device index is built from .pt); written so
  // that the reference's own `sigmap -m` can use the index
  if (smbh_si_write(a.output.c_str(), val, n, a.dimension, a.max_leaf))
    die("Cannot write index file!");
  smbh_free(pos);
  smbh_free(val);
  smbh_fasta_free(&fa);
  fprintf(stderr, "Built index successfully in %fs.\n", now() - t0);
  return 0;
}

int map_reads(const Args &a) {
  fprintf(stderr, "Number of threads: %d\n", a.threads);
  if (a.ref.empty()) die("No reference file specified!");
  if (a.model.empty()) die("No pore model file specified!");
  if (a.ref_index.empty() && !a.index_from_ref) die("No reference index file specified!");
  if (a.sig_dir.empty()) die("No signal data directory specified!");
  if (a.output.empty()) die("No output file specified!");
  fprintf(stderr, "Reference file: %s\nPore model file: %s\nReference index file: %s\nSignal directory: %s\nOutput file: %s\n",
          a.ref.c_str(), a.model.c_str(), a.index_from_ref ? "(built from the reference)" : a.ref_index.c_str(),
          a.sig_dir.c_str(), a.output.c_str());
  std::vector<float> level_mean(4096), level_stdv(4096);
  if (a.index_from_ref && smbh_pore_model_load(a.model.c_str(), level_mean.data(), level_stdv.data()))
    die("Cannot load pore model!");
  if (!is_dir(a.sig_dir)) die("Signal directory is in valid!");
  double t0 = now();
  std::vector<std::string> files;
  collect_blow5(a.sig_dir, files);
  smbh_reads reads;
  memset(&reads, 0, sizeof reads);
  for (const std::string &f : files)
    if (smbh_blow5_read(f.c_str(), &reads)) die("Error in opening file " + f + " (" + smbh_last_error() + ")");
  fprintf(stderr, "Loaded %zu reads in %fs.\n", reads.n, now() - t0);
  smbh_fasta fa;
  if (smbh_fasta_load(a.ref.c_str(), &fa)) die("Cannot find sequence file!");
  const std::vector<int> devs = a.gpus.empty() ? std::vector<int>{a.gpu} : a.gpus;
  const size_t G = devs.size();
  std::vector<smb_ctx *> ctxs(G, nullptr);
  for (size_t g = 0; g < G; ++g)
    if (smb_create(&ctxs[g], devs[g])) die(std::string("smb_create: ") + smb_last_error(nullptr));
  t0 = now();
  const bool by_contig = a.shard_contigs && G > 1;
  if (by_contig) {
    // every context gets the windows of its own contigs out of the same point cloud
    uint64_t *pos = nullptr;
    float *val = nullptr;
    size_t n_points = 0;
    int dim = 0, max_leaf = 0;
    if (!a.index_from_ref && smbh_pt_read(a.ref_index.c_str(), &pos, &val, &n_points, &dim, &max_leaf))
      die("Cannot read index file!");
    std::vector<uint32_t> owner(std::max(fa.n, 1u), 0);
    smbh_assign_contigs(fa.lengths, fa.n, (uint32_t)G, owner.data());
    if (smb_shard_local_group(ctxs.data(), (uint32_t)G)) die(std::string("smb_shard_local_group: ") + smb_last_error(ctxs[0]));
    std::vector<std::string> err(G);
    std::vector<std::thread> th;
    for (size_t g = 0; g < G; ++g)
      th.emplace_back([&, g] {
        if ((a.index_from_ref ? smb_index_build(ctxs[g], fa.seqs, fa.lengths, fa.n, level_mean.data(), owner.data())
                              : smb_index_set_points_sharded(ctxs[g], pos, val, n_points, owner.data(), fa.n)) ||
            smb_index_set_contigs(ctxs[g], fa.lengths, fa.n))
          err[g] = smb_last_error(ctxs[g]);
      });
    for (auto &t : th) t.join();
    for (size_t g = 0; g < G; ++g)
      if (!err[g].empty()) die("index shard " + std::to_string(g) + ": " + err[g]);
    smbh_free(pos);
    smbh_free(val);
  } else {
    for (size_t g = 0; g < G; ++g) {
      if (a.index_from_ref) {
        if (smb_index_build(ctxs[g], fa.seqs, fa.lengths, fa.n, level_mean.data(), nullptr))
          die(std::string("smb_index_build: ") + smb_last_error(ctxs[g]));
      } else if (smb_index_load(ctxs[g], a.ref_index.c_str())) {
        die(std::string("smb_index_load: ") + smb_last_error(ctxs[g]));
      }
      if (smb_index_set_contigs(ctxs[g], fa.lengths, fa.n)) die(std::string("smb_index_set_contigs: ") + smb_last_error(ctxs[g]));
    }
  }
  fprintf(stderr, "Loaded index successfully in %fs.\n", now() - t0);
  std::vector<smb_mapping> rows(reads.n ? reads.n : 1);
  t0 = now();
  uint64_t zero_off[1] = {0};
  // A device holds the raw samples of a call twice (as read and filtered, 2 B each): map a signal
  // directory larger than kMaxCallSamples per device in several calls -- reads are independent, so
  // the rows are the same -- instead of failing in cudaMalloc (the reference only needs host RAM).
  const uint64_t kMaxCallSamples = 12ull << 30;  // 48 GB of the 180 GB HBM
  if (G == 1) {
    for (size_t lo = 0; lo < reads.n || lo == 0;) {
      size_t hi = lo;
      while (hi < reads.n && (hi == lo || reads.read_off[hi + 1] - reads.read_off[lo] <= kMaxCallSamples)) ++hi;
      const size_t cnt = hi - lo;
      std::vector<uint64_t> off(cnt + 1, 0);
      for (size_t r = 0; r <= cnt && reads.n; ++r) off[r] = reads.read_off[lo + r] - reads.read_off[lo];
      const int16_t *raw = reads.n ? reads.raw + reads.read_off[lo] : reads.raw;
      if (smb_map_reads(ctxs[0], raw, reads.n ? off.data() : zero_off, reads.digitisation + lo, reads.range + lo,
                        reads.offset + lo, cnt, &a.prm, rows.data() + lo))
        die(std::string("smb_map_reads: ") + smb_last_error(ctxs[0]));
      if (hi >= reads.n) break;
      lo = hi;
    }
  } else {
    // reads: context g maps the g-th block of the reads; contigs: every context maps every read
    // (all calls identical, as the collectives require) and context 0's rows are the result
    std::vector<std::string> err(G);
    std::vector<std::vector<smb_mapping>> all(by_contig ? G : 0);
    std::vector<std::thread> th;
    for (size_t g = 0; g < G; ++g)
      th.emplace_back([&, g] {
        size_t lo = 0, hi = reads.n;
        if (!by_contig) {
          lo = reads.n * g / G;
          hi = reads.n * (g + 1) / G;
        }
        const size_t cnt = hi - lo;
        std::vector<uint64_t> off(cnt + 1, 0);
        for (size_t r = 0; r <= cnt && reads.n; ++r) off[r] = reads.read_off[lo + r] - reads.read_off[lo];
        smb_mapping *dst = rows.data() + lo;
        if (by_contig && g > 0) {
          all[g].resize(cnt ? cnt : 1);
          dst = all[g].data();
        }
        // (in several calls when the device's share is larger than kMaxCallSamples; contig shards
        // must all make the same calls, which they do: the split depends on the reads only)
        for (size_t b0 = 0; b0 < cnt || b0 == 0;) {
          size_t b1 = b0;
          while (b1 < cnt && (b1 == b0 || off[b1 + 1] - off[b0] <= kMaxCallSamples)) ++b1;
          std::vector<uint64_t> boff(b1 - b0 + 1, 0);
          for (size_t r = 0; r <= b1 - b0; ++r) boff[r] = off[b0 + r] - off[b0];
          const int16_t *raw = reads.n ? reads.raw + reads.read_off[lo] + off[b0] : reads.raw;
          if (smb_map_reads(ctxs[g], raw, boff.data(), reads.digitisation + lo + b0, reads.range + lo + b0,
                            reads.offset + lo + b0, b1 - b0, &a.prm, dst + b0)) {
            err[g] = smb_last_error(ctxs[g]);
            break;
          }
          if (b1 >= cnt) break;
          b0 = b1;
        }
      });
    for (auto &t : th) t.join();
    for (size_t g = 0; g < G; ++g)
      if (!err[g].empty()) die("smb_map_reads on device " + std::to_string(devs[g]) + ": " + err[g]);
  }
  const double dt = now() - t0;
  fprintf(stderr, "Finished mapping in %f, # reads: %zu\n", dt, reads.n);
  for (size_t g = 0; g < G; ++g) {
    smb_stats st;
    smb_stats_get(ctxs[g], &st);
    fprintf(stderr, "GPU %d: %.3f ms kernels (events %.3f, search %.3f, sort %.3f, chain %.3f), %llu samples, %llu queries, %llu hits\n",
            devs[g], st.ms_total, st.ms_events, st.ms_search, st.ms_sort, st.ms_chain, (unsigned long long)st.samples,
            (unsigned long long)st.queries, (unsigned long long)st.hits);
  }
  // rows grouped by contig (unmapped under contig 0), arrival order inside: sigmap.cc:197-241
  FILE *out = fopen(a.output.c_str(), "w");
  if (!out) die("Cannot open output file!");
  const double mt = reads.n ? dt * 1000.0 / reads.n : 0.0;
  std::vector<char> line(4096);
  std::vector<std::vector<uint32_t>> by_contig_rows(std::max(fa.n, 1u));
  for (size_t r = 0; r < reads.n; ++r) {
    const uint32_t bin = rows[r].mapped && rows[r].contig < fa.n ? rows[r].contig : 0;
    by_contig_rows[bin].push_back((uint32_t)r);
  }
  for (uint32_t c = 0; c < std::max(fa.n, 1u); ++c) {
    for (uint32_t r : by_contig_rows[c]) {
      const smb_mapping &m = rows[r];
      const char *cname = m.mapped && m.contig < fa.n ? fa.names[m.contig] : "*";
      const uint32_t clen = m.mapped && m.contig < fa.n ? fa.lengths[m.contig] : 0;
      smbh_format_paf(&m, reads.names[r], cname, clen, mt, line.data(), line.size());
      fputs(line.data(), out);
    }
  }
  fclose(out);
  for (smb_ctx *c : ctxs) smb_destroy(c);
  smbh_reads_free(&reads);
  smbh_fasta_free(&fa);
  return 0;
}

}  // namespace

int main(int argc, char **argv) {
  Args a = parse(argc, argv);
  if (a.index) return build_index(a);
  if (a.map) return map_reads(a);
  fputs(kHelp, stderr);
  return 0;
}
