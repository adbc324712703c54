// create_mega_reads: drop-in for the reference binary of the same name
// (src_jf_aligner/create_mega_reads.cc:95-167).  Same options (create_mega_reads_cmdline.yaggo),
// same inputs, same text records; the per-read work runs on the GPU through the C ABI.
#include <chrono>
#include <iostream>
#include <stdexcept>

#include "cmdline.hpp"
#include "pipeline.hpp"

static const char* usage_text =
  "Usage: create_mega_reads [options]\n"
  "Align PacBio reads and SuperReads, and create mega reads\n\n"
  " -s, --size=uint64            Number of k-mers in SuperReads (required, unused)\n"
  " -m, --mer=uint32             Mer size (required)\n"
  " -F, --fine-mer=uint32        Mer size for fine alignment\n"
  "     --psa-min=uint32         Min suffix length in SA (13)\n"
  " -l, --unitigs-lengths=path   Length of k-unitigs\n"
  " -u, --unitigs-sequences=path Fasta file containing the sequence of the k-unitigs\n"
  " -k, --k-mer=uint32           Length of k-mer used to create k-unitigs (required)\n"
  " -t, --threads=uint32         Number of host threads (1)\n"
  " -o, --output=path            Output file (stdout)\n"
  "     --dot=path               Write an overlap graph (not implemented)\n"
  "     --stretch-constant=int   (10)   --stretch-factor=double (1.3)   --stretch-cap=double (10000.0)\n"
  "     --window-size=uint32     (1)\n"
  " -O, --overlap-play=double    (1.3)  -e, --errors=double (3.0)\n"
  " -B, --bases-matching=double  (17.0) -M, --mers-matching=double (0.0)\n"
  "     --max-match              Use secondary matches\n"
  "     --max-count=uint32       (5000) -b, --bases\n"
  " -d, --density=double         (0.029) -L, --min-length=double (100.0)\n"
  " -T, --tiling=none|greedy|maximal|weighted (greedy)   --trim=none|match|branch (none)\n"
  " -r, --superreads=path        SuperReads sequence file (multiple)\n"
  " -p, --pacbio=path            PacBio read sequence file (multiple)\n"
  "GPUs: MR_DEVICES=0,1,.. or MR_GPUS=N (reads are sharded across them); MR_BATCH_BASES=bases per batch\n";

int main(int argc, char* argv[]) {
  using namespace cmdline;
  bool size_given = false, mer_given = false, k_given = false, l_given = false, u_given = false;
  uint32_t mer = 0, psa_min = 13, k_mer = 0, threads = 1;
  std::string unitigs_lengths, unitigs_sequences, output, dot_path;
  mr_params P;
  mr_params_default(&P);
  double bases_matching = 17.0, mers_matching = 0.0;
  mrh::graph_options G;
  std::vector<std::string> superreads, pacbio;
  bool show_timing = getenv("MR_SHOW_TIMING") != nullptr;

  enum { O_PSA_MIN = 1000, O_DOT, O_SC, O_SF, O_SCAP, O_WS, O_MAXMATCH, O_MAXCOUNT, O_TRIM, O_USAGE };
  static struct option long_options[] = {
    {"size", 1, 0, 's'}, {"mer", 1, 0, 'm'}, {"fine-mer", 1, 0, 'F'}, {"psa-min", 1, 0, O_PSA_MIN},
    {"unitigs-lengths", 1, 0, 'l'}, {"unitigs-sequences", 1, 0, 'u'}, {"k-mer", 1, 0, 'k'},
    {"threads", 1, 0, 't'}, {"output", 1, 0, 'o'}, {"dot", 1, 0, O_DOT},
    {"stretch-constant", 1, 0, O_SC}, {"stretch-factor", 1, 0, O_SF}, {"stretch-cap", 1, 0, O_SCAP},
    {"window-size", 1, 0, O_WS}, {"overlap-play", 1, 0, 'O'}, {"errors", 1, 0, 'e'},
    {"bases-matching", 1, 0, 'B'}, {"mers-matching", 1, 0, 'M'}, {"max-match", 0, 0, O_MAXMATCH},
    {"max-count", 1, 0, O_MAXCOUNT}, {"bases", 0, 0, 'b'}, {"density", 1, 0, 'd'},
    {"min-length", 1, 0, 'L'}, {"tiling", 1, 0, 'T'}, {"trim", 1, 0, O_TRIM},
    {"superreads", 1, 0, 'r'}, {"pacbio", 1, 0, 'p'}, {"help", 0, 0, 'h'}, {"usage", 0, 0, O_USAGE},
    {"version", 0, 0, 'V'}, {0, 0, 0, 0}
  };
  while(true) {
    const int c = getopt_long(argc, argv, "hVs:m:F:l:u:k:t:o:O:e:B:M:bd:L:T:r:p:", long_options, nullptr);
    if(c == -1) break;
    switch(c) {
    case ':': case '?': error("Unrecognized or incomplete option");
    case 'h': case O_USAGE: fputs(usage_text, stdout); return 0;
    case 'V': puts("b200-mega-reads 0.1"); return 0;
    case 's': size_given = true; (void)to_uint64(optarg, "-s, --size=uint64", true); break;
    case 'm': mer_given = true; mer = to_uint32(optarg, "-m, --mer=uint32"); break;
    case 'F': P.fine_mer = to_uint32(optarg, "-F, --fine-mer=uint32"); break;
    case O_PSA_MIN: psa_min = to_uint32(optarg, "--psa-min=uint32"); break;
    case 'l': l_given = true; unitigs_lengths = optarg; break;
    case 'u': u_given = true; unitigs_sequences = optarg; break;
    case 'k': k_given = true; k_mer = to_uint32(optarg, "-k, --k-mer=uint32"); break;
    case 't': threads = to_uint32(optarg, "-t, --threads=uint32"); break;
    case 'o': output = optarg; break;
    case O_DOT: dot_path = optarg; break;
    case O_SC: P.stretch_constant = (double)to_int(optarg, "--stretch-constant=int"); break;
    case O_SF: P.stretch_factor = to_double(optarg, "--stretch-factor=double"); break;
    case O_SCAP: P.stretch_cap = to_double(optarg, "--stretch-cap=double"); break;
    case O_WS: P.window_size = to_uint32(optarg, "--window-size=uint32"); break;
    case 'O': P.overlap_play = G.overlap_play = to_double(optarg, "-O, --overlap-play=double"); break;
    case 'e': P.errors = to_double(optarg, "-e, --errors=double"); break;
    case 'B': bases_matching = to_double(optarg, "-B, --bases-matching=double"); break;
    case 'M': mers_matching = to_double(optarg, "-M, --mers-matching=double"); break;
    case O_MAXMATCH: P.max_match = 1; break;
    case O_MAXCOUNT: P.max_count = (int32_t)to_uint32(optarg, "--max-count=uint32"); break;
    case 'b': P.bases = 1; break;
    case 'd': G.density = to_double(optarg, "-d, --density=double"); break;
    case 'L': G.min_length = to_double(optarg, "-L, --min-length=double"); break;
    case 'T':
      if(!strcmp(optarg, "none")) G.tiling = 0; else if(!strcmp(optarg, "greedy")) G.tiling = 1;
      else if(!strcmp(optarg, "maximal")) G.tiling = 2; else if(!strcmp(optarg, "weighted")) G.tiling = 3;
      else error(std::string("Invalid enum '") + optarg + "' for [-T, --tiling]");
      break;
    case O_TRIM:
      if(!strcmp(optarg, "none")) G.trim = 0; else if(!strcmp(optarg, "match")) G.trim = 1;
      else if(!strcmp(optarg, "branch")) G.trim = 0;     // create_mega_reads.cc:47-49 only acts on `match`
      else error(std::string("Invalid enum '") + optarg + "' for [--trim]");
      break;
    case 'r': superreads.push_back(optarg); break;
    case 'p': pacbio.push_back(optarg); break;
    }
  }
  if(!size_given) error("[-s, --size=uint64] required switch");
  if(!mer_given) error("[-m, --mer=uint32] required switch");
  if(!k_given) error("[-k, --k-mer=uint32] required switch");
  if(l_given && u_given) error("Switches [-u, --unitigs-sequences=path] and [-l, --unitigs-lengths=path] are mutually exclusive");
  if(argc - optind != 0) error("Requires exactly 0 argument.");
  if(P.window_size < 1) error("[--window-size] must be at least 1");

  try {
    // open the output first, for early error reporting (create_mega_reads.cc:101-107)
    FILE* out = stdout;
    if(!output.empty()) {
      out = fopen(output.c_str(), "w");
      if(!out) throw std::runtime_error("Failed to open file '" + output + "'");
    }
    static char obuf[1 << 22];
    setvbuf(out, obuf, _IOFBF, sizeof(obuf));

    mrh::unitigs U;
    if(l_given) U.load_lengths(unitigs_lengths);
    else U.load_sequences(unitigs_sequences);       // like the reference, a missing -l/-u fails on open

    const auto t0 = std::chrono::steady_clock::now();
    mrh::super_reads SR;
    for(const auto& p : superreads) SR.append_fasta(p);
    if(SR.nseq() == 0) throw std::runtime_error("no super-read sequence");
    std::cerr << "compute_psa " << SR.nseq() << ' ' << SR.n << '\n';
    mrh::device_set DS;
    // the suffix array keeps suffixes down to min(fine mer, psa-min) bases (create_mega_reads.cc:131-132, jf_aligner.cc:202-203)
    mrh::build_indexes(DS, mrh::choose_devices(), SR, U, std::min<uint32_t>(P.fine_mer ? P.fine_mer : 22u, psa_min), mer);
    mrh::add_streams(DS, mrh::streams_per_device());
    const auto t1 = std::chrono::steady_clock::now();
    if(show_timing) std::cerr << "Starting Super read parse ... " << std::chrono::duration<double>(t1 - t0).count() << '\n';

    P.matching_mers = mers_matching / 100.0;
    P.matching_bases = bases_matching / 100.0;
    P.unitigs_k = k_mer;
    P.forward = 1;
    P.run_graph = 1;
    G.k_len = k_mer;
    const unsigned fthreads = std::max(1u, threads);
    // --dot: the overlap graph of every read (overlap_graph.hpp:189-196); written by this one formatter thread, in read
    // order, which is what the reference gives with -t 1
    FILE* dot_file = nullptr;
    if(!dot_path.empty() && !(dot_file = fopen(dot_path.c_str(), "w"))) throw std::runtime_error("Failed to open file '" + dot_path + "'");
    mrh::dot_state dstate;
    dstate.errors = P.errors; dstate.bases = P.bases;
    mrh::text_buf dot_text;
    // the records are printed on the device (mr_records); --dot needs the host formatter, which recomputes the
    // graph's edges and carries the stream state of the --dot file
    mrh::device_unitigs DU;
    mrh::records_fn records;
    const mr_records_params RP = mrh::records_params(G);
    if(!dot_file) {
      DU.upload(DS, U);
      records = [&](mr_context* c, const mr_result* r, const mrh::read_batch& b) { return mrh::device_records(c, r, RP, DU.of(c), b.name); };
    }
    const uint64_t nb = mrh::run_pipeline(DS, pacbio, P,
      [&](const mr_result*, const mr_result_view& v, const mrh::read_batch& b, std::vector<mrh::text_buf>& parts) {
        parts.resize(1);
        parts[0].clear(); dot_text.clear();
        mrh::format_mega_reads(v, b, 0, v.nreads, SR, U, G, parts[0], &dot_text, &dstate);
        if(fwrite(dot_text.data(), 1, dot_text.size(), dot_file) != dot_text.size()) throw std::runtime_error("write error on the --dot file");
      }, out, fthreads, records);
    if(dot_file && fclose(dot_file) != 0) throw std::runtime_error("write error on the --dot file");
    const auto t2 = std::chrono::steady_clock::now();
    if(show_timing) std::cerr << "Starting create mega reads ... " << std::chrono::duration<double>(t2 - t1).count()
                              << " (" << nb << " bases)\n";
    if(out != stdout) fclose(out);
  } catch(std::exception& e) {
    std::cerr << "create_mega_reads: " << e.what() << std::endl;
    return 1;
  }
  return 0;
}
