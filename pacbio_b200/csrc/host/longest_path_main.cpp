// longest_path_overlap_graph2: drop-in for the reference binary of the same name
// (src_jf_aligner/longest_path_overlap_graph2.cc:33-118): the graph stage of create_mega_reads fed
// from a compact coords file (jf_aligner --coords) instead of from the aligner.  Same options
// (longest_path_overlap_graph2_cmdline.yaggo), same text records; the per-read overlap graph runs
// on the GPU through mr_graph_batch.
#include <iostream>
#include <stdexcept>

#include "cmdline.hpp"
#include "pipeline.hpp"

static const char* usage_text =
  "Usage: longest_path_overlap_graph2 [options] coords:path\n"
  "Find the longest path in the super-read overlap graph\n\n"
  " -t, --threads=uint32         Number of host threads (1)\n"
  " -o, --output=path            Output file (stdout)\n"
  "     --dot=path               Write an overlap graph (not implemented)\n"
  " -O, --overlap-play=double    (1.3)  -e, --errors=double (3.0)  -b, --bases\n"
  " -l, --unitigs-lengths=path   Length of k-unitigs\n"
  " -u, --unitigs-sequences=path Fasta file containing the sequence of the k-unitigs\n"
  " -k, --k-mer=uint32           Length of k-mer used to create k-unitigs (required)\n"
  " -d, --density=double         (0.029) -L, --min-length=double (100.0)\n"
  " -T, --tiling=none|greedy|maximal (greedy)   --trim=none|match|branch (none)\n";

int main(int argc, char* argv[]) {
  using namespace cmdline;
  bool k_given = false, l_given = false, u_given = false;
  uint32_t k_mer = 0;
  std::string unitigs_lengths, unitigs_sequences, output;
  mr_params P;
  mr_params_default(&P);
  mrh::graph_options G;

  enum { O_DOT = 1000, O_TRIM, O_USAGE };
  static struct option long_options[] = {
    {"threads", 1, 0, 't'}, {"output", 1, 0, 'o'}, {"dot", 1, 0, O_DOT}, {"overlap-play", 1, 0, 'O'},
    {"errors", 1, 0, 'e'}, {"bases", 0, 0, 'b'}, {"unitigs-lengths", 1, 0, 'l'}, {"unitigs-sequences", 1, 0, 'u'},
    {"k-mer", 1, 0, 'k'}, {"density", 1, 0, 'd'}, {"min-length", 1, 0, 'L'}, {"tiling", 1, 0, 'T'},
    {"trim", 1, 0, O_TRIM}, {"help", 0, 0, 'h'}, {"usage", 0, 0, O_USAGE}, {"version", 0, 0, 'V'}, {0, 0, 0, 0}
  };
  while(true) {
    const int c = getopt_long(argc, argv, "hVt:o:O:e:bl:u:k:d:L:T:", long_options, nullptr);
    if(c == -1) break;
    switch(c) {
    case ':': case '?': error("Unrecognized or incomplete option");
    case 'h': case O_USAGE: fputs(usage_text, stdout); return 0;
    case 'V': puts("b200-mega-reads 0.1"); return 0;
    case 't': (void)to_uint32(optarg, "-t, --threads=uint32"); break;     // accepted; the records are printed on the GPU
    case 'o': output = optarg; break;
    case O_DOT: error("[--dot] writing the overlap graph is not implemented in this build");
    case 'O': P.overlap_play = G.overlap_play = to_double(optarg, "-O, --overlap-play=double"); break;
    case 'e': P.errors = to_double(optarg, "-e, --errors=double"); break;
    case 'b': P.bases = 1; break;
    case 'l': l_given = true; unitigs_lengths = optarg; break;
    case 'u': u_given = true; unitigs_sequences = optarg; break;
    case 'k': k_given = true; k_mer = to_uint32(optarg, "-k, --k-mer=uint32"); break;
    case 'd': G.density = to_double(optarg, "-d, --density=double"); break;
    case 'L': G.min_length = to_double(optarg, "-L, --min-length=double"); break;
    case 'T':
      if(!strcmp(optarg, "none")) G.tiling = 0; else if(!strcmp(optarg, "greedy")) G.tiling = 1;
      else if(!strcmp(optarg, "maximal")) G.tiling = 2;
      else error(std::string("Invalid enum '") + optarg + "' for [-T, --tiling]");
      break;
    case O_TRIM:
      if(!strcmp(optarg, "none")) G.trim = 0; else if(!strcmp(optarg, "match")) G.trim = 1;
      else if(!strcmp(optarg, "branch")) G.trim = 0;     // longest_path_overlap_graph2.cc:46-48 only acts on `match`
      else error(std::string("Invalid enum '") + optarg + "' for [--trim]");
      break;
    }
  }
  if(!k_given) error("[-k, --k-mer=uint32] required switch");
  if(l_given && u_given) error("Switches [-u, --unitigs-sequences=path] and [-l, --unitigs-lengths=path] are mutually exclusive");
  if(argc - optind != 1) error("Requires exactly 1 argument.");
  if(!l_given && !u_given) error("One of --unitigs-lengths or --unitigs-sequences is required.");
  const std::string coords_path = argv[optind];

  try {
    FILE* out = stdout;
    if(!output.empty()) {
      out = fopen(output.c_str(), "w");
      if(!out) throw std::runtime_error("Failed to open file '" + output + "'");
    }
    static char obuf[1 << 22];
    setvbuf(out, obuf, _IOFBF, sizeof(obuf));
    mrh::unitigs U;
    if(l_given) U.load_lengths(unitigs_lengths); else U.load_sequences(unitigs_sequences);
    mrh::coords_file in(coords_path);

    mr_context* ctx = nullptr;
    if(mr_context_create(mrh::choose_devices()[0], &ctx) != MR_OK) throw std::runtime_error(std::string("mr_context_create: ") + mr_last_error(nullptr));
    P.unitigs_k = k_mer;
    P.run_graph = 1;
    G.k_len = k_mer;
    uint64_t max_rows = 1u << 20;
    if(const char* e = getenv("MR_BATCH_ROWS")) max_rows = strtoull(e, nullptr, 0);
    mrh::coords_batch b;
    const mr_records_params RP = mrh::records_params(G);
    mr_unitigs* DU = nullptr;
    if(U.has_sequences() && mr_unitigs_create(ctx, U.fwd.data(), U.off.data(), (uint32_t)U.len.size(), &DU) != MR_OK)
      throw std::runtime_error(std::string("mr_unitigs_create: ") + mr_last_error(ctx));
    while(in.next_batch(b, max_rows)) {
      const mr_result_view rows = b.view();
      mr_result* r = nullptr;
      static const uint32_t no_ids = 0;       // every name of the batch was unparsable: an empty table, but not a null one
      if(mr_graph_batch(ctx, &P, &rows, b.read_len.data(), b.paths.unitig_ids.empty() ? &no_ids : b.paths.unitig_ids.data(),
                        b.paths.unitig_off.data(), (uint32_t)b.paths.name.size(), U.len.data(), (uint32_t)U.len.size(), &r) != MR_OK)
        throw std::runtime_error(std::string("mr_graph_batch: ") + mr_last_error(ctx));
      // the records are printed on the device, from the rows and the path table mr_graph_batch left there
      mr_text* t = mrh::device_records(ctx, r, RP, DU, b.reads.name);
      const char* text = nullptr;
      uint64_t n = 0;
      mr_text_get(t, &text, &n);
      const bool ok = n == 0 || fwrite(text, 1, n, out) == n;
      mr_text_free(t);
      mr_result_free(r);
      if(!ok) throw std::runtime_error("write error on output file");
    }
    mr_unitigs_destroy(DU);
    mr_context_destroy(ctx);
    if(out != stdout) fclose(out);
  } catch(std::exception& e) {
    std::cerr << "longest_path_overlap_graph2: " << e.what() << std::endl;
    return 1;
  }
  return 0;
}
