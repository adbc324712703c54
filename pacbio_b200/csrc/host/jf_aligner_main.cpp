// jf_aligner: drop-in for the reference binary (src_jf_aligner/jf_aligner.cc:161-233): same path
// as create_mega_reads but stops after the coords (jf_aligner.cc:41-70).
#include <iostream>
#include <stdexcept>

#include "cmdline.hpp"
#include "pipeline.hpp"

static const char* usage_text =
  "Usage: jf_aligner [options]\n"
  "Align PacBio reads and SuperReads\n\n"
  " -s, --size=uint64  -m, --mer=uint32 (required)  -F, --fine-mer=uint32  --psa-min=uint32 (13)\n"
  " -t, --threads=uint32 (1)  --stretch-constant=int (10)  --stretch-factor=double (1.3)  --stretch-cap=double (10000.0)\n"
  "     --window-size=uint32 (1)  -f, --forward  -B, --bases-matching=double (17.0)  -M, --mers-matching=double (0.0)\n"
  "     --details=path  --coords=path (stdout)  --max-match\n"
  " -H, --no-header  -0, --zero-match  --max-count=uint32 (5000)  -l, --unitigs-lengths=path  -u, --unitigs-sequences=path\n"
  "     --compact (toggles the compact format off)  -k, --k-mer=uint32  -r, --superreads=path  -p, --pacbio=path\n";

int main(int argc, char* argv[]) {
  using namespace cmdline;
  bool size_given = false, mer_given = false, k_given = false, l_given = false, u_given = false;
  bool forward = false, no_header = false, zero_match = false, compact = true, coords_given = false, details_given = false;
  uint32_t mer = 0, psa_min = 13, k_mer = 0;
  std::string unitigs_lengths, unitigs_sequences, coords_path, details_path;
  mr_params P;
  mr_params_default(&P);
  double bases_matching = 17.0, mers_matching = 0.0;
  std::vector<std::string> superreads, pacbio;

  enum { O_PSA_MIN = 1000, O_SC, O_SF, O_SCAP, O_WS, O_DETAILS, O_COORDS, O_MAXMATCH, O_MAXCOUNT, O_COMPACT, O_USAGE };
  static struct option long_options[] = {
    {"size", 1, 0, 's'}, {"mer", 1, 0, 'm'}, {"fine-mer", 1, 0, 'F'}, {"psa-min", 1, 0, O_PSA_MIN},
    {"threads", 1, 0, 't'}, {"stretch-constant", 1, 0, O_SC}, {"stretch-factor", 1, 0, O_SF},
    {"stretch-cap", 1, 0, O_SCAP}, {"window-size", 1, 0, O_WS}, {"forward", 0, 0, 'f'},
    {"bases-matching", 1, 0, 'B'}, {"mers-matching", 1, 0, 'M'}, {"details", 1, 0, O_DETAILS},
    {"coords", 1, 0, O_COORDS}, {"max-match", 0, 0, O_MAXMATCH}, {"no-header", 0, 0, 'H'},
    {"zero-match", 0, 0, '0'}, {"max-count", 1, 0, O_MAXCOUNT}, {"unitigs-lengths", 1, 0, 'l'},
    {"unitigs-sequences", 1, 0, 'u'}, {"compact", 0, 0, O_COMPACT}, {"k-mer", 1, 0, 'k'},
    {"superreads", 1, 0, 'r'}, {"pacbio", 1, 0, 'p'}, {"help", 0, 0, 'h'}, {"usage", 0, 0, O_USAGE},
    {"version", 0, 0, 'V'}, {0, 0, 0, 0}
  };
  while(true) {
    const int c = getopt_long(argc, argv, "hVs:m:F:t:fB:M:H0l:u:k:r:p:", long_options, nullptr);
    if(c == -1) break;
    switch(c) {
    case ':': case '?': error("Unrecognized or incomplete option");
    case 'h': case O_USAGE: fputs(usage_text, stdout); return 0;
    case 'V': puts("b200-mega-reads 0.1"); return 0;
    case 's': size_given = true; (void)to_uint64(optarg, "-s, --size=uint64", true); break;
    case 'm': mer_given = true; mer = to_uint32(optarg, "-m, --mer=uint32"); break;
    case 'F': P.fine_mer = to_uint32(optarg, "-F, --fine-mer=uint32"); break;
    case O_PSA_MIN: psa_min = to_uint32(optarg, "--psa-min=uint32"); break;
    case 't': (void)to_uint32(optarg, "-t, --threads=uint32"); break;
    case O_SC: P.stretch_constant = (double)to_int(optarg, "--stretch-constant=int"); break;
    case O_SF: P.stretch_factor = to_double(optarg, "--stretch-factor=double"); break;
    case O_SCAP: P.stretch_cap = to_double(optarg, "--stretch-cap=double"); break;
    case O_WS: P.window_size = to_uint32(optarg, "--window-size=uint32"); break;
    case 'f': forward = true; break;
    case 'B': bases_matching = to_double(optarg, "-B, --bases-matching=double"); break;
    case 'M': mers_matching = to_double(optarg, "-M, --mers-matching=double"); break;
    case O_DETAILS: details_given = true; details_path = optarg; break;
    case O_COORDS: coords_given = true; coords_path = optarg; break;
    case O_MAXMATCH: P.max_match = 1; break;
    case 'H': no_header = true; break;
    case '0': zero_match = true; break;
    case O_MAXCOUNT: P.max_count = (int32_t)to_uint32(optarg, "--max-count=uint32"); break;
    case 'l': l_given = true; unitigs_lengths = optarg; forward = true; break;
    case 'u': u_given = true; unitigs_sequences = optarg; forward = true; break;
    case O_COMPACT: compact = false; break;
    case 'k': k_given = true; k_mer = to_uint32(optarg, "-k, --k-mer=uint32"); break;
    case 'r': superreads.push_back(optarg); break;
    case 'p': pacbio.push_back(optarg); break;
    }
  }
  if(!size_given) error("[-s, --size=uint64] required switch");
  if(!mer_given) error("[-m, --mer=uint32] required switch");
  if(l_given && u_given) error("Switches [-u, --unitigs-sequences=path] and [-l, --unitigs-lengths=path] are mutually exclusive");
  if(argc - optind != 0) error("Requires exactly 0 argument.");
  if(!details_given && !coords_given) error("No output file given. Doing nothing ungracefully.");
  if(details_given && P.fine_mer) error("[--details] is not available together with -F in this build");
  if(P.window_size < 1) error("[--window-size] must be at least 1");
  if((l_given || u_given) && !k_given)
    error("The mer length used for generating the k-unitigs (-k, --k-mer) is required if the unitig lengths (-l, --unitig-lengths or -u, --unitigs-sequences) is passed.");

  try {
    FILE* out = coords_given ? fopen(coords_path.c_str(), "w") : stdout;     // jf_aligner.cc:175-179
    if(!out) throw std::runtime_error("Failed to open file '" + coords_path + "'");
    FILE* details = nullptr;
    if(details_given) {
      details = fopen(details_path.c_str(), "w");
      if(!details) throw std::runtime_error("Failed to open file '" + details_path + "'");
    }
    mrh::unitigs U;
    if(l_given) U.load_lengths(unitigs_lengths);
    else if(u_given) U.load_sequences(unitigs_sequences);
    mrh::super_reads SR;
    for(const auto& p : superreads) SR.append_fasta(p);
    if(SR.nseq() == 0) throw std::runtime_error("no super-read sequence");
    std::cerr << "compute_psa " << SR.nseq() << ' ' << SR.n << '\n';
    mrh::device_set DS;
    // the suffix array keeps suffixes down to min(fine mer, psa-min) bases (create_mega_reads.cc:131-132, jf_aligner.cc:202-203)
    mrh::build_indexes(DS, mrh::choose_devices(), SR, U, std::min<uint32_t>(P.fine_mer ? P.fine_mer : 22u, psa_min), mer);
    mrh::add_streams(DS, mrh::streams_per_device());
    P.matching_mers = mers_matching / 100.0;
    P.matching_bases = bases_matching / 100.0;
    P.unitigs_k = U.len.empty() ? 0 : k_mer;
    P.forward = forward;
    P.run_graph = 0;
    if(!no_header) {                                          // print_coords_header, jf_aligner.cc:32-39
      fputs("Rstart Rend Qstart Qend Nmers Rcons Qcons Rcover Qcover Rlen Qlen Stretch Offset Err", out);
      if(!compact) fputs(" Rname", out);
      fputs(" Qname\n", out);
    }
    if(details) for(auto c : DS.ctx) mr_context_keep_taps(c, 1);
    // The coords lines are printed on the device right after each batch (mr_coords_records); --details keeps both
    // files on the host formatter, which needs the taps of the result there.
    mrh::device_sr_names DN;
    mrh::records_fn device;
    const mr_coords_params cp = { compact ? 1 : 0, zero_match ? 1 : 0 };
    if(!details) {
      DN.upload(DS, SR);
      device = [&](mr_context* c, const mr_result* r, const mrh::read_batch& b) { return mrh::device_coords(c, r, cp, DN.of(c), b.name); };
    }
    mrh::text_buf dtext;
    mrh::run_pipeline(DS, pacbio, P,
      [&](const mr_result* r, const mr_result_view& v, const mrh::read_batch& b, std::vector<mrh::text_buf>& parts) {
        parts.resize(1);
        mrh::format_coords(v, b, 0, v.nreads, SR, compact, !zero_match, parts[0]);
        if(details) {                      // single formatter thread: no lock needed
          dtext.clear();
          mrh::format_details(r, b, SR, dtext);
          fwrite(dtext.data(), 1, dtext.size(), details);
        }
      }, out, 0, device);
    if(out != stdout) fclose(out);
    if(details) fclose(details);
  } catch(std::exception& e) {
    std::cerr << "jf_aligner: " << e.what() << std::endl;
    return 1;
  }
  return 0;
}
