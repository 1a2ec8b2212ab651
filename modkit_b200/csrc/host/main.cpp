// `modkit` drop-in entry point for the pileup path: `modkit pileup [flags] <in.bam> <out.bed>`
// (src/bin/main.rs:15-29, src/commands.rs:59-160), plus `modkit pileup-hemi` and `modkit summary` / `modkit sample-probs`. Other subcommands are
// out of scope (SURVEY 2.1).
#include "pileup_run.hpp"

extern "C" int mkh_pileup_main(int argc, const char* const* argv);
extern "C" int mkh_pileup_hemi_main(int argc, const char* const* argv);
extern "C" int mkh_summary_main(int argc, const char* const* argv);
extern "C" int mkh_sample_probs_main(int argc, const char* const* argv);

int main(int argc, char** argv) {
    const std::string cmd = argc >= 2 ? argv[1] : "";
    if (cmd == "pileup-hemi") return mkh_pileup_hemi_main(argc - 2, argv + 2);
    if (cmd == "summary") return mkh_summary_main(argc - 2, argv + 2);
    if (cmd == "sample-probs") return mkh_sample_probs_main(argc - 2, argv + 2);
    if (cmd != "pileup") {
        fprintf(stderr, "Usage: modkit pileup [OPTIONS] <IN_BAM> <OUT_BED>\n       modkit pileup-hemi [OPTIONS] --ref <FASTA> (--cpg | --motif <SEQ> <OFFSET>) <IN_BAM> [-o <OUT_BED>]\n       modkit summary [OPTIONS] <IN_BAM>\n       modkit sample-probs [OPTIONS] <IN_BAM>\n(the pileup path, pileup-hemi and the two sampling reports are what this build provides)\n");
        return 2;
    }
    return mkh_pileup_main(argc - 2, argv + 2);
}
