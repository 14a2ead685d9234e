// Internal: the BAM reader shared by computeCounts (as_bam.cpp) and the two programs (as_host.cpp).  It walks the BGZF
// container of one file, inflates its blocks on host threads (zlib, CRC checked), maps the header's reference names to
// panel contigs, indexes the records and hands them to the GPU pileup (as_pileup_add_host) on a helper thread while the
// next piece inflates.  What the caller does with the finished pileup -- ASEQ text or a wire tensor -- is not its business.
#pragma once
#include <stdint.h>

#include <functional>
#include <map>
#include <memory>
#include <string>

#include "amplisolve_b200.h"

namespace asbam {

class Reader {
  public:
    Reader();
    ~Reader();
    // Piles up every record of `bam` into the pileup that begin() opens (as_pileup_begin) and returns its context, or
    // nullptr after printing why not.  begin() is called once the first records are ready (so a context that is still
    // starting up overlaps the first inflate), or at the end for a file without records.  Reads count when
    // mapq >= mrq and no flag bit of 0x704 is set; contig_id maps reference names to panel contigs.  Returns 0, or 1
    // after printing a computeCounts error message; *n_records receives the number of records (may be NULL).
    int pileup(const std::string& bam, const std::map<std::string, int32_t>& contig_id, int threads, int mbq, int mrq,
               const std::function<as_ctx*()>& begin, uint64_t* n_records);

  private:
    struct Impl;  // two piece buffers and the GPU helper thread, reused from file to file
    std::unique_ptr<Impl> impl_;
};

}  // namespace asbam
