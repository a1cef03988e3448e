// align.h -- the OPAL_SEARCH_ALIGNMENT stage (start location + operation string).
#pragma once
#include "../../include/opal.h"
#include "engine.h"

#include <vector>

namespace opalb200 {
// The records of one search to align: n of them; record j belongs to database entry subset[j] (subset NULL: entry j).
// Cells are scored as `s` says (with a PSSM its query residues are needed to label diagonal steps MATCH / MISMATCH);
// the band's M is the largest entry that can score a cell.
struct AlignSet {
    const Scoring* s;
    OpalSearchResult* const* results;
    int n;
    const int* subset;
};
// For every record of every set: derive start location and alignment from its (score, end location), as reference
// src/opal.cpp:1475-1507 does with findAlignment (:1236-1431), on `stream` of the database's device, whose upload has
// finished.  The records of all sets share the launches.  db / lens may be NULL (the database's own host copy is used).
int align_database(const DbArrays& ddb, cudaStream_t stream, const std::vector<AlignSet>& sets, unsigned char* const* db = nullptr, const int* lens = nullptr);
}  // namespace opalb200
