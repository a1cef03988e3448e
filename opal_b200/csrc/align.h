// align.h -- the OPAL_SEARCH_ALIGNMENT stage (start location + operation string).
#pragma once
#include "../../include/opal.h"
#include "engine.h"

namespace opalb200 {
// For every database entry: derive start location and alignment from its (score, end location),
// as reference src/opal.cpp:1475-1507 does with findAlignment (:1236-1431).  db / lens may be NULL (the
// database's own host copy is used); with `subset`, record j belongs to database entry subset[j] and n counts records.
// Cells are scored as `s` says (with a PSSM its query residues are needed to label diagonal steps MATCH / MISMATCH);
// the band's M is the largest entry that can score a cell.
int align_database(DeviceDb* ddb, const Scoring& s, unsigned char* const* db, int n, const int* lens, OpalSearchResult* results[],
                   const int* subset = nullptr);
}  // namespace opalb200
