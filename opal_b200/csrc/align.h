// align.h -- the OPAL_SEARCH_ALIGNMENT stage (start location + operation string).
#pragma once
#include "../../include/opal.h"
#include "engine.h"

namespace opalb200 {
// For every database entry: derive start location and alignment from its (score, end location),
// as reference src/opal.cpp:1475-1507 does with findAlignment (:1236-1431).  db / lens may be NULL (the
// database's own host copy is used); with `subset`, record j belongs to database entry subset[j] and n counts records.
// With `pssm` (Q x A, see DeviceDb::search) cells are scored by it and `matrix` is unused; `query` (codes < A) then
// only labels diagonal steps MATCH / MISMATCH, and the band's M is the largest PSSM entry.
int align_database(DeviceDb* ddb, const unsigned char* query, int Q, unsigned char* const* db, int n, const int* lens,
                   int Go, int Ge, const int* matrix, int A, OpalSearchResult* results[], int mode, const int* subset = nullptr,
                   const int* pssm = nullptr);
}  // namespace opalb200
