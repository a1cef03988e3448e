/*
 * oracle_pssm.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The scalar oracle (oracle/opal_oracle.c) restated for a position-specific scoring matrix: pssm is Q x A ints,
 * row-major, and pssm[r * A + y] scores query position r against target residue y where the matrix search reads
 * S[q[r] * A + y].  Everything else -- Gotoh recurrence and visiting order, end-location key, empty query / target
 * results, band borders, reverse DP and traceback, reuse rule for prefilled records -- is the oracle's, and so is the
 * code where it can be shared: opal_oracle.c is included as it stands (its golden vectors stay pinned) and only the two
 * loops that read a score are restated here with a row of the PSSM instead of a row of the matrix.
 *
 * Differences forced by the PSSM:
 *   - the alignment stage runs on the reversed prefixes with the PSSM rows reversed as well, and the band's M is the
 *     largest of all Q x A entries;
 *   - diagonal steps are labelled MATCH / MISMATCH from `query`, the residues the PSSM was built for (required for
 *     OPAL_SEARCH_ALIGNMENT, unused otherwise).
 * Built by the tests (cc -shared) into a temporary directory; it exports the oracle's symbols plus oracle_search_pssm.
 */
#include "../oracle/opal_oracle.c"

/* oracle_score_end with P (a PSSM) in place of S[q[r] * A + .]: same loops, same key. */
static int pssm_score_end(const int* P, int Q, const unsigned char* t, int T, int Go, int Ge, int A, int mode,
                          int* score, int* endQ, int* endT) {
    i64* prevH = (i64*)malloc(sizeof(i64) * (size_t)(Q > 0 ? Q : 1));
    i64* prevE = (i64*)malloc(sizeof(i64) * (size_t)(Q > 0 ? Q : 1));
    int rc = 0;
    i64 best;
    int bq = -1, bt = -1;

    if (mode == OPAL_MODE_SW) {
        for (int r = 0; r < Q; r++) prevH[r] = prevE[r] = 0;
        best = 0;
        for (int c = 0; c < T; c++) {
            i64 uF = 0, uH = 0, ulH = 0;
            for (int r = 0; r < Q; r++) {
                i64 E = max2(prevH[r] - Go, prevE[r] - Ge);
                i64 F = max2(uH - Go, uF - Ge);
                i64 d = ulH + P[(size_t)r * A + t[c]];
                if (d > INT_MAX) rc = 1;
                i64 H = max2(max2(E, F), max2(d, 0));
                if (H > best) { best = H; bq = r; bt = c; }
                uF = F; uH = H; ulH = prevH[r];
                prevH[r] = H; prevE[r] = E;
            }
        }
    } else {
        for (int r = 0; r < Q; r++) {
            prevH[r] = (mode == OPAL_MODE_OV) ? 0 : -(i64)Go - (i64)r * Ge;
            prevE[r] = NEG_INF;
        }
        best = NEG_INF;
        i64 H = NEG_INF;
        for (int c = 0; c < T; c++) {
            i64 uF = NEG_INF, uH, ulH;
            if (mode == OPAL_MODE_NW) {
                uH = -(i64)Go - (i64)c * Ge;
                ulH = (c == 0) ? 0 : uH + Ge;
            } else {
                uH = ulH = 0;
            }
            for (int r = 0; r < Q; r++) {
                i64 E = max2(prevH[r] - Go, prevE[r] - Ge);
                i64 F = max2(uH - Go, uF - Ge);
                H = max2(max2(E, F), ulH + P[(size_t)r * A + t[c]]);
                if (mode == OPAL_MODE_OV && c == T - 1 && H > best) { best = H; bq = r; bt = c; }
                uF = F; uH = H; ulH = prevH[r];
                prevH[r] = H; prevE[r] = E;
            }
            if (mode != OPAL_MODE_NW && Q > 0 && H > best) { best = H; bq = Q - 1; bt = c; }
        }
        if (mode == OPAL_MODE_NW) {
            if (T > 0 && Q > 0) best = H;
            else if (Q > 0) best = -(i64)Go - (i64)(Q - 1) * Ge;
            else if (T > 0) best = -(i64)Go - (i64)(T - 1) * Ge;
            else best = 0;
            bq = Q - 1; bt = T - 1;
        } else if (best == NEG_INF) {
            best = (mode == OPAL_MODE_HW && Q > 0) ? -(i64)Go - (i64)(Q - 1) * Ge : 0;
            bq = Q - 1; bt = T - 1;
        }
        if (best > INT_MAX || best < INT_MIN) rc = 1;
    }
    free(prevH); free(prevE);
    if (rc) return 1;
    *score = (int)best;
    if (mode == OPAL_MODE_SW && best == 0) { *endQ = -1; *endT = -1; }
    else { *endQ = bq; *endT = bt; }
    return 0;
}

/* oracle_find_alignment with P in place of S[q[r] * A + .] and the band's M given (the PSSM maximum); q only labels
 * the diagonal steps. */
static int pssm_find_alignment(const unsigned char* q, const int* P, int Q, const unsigned char* t, int T,
                               int Go, int Ge, int A, int M, int scoreLimit, int mode,
                               int* outScore, int* outEndQ, int* outEndT, unsigned char** ops, int* opsLen) {
    int bottom, top;
    if (oracle_band_borders(scoreLimit, mode, Q, T, Go, Ge, M, &bottom, &top) != 0) {
        bottom = Q - 1; top = T - 1;
    }

    Cell** mat = (Cell**)calloc((size_t)T, sizeof(Cell*));
    Cell* init = (Cell*)malloc(sizeof(Cell) * (size_t)Q);
    for (int r = 0; r < Q; r++) { init[r].H = -(i64)Go - (i64)r * Ge; init[r].E = NEG_INF; init[r].F = NEG_INF; }

    Cell* prev = init;
    i64 maxScore = NEG_INF, H = NEG_INF;
    int c;
    for (c = 0; c < T && maxScore < scoreLimit; c++) {
        Cell* col = mat[c] = (Cell*)malloc(sizeof(Cell) * (size_t)Q);
        int r0 = imax(0, c - top), r1 = imin(Q - 1, c + bottom);
        i64 uF, uH, ulH;
        if (r0 == 0) { uF = NEG_INF; uH = -(i64)Go - (i64)c * Ge; ulH = (c == 0) ? 0 : uH + Ge; }
        else { uH = uF = NEG_INF; ulH = prev[r0 - 1].H; }
        for (int r = r0; r <= r1; r++) {
            i64 E = max2(prev[r].H > NEG_INF ? prev[r].H - Go : NEG_INF, prev[r].E > NEG_INF ? prev[r].E - Ge : NEG_INF);
            i64 F = max2(uH > NEG_INF ? uH - Go : NEG_INF, uF > NEG_INF ? uF - Ge : NEG_INF);
            i64 d = ulH > NEG_INF ? ulH + P[(size_t)r * A + t[c]] : NEG_INF;
            H = max2(E, max2(F, d));
            if (mode == OPAL_MODE_SW || (mode == OPAL_MODE_OV && c == T - 1)) maxScore = max2(maxScore, H);
            uF = F; uH = H; ulH = prev[r].H;
            col[r].H = H; col[r].E = E; col[r].F = F;
        }
        for (int r = 0; r < r0; r++) col[r].H = col[r].E = col[r].F = NEG_INF;
        for (int r = r1 + 1; r < Q; r++) col[r].H = col[r].E = col[r].F = NEG_INF;
        if (mode == OPAL_MODE_HW || mode == OPAL_MODE_OV) maxScore = max2(maxScore, H);
        prev = col;
    }
    int lastCol = c - 1;
    int rc = 0, eq = -1, et = -1;
    i64 sc = NEG_INF;
    if (lastCol < 0) rc = -1;
    else if (mode == OPAL_MODE_NW) { sc = H; et = T - 1; eq = Q - 1; if (lastCol != T - 1) rc = -1; }
    else if (mode == OPAL_MODE_HW) { sc = maxScore; et = lastCol; eq = Q - 1; }
    else {
        sc = maxScore; et = lastCol;
        int r = 0;
        while (r < Q && mat[lastCol][r].H != maxScore) r++;
        if (r >= Q) rc = -1;
        eq = r;
    }
    if (rc == 0 && sc < scoreLimit && mode != OPAL_MODE_NW) rc = -1;

    unsigned char* a = NULL;
    int n = 0;
    if (rc == 0) {
        a = (unsigned char*)malloc((size_t)(Q + T + 2));
        int ri = eq, ci = et;
        int field = 0;
        while (ri >= 0 && ci >= 0) {
            Cell cell = mat[ci][ri];
            if (field == 0) {
                if (cell.H == cell.E) field = 1;
                else if (cell.H == cell.F) field = 2;
                else { a[n++] = (q[ri] == t[ci]) ? OPAL_ALIGN_MATCH : OPAL_ALIGN_MISMATCH; ci--; ri--; }
            } else if (field == 1) {
                i64 leftH = (ci > 0) ? mat[ci - 1][ri].H : init[ri].H;
                field = (cell.E == leftH - Go) ? 0 : 1;
                a[n++] = OPAL_ALIGN_INS; ci--;
            } else {
                i64 upH = (ri > 0) ? mat[ci][ri - 1].H : -(i64)Go - (i64)ci * Ge;
                field = (cell.F == upH - Go) ? 0 : 2;
                a[n++] = OPAL_ALIGN_DEL; ri--;
            }
        }
        while (ri >= 0) { a[n++] = OPAL_ALIGN_DEL; ri--; }
        while (ci >= 0) { a[n++] = OPAL_ALIGN_INS; ci--; }
        for (int i = 0; i < n / 2; i++) { unsigned char x = a[i]; a[i] = a[n - 1 - i]; a[n - 1 - i] = x; }
    }
    for (int i = 0; i <= lastCol; i++) free(mat[i]);
    free(mat); free(init);
    if (rc) return rc;
    *outScore = (int)sc; *outEndQ = eq; *outEndT = et; *ops = a; *opsLen = n;
    return 0;
}

/*
 * opalSearchDatabase of the oracle with a PSSM: same flow (reuse rule, score + end, reversed-prefix alignment, fills).
 * Returns 0, OPAL_ERR_INVALID_MODE, OPAL_ERR_OVERFLOW (an entry or gap outside (INT_MIN / 2, INT_MAX / 2), or a score
 * outside int) or OPAL_ERR_INVALID_ARGUMENT (pssm NULL with Q > 0, alphabet outside [1, 256], negative gaps, database
 * codes >= A, query NULL or codes >= A at OPAL_SEARCH_ALIGNMENT).
 */
int oracle_search_pssm(const unsigned char* query, const int* pssm, int Q, unsigned char* db[], int N, const int lens[],
                       int Go, int Ge, int A, OpalSearchResult* results[], int searchType, int mode) {
    if (mode != OPAL_MODE_NW && mode != OPAL_MODE_HW && mode != OPAL_MODE_OV && mode != OPAL_MODE_SW) return OPAL_ERR_INVALID_MODE;
    if (A < 1 || A > 256 || (Q > 0 && !pssm)) return OPAL_ERR_INVALID_ARGUMENT;
    if (Go <= INT_MIN / 2 || INT_MAX / 2 <= Go || Ge <= INT_MIN / 2 || INT_MAX / 2 <= Ge) return OPAL_ERR_OVERFLOW;
    int M = 0;
    for (i64 i = 0; i < (i64)Q * A; i++) {
        if (pssm[i] <= INT_MIN / 2 || INT_MAX / 2 <= pssm[i]) return OPAL_ERR_OVERFLOW;
        if (i == 0 || pssm[i] > M) M = pssm[i];
    }
    if (Go < 0 || Ge < 0) return OPAL_ERR_INVALID_ARGUMENT;
    for (int i = 0; i < N; i++)
        for (int c = 0; c < lens[i]; c++)
            if (db[i][c] >= A) return OPAL_ERR_INVALID_ARGUMENT;
    if (searchType == OPAL_SEARCH_ALIGNMENT && Q > 0) {
        if (!query) return OPAL_ERR_INVALID_ARGUMENT;
        for (int r = 0; r < Q; r++)
            if (query[r] >= A) return OPAL_ERR_INVALID_ARGUMENT;
    }

    int status = 0;
    for (int i = 0; i < N; i++) {
        OpalSearchResult* r = results[i];
        int skip = r->scoreSet && (searchType == OPAL_SEARCH_SCORE || (r->endLocationQuery >= 0 && r->endLocationTarget >= 0));
        if (skip) continue;
        int sc, eq, et;
        if (pssm_score_end(pssm, Q, db[i], lens[i], Go, Ge, A, mode, &sc, &eq, &et)) { status = OPAL_ERR_OVERFLOW; continue; }
        opalSearchResultSetScore(r, sc);
        if (searchType == OPAL_SEARCH_SCORE) { r->endLocationQuery = -1; r->endLocationTarget = -1; }
        else { r->endLocationQuery = eq; r->endLocationTarget = et; }
    }
    if (status) return status;

    if (searchType == OPAL_SEARCH_ALIGNMENT) {
        /* the reversed problem: reversed query and reversed PSSM rows (row Q - 1 - r of the PSSM is row r of rp) */
        unsigned char* rq = reversed_copy(query, Q);
        int* rp = (int*)malloc(sizeof(int) * (size_t)(Q > 0 ? Q : 1) * (size_t)A);
        for (int r = 0; r < Q; r++) memcpy(rp + (size_t)r * A, pssm + (size_t)(Q - 1 - r) * A, sizeof(int) * (size_t)A);
        for (int i = 0; i < N; i++) {
            OpalSearchResult* r = results[i];
            if ((mode == OPAL_MODE_SW && r->score == 0) || r->endLocationQuery < 0 || r->endLocationTarget < 0) {
                r->alignment = NULL; r->alignmentLength = 0;
                r->startLocationQuery = r->startLocationTarget = -1;
                r->endLocationQuery = r->endLocationTarget = -1;
                continue;
            }
            int aq = r->endLocationQuery + 1, at = r->endLocationTarget + 1;
            unsigned char* rt = reversed_copy(db[i], at);
            int sc, eq, et, n; unsigned char* ops;
            if (pssm_find_alignment(rq + Q - aq, rp + (size_t)(Q - aq) * A, aq, rt, at, Go, Ge, A, M, r->score, mode,
                                    &sc, &eq, &et, &ops, &n) == 0) {
                r->startLocationQuery = aq - eq - 1;
                r->startLocationTarget = at - et - 1;
                for (int k = 0; k < n / 2; k++) { unsigned char x = ops[k]; ops[k] = ops[n - 1 - k]; ops[n - 1 - k] = x; }
                r->alignment = (unsigned char*)realloc(ops, (size_t)(n > 0 ? n : 1));
                r->alignmentLength = n;
            } else {
                r->alignment = NULL; r->alignmentLength = 0;
                r->startLocationQuery = r->startLocationTarget = -1;
                status = -1;
            }
            free(rt);
        }
        free(rq); free(rp);
    } else {
        for (int i = 0; i < N; i++) {
            results[i]->alignment = NULL;
            results[i]->alignmentLength = -1;
            results[i]->startLocationQuery = -1;
            results[i]->startLocationTarget = -1;
        }
    }
    return status < 0 ? 0 : status;
}
