// deflate.cuh -- raw-deflate compressed-size kernels (K3 of SURVEY.md 2.3), sm_100a.
//
// Reproduces the byte count of the reference's gzip.compress(b) (pairwise_ncd.py:74: zlib level 9,
// raw + 18) and zlib.compress(b) (pairwise_ncd.py:78: level 6, raw + 6) as produced by CPython over
// zlib 1.3 with memLevel 8, windowBits 15, default strategy.  Only bit COUNTS are produced.
//
// zlib's deflate_slow is a serial loop whose cost on DNA is the hash-chain walk (hundreds of
// candidates per position).  The GPU design (DESIGN.md "deflate") separates what is parallel from what
// is serial:
//
//   1. every position of a stream is inserted into the hash chains whatever the parse does, so
//      "longest_match at position i" is a pure function of the bytes: F(i) = (length, distance) of the
//      first longest candidate among the K most recent same-hash positions within MAX_DIST.  It is
//      computed for ALL positions in parallel (dfl_match_kernel), one thread per position, candidates
//      enumerated from a per-sequence index sorted by (hash, position) instead of a linked list;
//   2. F of a sequence is the same in every stream that contains it, except near the x|y boundary:
//      F_x(p) holds for p <= len(x)-258, F_y(q) for q >= 32507 (window entirely inside y).  It is computed
//      once per SEQUENCE; each pair job only recomputes the junction (<= 257 + 32768 positions);
//   3. what remains serial per stream is the lazy-evaluation state machine over F (one table read per
//      step) plus the Huffman cost of each 16383-symbol block; the parse of the x part is shared through a
//      per-x checkpoint taken at the junction start, and the parse of the y part -- once it has
//      synchronised with the parse of y alone, a few symbols after the junction -- is taken from the
//      recorded symbol stream of y (cumulative histograms give each block's symbol counts): see
//      "canonical symbol stream" below.  A pair stream then costs its junction plus ~34 tree constructions;
//   4. the 3-byte hash chain itself is rarely walked: a second index on a hash of 6 bytes finds the
//      handful of candidates that can still matter (dfl_match_word, dfl_longest_k6), and the junction walk
//      of a position continues the walk the position had in y alone (dfl_longest_cont).  Every shortcut
//      is taken only where it is provably the same as the chain walk and has a switch for tests.
//
// Kernels, in the order a call runs them: dfl_radix_kernel / dfl_radix_scan_kernel / dfl_index_bounds_kernel /
// dfl_index_fill_kernel (indexes), dfl_head_kernel, dfl_tail6_kernel (head order, tail packs),
// dfl_match_kernel (F), dfl_prep_kernel (sequence alone: size, checkpoint, symbol stream),
// dfl_cum_chunk_kernel / dfl_cum_scan_kernel (cumulative histograms), then per batch of pair streams
// dfl_junction_kernel and dfl_parse_kernel.
//
// Rules restated from zlib 1.3 (each pinned by oracle/deflate_oracle.c against libz): hash =
// ((b0<<10)^(b1<<5)^b2)&0x7fff; a search happens only if the chain head is within MAX_DIST (32506) and is
// not stream position 0 (window index 0 doubles as NIL before the first slide); later candidates need
// distance < MAX_DIST; at most max_chain candidates (quartered when prev_length >= good_length); a
// candidate replaces the best only when strictly longer; the walk stops at nice_length; lengths are
// capped by min(258, bytes left); a length-3 match farther than 4096 is dropped.
#pragma once
#include "../../include/snacc_b200.h"     // status codes (SNACC_ERR_TOO_LARGE)
#include "common.cuh"
#include <algorithm>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

namespace snacc {

constexpr uint32_t DFL_WSIZE = 32768, DFL_MIN_MATCH = 3, DFL_MAX_MATCH = 258;
constexpr uint32_t DFL_MAX_DIST = DFL_WSIZE - (DFL_MAX_MATCH + DFL_MIN_MATCH + 1);   // 32506
constexpr uint32_t DFL_TOO_FAR = 4096, DFL_HASH = 32768;
constexpr uint32_t DFL_SYMS_PER_BLOCK = 16383;        // lit_bufsize - 1 at memLevel 8
constexpr uint32_t DFL_JY = 32768;                    // junction: first DFL_JY positions of y ...
constexpr uint32_t DFL_JX = 264;                      // ... and the last DFL_JX positions of x (>= 262: no end-of-input
                                                      // effect of x alone may precede the junction)
constexpr uint32_t DFL_QDIFF = 0x80000000u;           // F flag: the quartered-chain result differs

struct DflConfig { int good_length, max_lazy, nice_length, max_chain; };
SNACC_HD DflConfig dfl_config(int level)
{
    return level == 9 ? DflConfig{32, 258, 258, 4096} : DflConfig{8, 16, 128, 128};
}

SNACC_HD uint32_t dfl_hash3(uint32_t b0, uint32_t b1, uint32_t b2) { return ((b0 << 10) ^ (b1 << 5) ^ b2) & (DFL_HASH - 1); }

// per-sequence index: positions sorted by (hash, position); bstart has DFL_HASH + 1 entries
struct DflIndex {
    const uint32_t *order;
    const uint32_t *bstart;
};

// a stream (x, or x followed by y) with the indexes of its parts
struct DflStream {
    Stream s;
    DflIndex ix, iy;      // iy unused for singles
    bool pair;
};

SNACC_HD uint32_t dfl_hash_at(const Stream &s, uint32_t p)
{
    const uint32_t w = (uint32_t)ld64(s, p);
    return dfl_hash3(w & 0xff, (w >> 8) & 0xff, (w >> 16) & 0xff);
}

// number of entries of [lo, hi) of `order` that are < key
SNACC_HD uint32_t dfl_lower_bound(const uint32_t *order, uint32_t lo, uint32_t hi, uint32_t key)
{
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (SNACC_LDG(order + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Candidates of stream position p with hash h, most recent first, as stream positions (0xffffffff = end).
// Mirrors the order in which zlib's chain visits them: same-hash positions of y before p, then the two
// positions lx-1, lx-2 whose hash straddles the boundary, then the same-hash positions of x.
struct DflCandIter {
    const DflStream *d;
    uint32_t h, p;
    uint32_t stage;       // 0: y bucket, 1: lx-1, 2: lx-2, 3: x bucket, 4: end
    uint32_t ycur, ylo, xcur, xlo;
    // hint: index of p itself inside its own bucket when the caller already knows it (0xffffffff: search)
    SNACC_HD void init(const DflStream *ds, uint32_t pos, uint32_t hash, uint32_t hint)
    {
        d = ds; h = hash; p = pos;
        const uint32_t lx = d->s.lx;
        xlo = SNACC_LDG(d->ix.bstart + h);
        const uint32_t xhi = SNACC_LDG(d->ix.bstart + h + 1);
        ycur = ylo = 0;
        if (d->pair && p >= lx) {
            stage = 0;
            ylo = SNACC_LDG(d->iy.bstart + h);
            ycur = hint != 0xffffffffu ? hint : dfl_lower_bound(d->iy.order, ylo, SNACC_LDG(d->iy.bstart + h + 1), p - lx);
            xcur = xhi;
        } else if (d->pair && p + 2 >= lx) {
            // lx-2, lx-1: not in x's index (their hash needs bytes of y); every indexed position of x precedes them
            stage = p == lx - 1 ? 2 : 3;
            xcur = xhi;
        } else {
            stage = 3;
            xcur = hint != 0xffffffffu ? hint : dfl_lower_bound(d->ix.order, xlo, xhi, p);
        }
    }
    SNACC_HD uint32_t next()
    {
        const uint32_t lx = d->s.lx;
        for (;;) {
            if (stage == 0) {
                if (ycur > ylo) return lx + SNACC_LDG(d->iy.order + --ycur);
                stage = 1;
            } else if (stage == 1) {
                stage = 2;
                if (lx >= 1 && d->s.n - (lx - 1) >= 3 && dfl_hash_at(d->s, lx - 1) == h) return lx - 1;
            } else if (stage == 2) {
                stage = 3;
                if (lx >= 2 && d->s.n - (lx - 2) >= 3 && dfl_hash_at(d->s, lx - 2) == h) return lx - 2;
            } else if (stage == 3) {
                if (xcur > xlo) return SNACC_LDG(d->ix.order + --xcur);
                stage = 4;
            } else {
                return 0xffffffffu;
            }
        }
    }
};

// common prefix length of stream[a..] and stream[b..] (b < a), at most maxcmp
SNACC_HD uint32_t dfl_match_len(const Stream &s, uint32_t a, uint32_t b, uint32_t maxcmp)
{
    uint32_t len = 0;
    while (len < maxcmp) {
        const uint64_t d = ld64(s, a + len) ^ ld64(s, b + len);
        if (d) { len += (uint32_t)(SNACC_FFS64(d) - 1) >> 3; break; }
        len += 8;
    }
    return len < maxcmp ? len : maxcmp;
}

// base of zlib's window at a loop top with this strstart when input is still plentiful (oracle
// fill_window): the first slide happens at the first loop top >= 65275, then one every 32768 positions
SNACC_HD uint32_t dfl_window_base(uint32_t strstart)
{
    return strstart < 65275u ? 0u : DFL_WSIZE * ((strstart - 65275u) / DFL_WSIZE + 1);
}

// longest_match over the first `chain` candidates; returns (len << 16) | dist, 0 when there is no match of
// 3+ bytes (or no search at all).  `base`: window base at this loop top (positions <= base are NIL).  When
// `quarter` is non-null it also receives the result restricted to the first chain/4 candidates.
// `visit` (optional) receives how the walk went: number of candidates visited, DFL_V_NICE when it stopped at
// nice_length, DFL_V_HEADFAR when there was no search because the chain head is farther than MAX_DIST.
constexpr uint32_t DFL_V_COUNT = 0x1fffu, DFL_V_HEADFAR = 0x4000u, DFL_V_NICE = 0x8000u;
SNACC_HD uint32_t dfl_longest(const DflStream &d, uint32_t p, uint32_t base, uint32_t chain, uint32_t nice, uint32_t hint,
                              uint32_t *quarter, uint32_t *visit = nullptr)
{
    const Stream &s = d.s;
    if (quarter) *quarter = 0;
    if (visit) *visit = 0;
    if (s.n - p < DFL_MIN_MATCH) return 0;                 // the string at p is not even inserted
    const uint32_t maxcmp = tmin(DFL_MAX_MATCH, s.n - p);
    const uint32_t nice_match = tmin(nice, maxcmp);
    const uint32_t h = dfl_hash_at(s, p);
    DflCandIter it;
    it.init(&d, p, h, hint);
    uint32_t c = it.next();
    // chain head: must exist, not be NIL and be within MAX_DIST
    if (c == 0xffffffffu || c <= base) return 0;
    if (p - c > DFL_MAX_DIST) { if (visit) *visit = DFL_V_HEADFAR; return 0; }
    const uint32_t limit = (p - base > DFL_MAX_DIST) ? p - DFL_MAX_DIST : base;
    const uint64_t scan = ld64(s, p);
    uint32_t best = 2, bdist = 0, qbest = 0;
    const uint32_t qcount = chain >> 2;
    uint32_t count = 0;
    bool nice_stop = false;
    for (;;) {
        // quick test on the first 8 bytes, full compare only when they all agree
        const uint64_t x = scan ^ ld64(s, c);
        uint32_t len = x ? (uint32_t)(SNACC_FFS64(x) - 1) >> 3 : 8 + dfl_match_len(s, p + 8, c + 8, maxcmp > 8 ? maxcmp - 8 : 0);
        if (len > maxcmp) len = maxcmp;
        if (len > best) {
            best = len; bdist = p - c;
            if (len >= nice_match) { ++count; nice_stop = true; break; }
        }
        ++count;
        if (count == qcount) qbest = best > 2 ? (best << 16) | bdist : 0;
        if (count >= chain) break;
        c = it.next();
        if (c == 0xffffffffu || c <= limit) break;
    }
    const uint32_t full = best > 2 ? (best << 16) | bdist : 0;
    if (quarter) *quarter = count <= qcount ? full : qbest;
    if (visit) *visit = count | (nice_stop ? DFL_V_NICE : 0u);
    return full;
}

// longest_match of a position p = lx + q in the head of y of a pair stream, continued from the walk that
// the same position had in y ALONE (f_s = its F word, visit = how that walk went, q_s = its quartered result
// when q_known).  For q < DFL_JY the candidates inside y are visited in the same order, with the same
// distance rules, in both streams -- except y's position 0, which is NIL in y alone and an ordinary
// candidate here -- so the walk only has to go on where the other one ran out of y: position 0 of y, the
// two positions whose hash straddles the boundary, then x's bucket.  Returns the F word (QDIFF flag set
// when the quartered result differs or cannot be told without a second walk); *quarter = quartered result
// (exact whenever q_known).
SNACC_HD uint32_t dfl_longest_cont(const DflStream &d, uint32_t p, uint32_t chain, uint32_t nice, uint32_t f_s, uint32_t visit,
                                   bool q_known, uint32_t q_s, uint32_t *quarter)
{
    const Stream &s = d.s;
    const bool flag_s = (f_s & DFL_QDIFF) != 0;
    f_s &= ~DFL_QDIFF;
    if (!q_known && !flag_s) { q_known = true; q_s = f_s; }
    if (quarter) *quarter = 0;
    if (s.n - p < DFL_MIN_MATCH) return 0;
    uint32_t count = visit & DFL_V_COUNT;
    const uint32_t qcount = chain >> 2;
    if ((visit & (DFL_V_NICE | DFL_V_HEADFAR)) || count >= chain) {       // the walk ended inside y: nothing changes
        if (quarter) *quarter = q_known ? q_s : 0;
        return f_s | (flag_s ? DFL_QDIFF : 0u);
    }
    const uint32_t lx = s.lx, base = dfl_window_base(p);
    const uint32_t maxcmp = tmin(DFL_MAX_MATCH, s.n - p);
    const uint32_t nice_match = tmin(nice, maxcmp);
    const uint32_t h = dfl_hash_at(s, p);
    DflCandIter it;
    it.d = &d; it.h = h; it.p = p; it.stage = 0;
    it.ylo = SNACC_LDG(d.iy.bstart + h);
    const uint32_t yhi = SNACC_LDG(d.iy.bstart + h + 1);
    it.ycur = (p > lx && yhi > it.ylo && SNACC_LDG(d.iy.order + it.ylo) == 0) ? it.ylo + 1 : it.ylo;   // y's position 0
    it.xlo = SNACC_LDG(d.ix.bstart + h);
    it.xcur = SNACC_LDG(d.ix.bstart + h + 1);
    const uint32_t limit = (p - base > DFL_MAX_DIST) ? p - DFL_MAX_DIST : base;
    uint32_t best = (f_s >> 16) ? (f_s >> 16) : 2, bdist = f_s & 0xffff;
    bool q_fixed = count >= qcount;                  // the quartered result was settled inside y
    uint32_t qbest = q_fixed && q_known ? q_s : 0;
    bool q_lost = q_fixed && !q_known;
    uint32_t c = it.next();
    bool stop;
    if (count == 0) stop = c == 0xffffffffu || c <= base || p - c > DFL_MAX_DIST;   // this candidate is the chain head
    else stop = c == 0xffffffffu || c <= limit;
    if (!stop) {
        const uint64_t scan = ld64(s, p);
        // one candidate; `over` when the walk has ended
#define DFL_VISIT(c_) do {                                                                                          \
            const uint64_t x_ = scan ^ ld64(s, (c_));                                                               \
            uint32_t len_ = x_ ? (uint32_t)(SNACC_FFS64(x_) - 1) >> 3                                                \
                               : 8 + dfl_match_len(s, p + 8, (c_) + 8, maxcmp > 8 ? maxcmp - 8 : 0);                \
            if (len_ > maxcmp) len_ = maxcmp;                                                                       \
            if (len_ > best) {                                                                                      \
                best = len_; bdist = p - (c_);                                                                      \
                if (len_ >= nice_match) { ++count; over = true; break; }                                            \
            }                                                                                                       \
            ++count;                                                                                                \
            if (count == qcount) qbest = best > 2 ? (best << 16) | bdist : 0;                                       \
            if (count >= chain) over = true;                                                                        \
        } while (0)
        bool over = false;
        // y's position 0 and the two straddling positions through the general iterator ...
        while (!over && it.stage < 3) {
            DFL_VISIT(c);
            if (over) break;
            c = it.next();
            if (c == 0xffffffffu || c <= limit) { over = true; break; }
            if (it.stage == 3) break;              // c is the first candidate out of x's bucket
        }
        // ... then x's bucket, most recent first, in a tight loop (the lanes of a warp walk it together)
        if (!over) {
            const uint32_t *ox = d.ix.order;
            uint32_t k = it.xcur;                   // c == ox[k] has been fetched already
            for (;;) {
                DFL_VISIT(c);
                if (over || k == it.xlo) break;
                c = SNACC_LDG(ox + --k);
                if (c <= limit) break;
            }
        }
#undef DFL_VISIT
    }
    const uint32_t full = best > 2 ? (best << 16) | bdist : 0;
    const uint32_t qres = count <= qcount ? full : qbest;
    if (quarter) *quarter = qres;
    const bool differs = count <= qcount ? false : (q_lost ? true : qbest != full);
    return full | (differs ? DFL_QDIFF : 0u);
}

// ---- 6-byte index of a sequence's tail -----------------------------------------------------------
// When the walk of a head position of y leaves y with a best match of 5+ bytes -- or when x holds a candidate of
// 6+ bytes at all -- only candidates of x that agree on 6+ bytes decide the result, and the chain visits them in
// the same (most recent first) order whether or not the shorter ones are skipped.  Those candidates are found through a second index of the last
// 32 KiB of every sequence, keyed by a hash of 6 bytes (a handful of entries per bucket on DNA instead of ~500
// in the 3-byte bucket).  The shortcut is only taken when no chain limit can bind: the walk inside y visited
// cnt candidates, x's whole 3-byte bucket holds at most U inside any window, and cnt + 3 + U stays below
// max_chain / 4 -- then neither max_chain nor the quartered chain cuts the walk short and the visit count does
// not matter.  Everything else takes dfl_longest_cont.
constexpr uint32_t DFL_T6 = 32768;                    // tail positions indexed: [max(0, len - DFL_T6), len - 6]
constexpr uint32_t DFL_H6 = 8192;                     // buckets of the 6-byte index
SNACC_HD uint32_t dfl_hash6(uint64_t v) { return (uint32_t)(((v & 0xffffffffffffull) * 0x9E3779B97F4A7C15ull) >> 51); }
struct DflTail6 {
    const uint16_t *order;      // offsets from t0, sorted by (hash6, position)
    const uint16_t *start;      // DFL_H6 + 1 bucket starts
    uint32_t t0;                // stream position of offset 0
};
SNACC_HD uint32_t dfl_tail6_t0(uint32_t len) { return len > DFL_T6 ? len - DFL_T6 : 0; }
SNACC_HD uint32_t dfl_tail6_count(uint32_t len) { return len >= 6 ? len - 5 - dfl_tail6_t0(len) : 0; }
SNACC_HD uint32_t dfl_tail3_from(uint32_t len) { return len > DFL_MAX_DIST - 1 ? len - (DFL_MAX_DIST - 1) : 0; }  // first x position any head walk can reach

// preconditions (checked by dfl_junction_word): the walk inside y started, did not stop at nice_length, and no
// chain limit can bind; the result only stands when it is 6+ bytes long or y alone had found 5+ bytes
SNACC_HD uint32_t dfl_longest_k6(const DflStream &d, uint32_t p, uint32_t nice, uint32_t f_s, const DflTail6 &t6,
                                 const uint64_t *edge = nullptr)   // edge[k] = ld64(s, lx - k), k = 0..5, when the caller has them
{
    const Stream &s = d.s;
    const uint32_t lx = s.lx, base = dfl_window_base(p);
    const uint32_t maxcmp = tmin(DFL_MAX_MATCH, s.n - p);
    const uint32_t nice_match = tmin(nice, maxcmp);
    const uint32_t limit = (p - base > DFL_MAX_DIST) ? p - DFL_MAX_DIST : base;
    uint32_t best = (f_s >> 16) ? (f_s >> 16) : 2, bdist = f_s & 0xffff;
    const uint64_t scan = ld64(s, p);
    bool over = false;
#define DFL_K6_VISIT(c_) DFL_K6_VISIT8(c_, ld64(s, (c_)))
#define DFL_K6_VISIT8(c_, bytes_) do {                                                                              \
        const uint64_t x_ = scan ^ (bytes_);                                                                        \
        uint32_t len_ = x_ ? (uint32_t)(SNACC_FFS64(x_) - 1) >> 3                                                    \
                           : 8 + dfl_match_len(s, p + 8, (c_) + 8, maxcmp > 8 ? maxcmp - 8 : 0);                    \
        if (len_ > maxcmp) len_ = maxcmp;                                                                           \
        if (len_ > best) { best = len_; bdist = p - (c_); if (len_ >= nice_match) over = true; }                    \
    } while (0)
    // y's position 0 (p > lx), then lx-1 .. lx-5: the positions of x whose 6 bytes run into y
    for (uint32_t k = p > lx ? 0u : 1u; k <= 5 && !over; ++k) {
        if (lx < k) break;
        const uint32_t c = lx - k;
        if (c <= limit) { over = true; break; }
        if (edge) {
            // a candidate only counts from 6 equal bytes on: most positions are done with one compare
            if (((scan ^ edge[k]) & 0xffffffffffffull) == 0) DFL_K6_VISIT8(c, edge[k]);
        } else {
            DFL_K6_VISIT(c);
        }
    }
    if (!over) {
        const uint32_t h6 = dfl_hash6(scan);
        const uint32_t lo = SNACC_LDG(t6.start + h6);
        uint32_t k = SNACC_LDG(t6.start + h6 + 1);
        while (k > lo) {
            const uint32_t c = t6.t0 + SNACC_LDG(t6.order + --k);
            if (c <= limit) break;
            DFL_K6_VISIT(c);
            if (over) break;
        }
    }
#undef DFL_K6_VISIT
#undef DFL_K6_VISIT8
    return best > 2 ? (best << 16) | bdist : 0;
}

// junction F word of head position p = lx + q of a pair stream (see dfl_longest_cont for the arguments);
// tail_cnt: per 3-byte bucket of x, the entries at or after dfl_tail3_from(lx); t6 == null: no shortcut
SNACC_HD uint32_t dfl_junction_word(const DflStream &d, uint32_t p, const DflConfig &cfg, uint32_t f_s, uint32_t visit, bool q_known,
                                    uint32_t q_s, const DflTail6 *t6, const uint16_t *tail_cnt, uint32_t *quarter,
                                    const uint64_t *edge = nullptr)
{
    const uint32_t cnt = visit & DFL_V_COUNT, f = f_s & ~DFL_QDIFF, chain = (uint32_t)cfg.max_chain;
    if (t6 && !(visit & (DFL_V_NICE | DFL_V_HEADFAR)) && d.s.n - p >= 6) {
        const Stream &s = d.s;
        const uint32_t h = dfl_hash_at(s, p), lx = s.lx;
        bool ok = cnt + 3 + SNACC_LDG(tail_cnt + h) < (chain >> 2);
        if (ok && cnt == 0) {
            // the walk never started inside y: the first chain member met from here on is the chain head and has its
            // own test (not NIL, at most MAX_DIST away -- one byte farther than any later candidate may be)
            uint32_t head = 0xffffffffu;
            if (p > lx && dfl_hash_at(s, lx) == h) head = lx;
            else if (lx >= 1 && s.n - (lx - 1) >= 3 && dfl_hash_at(s, lx - 1) == h) head = lx - 1;
            else if (lx >= 2 && s.n - (lx - 2) >= 3 && dfl_hash_at(s, lx - 2) == h) head = lx - 2;
            else {
                const uint32_t xlo = SNACC_LDG(d.ix.bstart + h), xhi = SNACC_LDG(d.ix.bstart + h + 1);
                if (xhi > xlo) head = SNACC_LDG(d.ix.order + xhi - 1);
            }
            if (head == 0xffffffffu || head <= dfl_window_base(p) || p - head > DFL_MAX_DIST) {
                if (quarter) *quarter = 0;
                return 0;                                   // no search at all
            }
            ok = p - head != DFL_MAX_DIST;
        }
        if (ok) {
            // the 6-byte walk sees every candidate of 6+ bytes in chain order: when it ends with such a match, or when
            // y alone had already found 5+ bytes, no candidate it skipped can have mattered
            const uint32_t w = dfl_longest_k6(d, p, (uint32_t)cfg.nice_length, f, *t6, edge);
            if ((w >> 16) >= 6 || (f >> 16) >= 5) {
                if (quarter) *quarter = w;
                return w;
            }
        }
    }
    return dfl_longest_cont(d, p, chain, (uint32_t)cfg.nice_length, f_s, visit, q_known, q_s, quarter);
}

// F word of a position: the full-chain result, flagged when the quartered chain gives something else
SNACC_HD uint32_t dfl_f_word(const DflStream &d, uint32_t p, const DflConfig &c, uint32_t hint, uint32_t *qword,
                             uint32_t *visit = nullptr)
{
    uint32_t q;
    const uint32_t f = dfl_longest(d, p, dfl_window_base(p), (uint32_t)c.max_chain, (uint32_t)c.nice_length, hint, &q, visit);
    if (qword) *qword = q;
    return q != f ? f | DFL_QDIFF : f;
}

// ---- 6-byte index of a whole sequence (transient: only dfl_match_kernel reads it) ---------------------
// The same argument as for the junction gives F of a sequence alone without walking its 3-byte chain: when fewer
// than max_chain / 4 chain members lie inside the window (one index lookup: the member max_chain / 4 places
// back is out of reach), no limit binds, and if the candidates that share 6 bytes with p -- visited most recent
// first -- yield a match of 6+ bytes, that match is what the full walk would have returned.  Otherwise (no such
// candidate, head of the sequence, level 6 where the chain limit binds all the time) the full walk runs.
SNACC_HD uint32_t dfl_hash6w(uint64_t v) { return (uint32_t)(((v & 0xffffffffffffull) * 0x9E3779B97F4A7C15ull) >> 49); }   // 15 bits
struct DflIndex6 { const uint32_t *order6, *bstart6; };   // positions [0, len - 5) sorted by (hash6w, position)

SNACC_HD uint32_t dfl_match_word(const DflStream &d, uint32_t p, const DflConfig &cfg, uint32_t k, const DflIndex6 *i6,
                                 uint32_t *qword, uint32_t *visit)
{
    const Stream &s = d.s;
    if (i6 && p >= DFL_JY && s.n - p >= 6) {
        const uint32_t chain = (uint32_t)cfg.max_chain, qcount = chain >> 2;
        const uint32_t h = dfl_hash_at(s, p);
        const uint32_t lo3 = SNACC_LDG(d.ix.bstart + h);
        const uint32_t base = dfl_window_base(p);
        const uint32_t limit = (p - base > DFL_MAX_DIST) ? p - DFL_MAX_DIST : base;
        // chain head (the most recent member): no search at all when it is missing, NIL or too far
        bool fast = k > lo3;
        if (fast) {
            const uint32_t ch = SNACC_LDG(d.ix.order + k - 1);
            if (ch <= base || p - ch > DFL_MAX_DIST) { if (qword) *qword = 0; if (visit) *visit = 0; return 0; }
            fast = k - lo3 < qcount || SNACC_LDG(d.ix.order + k - qcount) <= limit;     // fewer than qcount members in reach
        }
        if (fast) {
            const uint32_t maxcmp = tmin(DFL_MAX_MATCH, s.n - p);
            const uint32_t nice_match = tmin((uint32_t)cfg.nice_length, maxcmp);
            const uint64_t scan = ld64(s, p);
            const uint32_t h6 = dfl_hash6w(scan);
            const uint32_t lo6 = SNACC_LDG(i6->bstart6 + h6);
            uint32_t j = dfl_lower_bound(i6->order6, lo6, SNACC_LDG(i6->bstart6 + h6 + 1), p);
            uint32_t best = 2, bdist = 0;
            while (j > lo6) {
                const uint32_t c = SNACC_LDG(i6->order6 + --j);
                if (c <= limit) break;
                const uint64_t x = scan ^ ld64(s, c);
                uint32_t len = x ? (uint32_t)(SNACC_FFS64(x) - 1) >> 3 : 8 + dfl_match_len(s, p + 8, c + 8, maxcmp > 8 ? maxcmp - 8 : 0);
                if (len > maxcmp) len = maxcmp;
                if (len > best) { best = len; bdist = p - c; if (len >= nice_match) break; }
            }
            if (best >= 6) {
                const uint32_t w = (best << 16) | bdist;
                if (qword) *qword = w;
                if (visit) *visit = 0;               // only kept for p < DFL_JY, which never comes here
                return w;
            }
        }
    }
    return dfl_f_word(d, p, cfg, k, qword, visit);
}

// ------------------------------------------------------------------------------------------------
// Huffman block cost (trees.c: _tr_flush_block and helpers), bit counts only
// ------------------------------------------------------------------------------------------------
constexpr int DFL_L_CODES = 286, DFL_D_CODES = 30, DFL_BL_CODES = 19, DFL_HEAP = 2 * DFL_L_CODES + 1;

struct DflNode { uint16_t freq, dad, len; };

struct DflTrees {                      // scratch of one block flush
    DflNode ltree[DFL_HEAP];
    DflNode dtree[2 * DFL_D_CODES + 1];
    DflNode bltree[2 * DFL_BL_CODES + 1];
    int32_t heap[DFL_HEAP];
    uint8_t depth[DFL_HEAP];
    uint16_t bl_count[16];
    int32_t heap_len, heap_max;
    uint64_t opt_len, static_len;
};

SNACC_HD int dfl_extra_lbits(int code) { return code < 8 ? 0 : code == 28 ? 0 : (code - 4) >> 2; }
SNACC_HD int dfl_extra_dbits(int code) { return code < 4 ? 0 : (code - 2) >> 1; }
SNACC_HD int dfl_static_llen(int n) { return n <= 143 ? 8 : n <= 255 ? 9 : n <= 279 ? 7 : 8; }
SNACC_HD int dfl_length_code(uint32_t len_minus3)
{
    // trees.c length_code[]: codes 0..27 cover 2^extra lengths each, 258 has its own code 28
    if (len_minus3 == 255) return 28;
    if (len_minus3 < 8) return (int)len_minus3;
    const int k = 31 - (int)
#ifdef __CUDA_ARCH__
        __clz((int)len_minus3);
#else
        __builtin_clz(len_minus3);
#endif
    // len_minus3 in [2^k, 2^(k+1)): extra bits k-2, four codes per k
    return 4 * (k - 1) + (int)((len_minus3 >> (k - 2)) & 3);
}
SNACC_HD int dfl_dist_code(uint32_t d /* distance - 1 */)
{
    if (d < 4) return (int)d;
    const int k = 31 - (int)
#ifdef __CUDA_ARCH__
        __clz((int)d);
#else
        __builtin_clz(d);
#endif
    return 2 * k + (int)((d >> (k - 1)) & 1);
}

struct DflTreeDesc { DflNode *tree; int max_code; int kind; int elems; int max_length; };   // kind 0: literal/length, 1: distance, 2: bit lengths

SNACC_HD bool dfl_smaller(const DflTrees &t, const DflNode *tree, int n, int m)
{
    return tree[n].freq < tree[m].freq || (tree[n].freq == tree[m].freq && t.depth[n] <= t.depth[m]);
}

SNACC_HD void dfl_pqdownheap(DflTrees &t, DflNode *tree, int k)
{
    const int v = t.heap[k];
    int j = k << 1;
    while (j <= t.heap_len) {
        if (j < t.heap_len && dfl_smaller(t, tree, t.heap[j + 1], t.heap[j])) j++;
        if (dfl_smaller(t, tree, v, t.heap[j])) break;
        t.heap[k] = t.heap[j]; k = j;
        j <<= 1;
    }
    t.heap[k] = v;
}

SNACC_HD int dfl_xbits(const DflTreeDesc &d, int n)
{
    if (d.kind == 0) return n >= 257 ? dfl_extra_lbits(n - 257) : 0;
    if (d.kind == 1) return dfl_extra_dbits(n);
    return n == 16 ? 2 : n == 17 ? 3 : n == 18 ? 7 : 0;
}
SNACC_HD int dfl_slen(const DflTreeDesc &d, int n) { return d.kind == 0 ? dfl_static_llen(n) : 5; }

static __host__ __device__ void dfl_gen_bitlen(DflTrees &t, DflTreeDesc &desc)
{
    DflNode *tree = desc.tree;
    const int max_code = desc.max_code, max_length = desc.max_length;
    int h, n, m, bits, overflow = 0;
    for (bits = 0; bits <= 15; bits++) t.bl_count[bits] = 0;
    tree[t.heap[t.heap_max]].len = 0;
    for (h = t.heap_max + 1; h < DFL_HEAP; h++) {
        n = t.heap[h];
        bits = tree[tree[n].dad].len + 1;
        if (bits > max_length) bits = max_length, overflow++;
        tree[n].len = (uint16_t)bits;
        if (n > max_code) continue;
        t.bl_count[bits]++;
        const int xbits = dfl_xbits(desc, n);
        const uint64_t f = tree[n].freq;
        t.opt_len += f * (unsigned)(bits + xbits);
        if (desc.kind != 2) t.static_len += f * (unsigned)(dfl_slen(desc, n) + xbits);
    }
    if (overflow == 0) return;
    do {
        bits = max_length - 1;
        while (t.bl_count[bits] == 0) bits--;
        t.bl_count[bits]--;
        t.bl_count[bits + 1] += 2;
        t.bl_count[max_length]--;
        overflow -= 2;
    } while (overflow > 0);
    for (bits = max_length; bits != 0; bits--) {
        n = t.bl_count[bits];
        while (n != 0) {
            m = t.heap[--h];
            if (m > max_code) continue;
            if ((unsigned)tree[m].len != (unsigned)bits) {
                t.opt_len += ((uint64_t)bits - tree[m].len) * tree[m].freq;
                tree[m].len = (uint16_t)bits;
            }
            n--;
        }
    }
}

static __host__ __device__ void dfl_build_tree(DflTrees &t, DflTreeDesc &desc)
{
    DflNode *tree = desc.tree;
    const int elems = desc.elems;
    int n, m, max_code = -1, node;
    t.heap_len = 0; t.heap_max = DFL_HEAP;
    for (n = 0; n < elems; n++) {
        if (tree[n].freq != 0) { t.heap[++t.heap_len] = max_code = n; t.depth[n] = 0; }
        else tree[n].len = 0;
    }
    while (t.heap_len < 2) {
        node = t.heap[++t.heap_len] = (max_code < 2 ? ++max_code : 0);
        tree[node].freq = 1;
        t.depth[node] = 0;
        t.opt_len--;
        if (desc.kind != 2) t.static_len -= (uint64_t)dfl_slen(desc, node);
    }
    desc.max_code = max_code;
    for (n = t.heap_len / 2; n >= 1; n--) dfl_pqdownheap(t, tree, n);
    node = elems;
    do {
        n = t.heap[1];
        t.heap[1] = t.heap[t.heap_len--];
        dfl_pqdownheap(t, tree, 1);
        m = t.heap[1];
        t.heap[--t.heap_max] = n;
        t.heap[--t.heap_max] = m;
        tree[node].freq = (uint16_t)(tree[n].freq + tree[m].freq);
        t.depth[node] = (uint8_t)((t.depth[n] >= t.depth[m] ? t.depth[n] : t.depth[m]) + 1);
        tree[n].dad = tree[m].dad = (uint16_t)node;
        t.heap[1] = node++;
        dfl_pqdownheap(t, tree, 1);
    } while (t.heap_len >= 2);
    t.heap[--t.heap_max] = t.heap[1];
    dfl_gen_bitlen(t, desc);
}

static __host__ __device__ void dfl_scan_tree(DflTrees &t, DflNode *tree, int max_code)
{
    int n, prevlen = -1, curlen, nextlen = tree[0].len, count = 0, max_count = 7, min_count = 4;
    if (nextlen == 0) max_count = 138, min_count = 3;
    tree[max_code + 1].len = 0xffff;
    for (n = 0; n <= max_code; n++) {
        curlen = nextlen; nextlen = tree[n + 1].len;
        if (++count < max_count && curlen == nextlen) continue;
        else if (count < min_count) t.bltree[curlen].freq += (uint16_t)count;
        else if (curlen != 0) {
            if (curlen != prevlen) t.bltree[curlen].freq++;
            t.bltree[16].freq++;
        } else if (count <= 10) t.bltree[17].freq++;
        else t.bltree[18].freq++;
        count = 0; prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

// Bits of one block given its symbol frequencies (lfreq[286] incl. END_BLOCK = 1, dfreq[30]); `bits` is
// the running total (the stored form aligns it).
static __host__ __device__ void dfl_flush_block(DflTrees &t, const uint16_t *lfreq, int lstride, const uint16_t *dfreq,
                                                int dstride, uint64_t stored_len, bool can_store, bool last, uint64_t &bits,
                                                bool *stored_cand = nullptr)
{
    const uint8_t bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (int n = 0; n < DFL_L_CODES; n++) t.ltree[n].freq = lfreq[n * lstride];
    for (int n = 0; n < DFL_D_CODES; n++) t.dtree[n].freq = dfreq[n * dstride];
    for (int n = 0; n < DFL_BL_CODES; n++) t.bltree[n].freq = 0;
    t.opt_len = t.static_len = 0;
    DflTreeDesc ld{t.ltree, 0, 0, DFL_L_CODES, 15}, dd{t.dtree, 0, 1, DFL_D_CODES, 15}, bd{t.bltree, 0, 2, DFL_BL_CODES, 7};
    dfl_build_tree(t, ld);
    dfl_build_tree(t, dd);
    dfl_scan_tree(t, t.ltree, ld.max_code);
    dfl_scan_tree(t, t.dtree, dd.max_code);
    dfl_build_tree(t, bd);
    int max_blindex;
    for (max_blindex = DFL_BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (t.bltree[bl_order[max_blindex]].len != 0) break;
    t.opt_len += 3 * ((uint64_t)max_blindex + 1) + 5 + 5 + 4;
    uint64_t opt_lenb = (t.opt_len + 3 + 7) >> 3;
    const uint64_t static_lenb = (t.static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    if (stored_cand) *stored_cand = stored_len + 4 <= opt_lenb;    // the stored form would win if the window still holds the block
    if (stored_len + 4 <= opt_lenb && can_store) {
        bits += 3;
        bits = (bits + 7) & ~7ull;
        bits += 32 + 8 * stored_len;
    } else if (static_lenb == opt_lenb) {
        bits += 3 + t.static_len;
    } else {
        bits += 3 + t.opt_len;
    }
    if (last) bits = (bits + 7) & ~7ull;
}

// ---- the same block cost on compacted trees ------------------------------------------------------
// A pair stream costs ~34 blocks and zlib's tree construction is a chain of dependent loads and stores; with the
// scratch of one thread at 6.5 KB (DflTrees) it lives in global memory and every step is a DRAM/L2 round trip.
// build_tree never looks at symbol numbers, only at frequencies, depths and heap positions, so it can run on the
// NONZERO symbols alone, renumbered in order (leaves 0..L-1, internal nodes from L): same heap, same tree, same code
// lengths.  On DNA a block uses ~25 literal/length codes and ~28 distance codes, so the scratch shrinks to under
// 1 KB per thread and fits shared memory.  Blocks with more than DFL_C_LEAVES codes in a tree, or fewer than two
// (zlib then invents symbols by number), take dfl_flush_block.
constexpr int DFL_C_LEAVES = 48, DFL_C_NODES = 2 * DFL_C_LEAVES;
struct DflCompactTrees {
    uint16_t freq[DFL_C_NODES];
    uint8_t dad[DFL_C_NODES], len[DFL_C_NODES], depth[DFL_C_NODES];
    uint8_t heap[DFL_C_NODES + 4];
    uint16_t map[DFL_C_LEAVES];                           // symbol of each leaf of the tree under construction
    uint16_t lmap[DFL_C_LEAVES]; uint8_t llen[DFL_C_LEAVES];   // finished literal/length tree
    uint8_t dmap[DFL_D_CODES + 2], dlen[DFL_D_CODES + 2];      // finished distance tree
    uint16_t blfreq[DFL_BL_CODES + 1];
    uint16_t bl_count[16];
    uint32_t pad_[2];                                     // sizeof = 964: an odd number of words, so the scratches of the
};                                                        // threads of a warp fall into different banks
static_assert(sizeof(DflCompactTrees) % 8 == 4, "DflCompactTrees: odd number of 32-bit words expected");

SNACC_HD bool dfl_c_smaller(const DflCompactTrees &t, int n, int m)
{
    return t.freq[n] < t.freq[m] || (t.freq[n] == t.freq[m] && t.depth[n] <= t.depth[m]);
}
SNACC_HD void dfl_c_downheap(DflCompactTrees &t, int heap_len, int k)
{
    const int v = t.heap[k];
    int j = k << 1;
    while (j <= heap_len) {
        if (j < heap_len && dfl_c_smaller(t, t.heap[j + 1], t.heap[j])) j++;
        if (dfl_c_smaller(t, v, t.heap[j])) break;
        t.heap[k] = t.heap[j]; k = j;
        j <<= 1;
    }
    t.heap[k] = (uint8_t)v;
}
// leaves 0..L-1 (freq, map) -> code lengths in len[0..L-1]; adds the tree's bits to opt_len / static_len
static __host__ __device__ void dfl_c_build(DflCompactTrees &t, int L, int kind, int max_length, uint64_t &opt_len, uint64_t &static_len)
{
    const int HS = 2 * L + 1;
    DflTreeDesc desc{nullptr, 0, kind, 0, max_length};
    int heap_len = 0, heap_max = HS;
    for (int n = 0; n < L; n++) { t.heap[++heap_len] = (uint8_t)n; t.depth[n] = 0; }
    for (int n = heap_len / 2; n >= 1; n--) dfl_c_downheap(t, heap_len, n);
    int node = L;
    do {
        const int n = t.heap[1];
        t.heap[1] = t.heap[heap_len--];
        dfl_c_downheap(t, heap_len, 1);
        const int m = t.heap[1];
        t.heap[--heap_max] = (uint8_t)n;
        t.heap[--heap_max] = (uint8_t)m;
        t.freq[node] = (uint16_t)(t.freq[n] + t.freq[m]);
        t.depth[node] = (uint8_t)((t.depth[n] >= t.depth[m] ? t.depth[n] : t.depth[m]) + 1);
        t.dad[n] = t.dad[m] = (uint8_t)node;
        t.heap[1] = (uint8_t)node++;
        dfl_c_downheap(t, heap_len, 1);
    } while (heap_len >= 2);
    t.heap[--heap_max] = t.heap[1];
    // gen_bitlen
    int h, bits, overflow = 0;
    for (bits = 0; bits <= 15; bits++) t.bl_count[bits] = 0;
    t.len[t.heap[heap_max]] = 0;
    for (h = heap_max + 1; h < HS; h++) {
        const int n = t.heap[h];
        bits = t.len[t.dad[n]] + 1;
        if (bits > max_length) bits = max_length, overflow++;
        t.len[n] = (uint8_t)bits;
        if (n >= L) continue;                            // not a leaf
        t.bl_count[bits]++;
        const int sym = t.map[n];
        const int xbits = dfl_xbits(desc, sym);
        const uint64_t f = t.freq[n];
        opt_len += f * (unsigned)(bits + xbits);
        if (kind != 2) static_len += f * (unsigned)(dfl_slen(desc, sym) + xbits);
    }
    if (overflow == 0) return;
    do {
        bits = max_length - 1;
        while (t.bl_count[bits] == 0) bits--;
        t.bl_count[bits]--;
        t.bl_count[bits + 1] += 2;
        t.bl_count[max_length]--;
        overflow -= 2;
    } while (overflow > 0);
    for (bits = max_length; bits != 0; bits--) {
        int n = t.bl_count[bits];
        while (n != 0) {
            const int m = t.heap[--h];
            if (m >= L) continue;
            if ((int)t.len[m] != bits) {
                opt_len += (uint64_t)((int64_t)(bits - (int)t.len[m]) * (int64_t)t.freq[m]);
                t.len[m] = (uint8_t)bits;
            }
            n--;
        }
    }
}
// scan_tree over symbols 0..max_code of a finished tree given by its leaves (map ascending) and their lengths
template <class MapT>
static __host__ __device__ void dfl_c_scan(DflCompactTrees &t, const MapT *map, const uint8_t *len, int L, int max_code)
{
    int j = 0;
#define DFL_C_LEN(sym_) ((j < L && (int)map[j] == (sym_)) ? (int)len[j++] : 0)
    int prevlen = -1, curlen, nextlen = DFL_C_LEN(0), count = 0, max_count = 7, min_count = 4;
    if (nextlen == 0) max_count = 138, min_count = 3;
    for (int n = 0; n <= max_code; n++) {
        curlen = nextlen;
        nextlen = n + 1 <= max_code ? DFL_C_LEN(n + 1) : 0xffff;
        if (++count < max_count && curlen == nextlen) continue;
        else if (count < min_count) t.blfreq[curlen] += (uint16_t)count;
        else if (curlen != 0) {
            if (curlen != prevlen) t.blfreq[curlen]++;
            t.blfreq[16]++;
        } else if (count <= 10) t.blfreq[17]++;
        else t.blfreq[18]++;
        count = 0; prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
#undef DFL_C_LEN
}
// dfl_flush_block on compacted trees; false (nothing changed) when the block does not qualify
static __host__ __device__ bool dfl_flush_block_compact(DflCompactTrees &t, const uint16_t *lfreq, int lstride, const uint16_t *dfreq,
                                                        int dstride, uint64_t stored_len, bool can_store, bool last, uint64_t &bits,
                                                        bool *stored_cand)
{
    const uint8_t bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint64_t opt_len = 0, static_len = 0;
    int L = 0;
    for (int n = 0; n < DFL_L_CODES; n++) {
        const uint16_t f = lfreq[n * lstride];
        if (!f) continue;
        if (L == DFL_C_LEAVES) return false;
        t.freq[L] = f; t.map[L] = (uint16_t)n; L++;
    }
    if (L < 2) return false;
    int D = 0;
    for (int n = 0; n < DFL_D_CODES; n++) D += dfreq[n * dstride] != 0;
    if (D < 2) return false;
    const int lmax = t.map[L - 1], Ls = L;
    dfl_c_build(t, L, 0, 15, opt_len, static_len);
    for (int n = 0; n < L; n++) { t.lmap[n] = t.map[n]; t.llen[n] = t.len[n]; }
    L = 0;
    for (int n = 0; n < DFL_D_CODES; n++) {
        const uint16_t f = dfreq[n * dstride];
        if (f) { t.freq[L] = f; t.map[L] = (uint16_t)n; L++; }
    }
    const int dmax = t.map[L - 1], Ds = L;
    dfl_c_build(t, L, 1, 15, opt_len, static_len);
    for (int n = 0; n < L; n++) { t.dmap[n] = (uint8_t)t.map[n]; t.dlen[n] = t.len[n]; }
    for (int n = 0; n < DFL_BL_CODES; n++) t.blfreq[n] = 0;
    dfl_c_scan(t, t.lmap, t.llen, Ls, lmax);
    dfl_c_scan(t, t.dmap, t.dlen, Ds, dmax);
    L = 0;
    for (int n = 0; n < DFL_BL_CODES; n++)
        if (t.blfreq[n]) { t.freq[L] = t.blfreq[n]; t.map[L] = (uint16_t)n; L++; }
    if (L < 2) return false;
    dfl_c_build(t, L, 2, 7, opt_len, static_len);
    // bit length of every bit-length code, by symbol (blfreq is free now)
    for (int n = 0; n < DFL_BL_CODES; n++) t.blfreq[n] = 0;
    for (int n = 0; n < L; n++) t.blfreq[t.map[n]] = t.len[n];
    int max_blindex;
    for (max_blindex = DFL_BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (t.blfreq[bl_order[max_blindex]] != 0) break;
    opt_len += 3 * ((uint64_t)max_blindex + 1) + 5 + 5 + 4;
    uint64_t opt_lenb = (opt_len + 3 + 7) >> 3;
    const uint64_t static_lenb = (static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    if (stored_cand) *stored_cand = stored_len + 4 <= opt_lenb;
    if (stored_len + 4 <= opt_lenb && can_store) {
        bits += 3;
        bits = (bits + 7) & ~7ull;
        bits += 32 + 8 * stored_len;
    } else if (static_lenb == opt_lenb) {
        bits += 3 + static_len;
    } else {
        bits += 3 + opt_len;
    }
    if (last) bits = (bits + 7) & ~7ull;
    return true;
}

// ------------------------------------------------------------------------------------------------
// canonical symbol stream of a sequence
// ------------------------------------------------------------------------------------------------
// deflate_slow's state right after it has emitted a match is just the position: match_available = 0,
// match_length = MIN_MATCH-1 (so prev_match is dead).  From such a loop top the symbols it emits are a pure
// function of F, and F_y(q) is the same in every stream that contains y once q >= DFL_JY.  So as soon as the
// parse of x.y stands, at y offset q >= DFL_JY, on a position where the parse of y ALONE also stood right
// after a match, the two emit the same symbols for the rest of y -- only the block boundaries (every 16383
// symbols, counted from wherever the pair stream's open block began) and the end-of-input window slide
// (a function of the absolute position) differ.  The parse of y alone is therefore recorded once per
// sequence: end offset and (length code, distance code) of every symbol, plus cumulative symbol
// histograms every DFL_CUM_G symbols.  A pair stream parses its junction serially, finds the
// synchronisation point (binary search in `end`), takes the histogram of each of its remaining blocks as
// a difference of two cumulative rows and only returns to the serial parser for the last DFL_TAIL bytes.
// A block for which zlib would consider the stored form (never on DNA) sends the job back to the full
// serial parse: whether that form is allowed depends on the window position, which the shortcut does not
// track.
constexpr uint32_t DFL_CUM_G = 256;                    // symbols per cumulative-histogram row
constexpr uint32_t DFL_CUM_W = 320;                    // row width: 286 literal/length + 30 distance counters, padded
constexpr uint32_t DFL_TAIL = 1024;                    // bytes of y always left to the serial parser (>= 262 + 258)
constexpr uint32_t DFL_CANON_MIN = DFL_JY + 4 * DFL_TAIL;   // shorter y: plain serial parse
constexpr uint32_t DFL_LIT = 31;                       // distance-code field of a literal
constexpr uint32_t DFL_NONE = 0xffffffffu;

struct DflRec {                        // where the parse of a sequence alone records its symbols
    uint32_t *end; uint16_t *code;     // end offset after the symbol; lcode | dcode << 9
    uint32_t cap, n;                   // n = DFL_NONE after an overflow
};
SNACC_HD void dfl_rec_emit(DflRec *r, uint32_t code, uint32_t end)
{
    if (!r || r->n == DFL_NONE) return;
    if (r->n >= r->cap) { r->n = DFL_NONE; return; }
    r->end[r->n] = end; r->code[r->n] = (uint16_t)code; r->n++;
}

struct DflCanon {
    const uint32_t *end; const uint16_t *code;
    const uint32_t *cum;               // row j: counts of the symbols [0, j * DFL_CUM_G)
    uint32_t n_sym;                    // 0: not available
};

// index of the canonical symbol that is a match and ends at y offset q, or DFL_NONE
SNACC_HD uint32_t dfl_canon_find(const DflCanon &cn, uint32_t q)
{
    uint32_t lo = 0, hi = cn.n_sym;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (SNACC_LDG(cn.end + mid) < q) lo = mid + 1; else hi = mid;
    }
    if (lo < cn.n_sym && SNACC_LDG(cn.end + lo) == q && (SNACC_LDG(cn.code + lo) >> 9) != DFL_LIT) return lo;
    return DFL_NONE;
}

// histogram of the canonical symbols [0, t) into acc[DFL_L_CODES + DFL_D_CODES]
SNACC_HD void dfl_cum_at(const DflCanon &cn, uint32_t t, uint32_t *acc)
{
    const uint32_t row = t / DFL_CUM_G;
    const uint32_t *src = cn.cum + (size_t)row * DFL_CUM_W;
    for (int c = 0; c < DFL_L_CODES + DFL_D_CODES; ++c) acc[c] = SNACC_LDG(src + c);
    for (uint32_t k = row * DFL_CUM_G; k < t; ++k) {
        const uint32_t code = SNACC_LDG(cn.code + k);
        acc[code & 511]++;
        if ((code >> 9) != DFL_LIT) acc[DFL_L_CODES + (code >> 9)]++;
    }
}

// ------------------------------------------------------------------------------------------------
// the serial part: deflate_slow's lazy evaluation over the F table
// ------------------------------------------------------------------------------------------------
struct DflParseState {                 // everything a stream needs to resume (the per-x checkpoint)
    uint32_t strstart, match_start, match_length, match_available;
    uint32_t sym_count, base, read, block_start;     // base/read: zlib's window refill state (oracle fill_window)
    uint64_t bits;
};
SNACC_HD void dfl_parse_fresh(DflParseState &st)
{
    st = DflParseState();
    st.match_length = DFL_MIN_MATCH - 1;
}

// where F of stream position p lives
struct DflFView {
    const uint32_t *fx;      // F of x alone, valid for p < jx0
    const uint32_t *fy;      // F of y alone, valid for p >= lx + DFL_JY
    const uint32_t *fj;      // junction of this pair: positions [jx0, jend)
    uint32_t jx0, jend, lx;
    // optional second tables holding the quartered-chain result of the flagged positions (level 6, where
    // prev_length >= good_length is the common case); null: recompute on demand
    const uint32_t *qx, *qy, *qj;
    // dfl_prep_kernel: the chunk of F around the parse position, staged in shared memory (ring of 2 * DFL_PREP_CHUNK
    // entries indexed by position); null elsewhere
    const uint32_t *ring = nullptr;
};
constexpr uint32_t DFL_PREP_CHUNK = 4096;
// The parse reads F at nearly consecutive positions (two reads per emitted match, a match is ~9 bytes on DNA) and
// each read is a dependent DRAM round trip, so the last 32-byte sector (8 entries) is kept in registers.
// All three tables start on 32-byte boundaries and are padded to a multiple of 8 entries.
struct DflFCache { const uint32_t *base; uint32_t v[8]; };
SNACC_HD uint32_t dfl_f_cached(DflFCache &c, const uint32_t *tab, uint32_t i)
{
    const uint32_t *blk = tab + (i & ~7u);
    if (blk != c.base) {
        c.base = blk;
#ifdef __CUDA_ARCH__
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(blk)), b = __ldg(reinterpret_cast<const uint4 *>(blk) + 1);
        c.v[0] = a.x; c.v[1] = a.y; c.v[2] = a.z; c.v[3] = a.w; c.v[4] = b.x; c.v[5] = b.y; c.v[6] = b.z; c.v[7] = b.w;
#else
        for (int k = 0; k < 8; ++k) c.v[k] = blk[k];
#endif
    }
    const uint32_t k = i & 7;
    const uint32_t lo = (k & 1) ? ((k & 2) ? c.v[3] : c.v[1]) : ((k & 2) ? c.v[2] : c.v[0]);
    const uint32_t hi = (k & 1) ? ((k & 2) ? c.v[7] : c.v[5]) : ((k & 2) ? c.v[6] : c.v[4]);
    return (k & 4) ? hi : lo;
}
SNACC_HD uint32_t dfl_f_at(const DflFView &v, uint32_t p, DflFCache &c)
{
    if (v.ring) return v.ring[p & (2 * DFL_PREP_CHUNK - 1)];
    if (p < v.jx0) return dfl_f_cached(c, v.fx, p);
    if (p < v.jend) return dfl_f_cached(c, v.fj, p - v.jx0);
    return dfl_f_cached(c, v.fy, p - v.lx);
}
SNACC_HD uint32_t dfl_q_at(const DflFView &v, uint32_t p)
{
    if (p < v.jx0) return SNACC_LDG(v.qx + p);
    if (p < v.jend) return SNACC_LDG(v.qj + (p - v.jx0));
    return SNACC_LDG(v.qy + (p - v.lx));
}

// Run deflate_slow from `st` until strstart >= stop (loop-top granularity) or the stream ends; lfreq/dfreq
// are the open block's counters (strided so that a kernel can keep them in shared memory).  At the end of
// the stream the last block is flushed and the function returns true.
// rec: record every emitted symbol (the parse of a sequence alone).  canon: the canonical stream of y; the
// function returns 2 -- with *sync_k = index of the canonical symbol just reproduced -- at the first match
// that ends at a stream position >= sync_from where the canonical parse also ended a match.
// Returns 0 when it stopped at `stop`, 1 when the stream is finished.
template <class TallyT>
static __host__ __device__ int dfl_parse(const DflStream &d, const DflFView &fv, const DflConfig &c, DflParseState &st,
                                         TallyT *lfreq, int lstride, TallyT *dfreq, int dstride, DflTrees &tr, uint32_t stop,
                                         DflRec *rec = nullptr, const DflCanon *canon = nullptr, uint32_t sync_from = 0,
                                         uint32_t *sync_k = nullptr)
{
    const Stream &s = d.s;
    const uint32_t n = s.n;
    uint32_t strstart = st.strstart, match_start = st.match_start, match_length = st.match_length;
    uint32_t match_available = st.match_available, sym_count = st.sym_count;
    uint32_t base = st.base, read = st.read, block_start = st.block_start;
    uint64_t bits = st.bits;
    bool done = false, synced = false;
    DflFCache fc;
    fc.base = nullptr;
#define DFL_FLUSH(last_) do {                                                                                   \
        dfl_flush_block(tr, lfreq, lstride, dfreq, dstride, strstart - block_start, block_start >= base, (last_), bits); \
        for (int n_ = 0; n_ < DFL_L_CODES; n_++) lfreq[n_ * lstride] = 0;                                        \
        for (int n_ = 0; n_ < DFL_D_CODES; n_++) dfreq[n_ * dstride] = 0;                                        \
        lfreq[256 * lstride] = 1; sym_count = 0; block_start = strstart; } while (0)
    for (;;) {
        if (strstart >= stop && strstart < n) break;
        // fill_window: slide and read ahead exactly as zlib does when all input is available
        if (read - strstart < DFL_MAX_MATCH + DFL_MIN_MATCH + 1) {
            for (;;) {
                uint32_t more = 2 * DFL_WSIZE - (read - base);
                if (strstart - base >= DFL_WSIZE + DFL_MAX_DIST) { base += DFL_WSIZE; more += DFL_WSIZE; }
                if (read == n) break;
                read += tmin(n - read, more);
                if (!(read - strstart < DFL_MAX_MATCH + DFL_MIN_MATCH + 1 && read != n)) break;
            }
            if (read == strstart) { done = true; break; }
        }
        const uint32_t prev_length = match_length, prev_match = match_start;
        match_length = DFL_MIN_MATCH - 1;
        if (prev_length < (uint32_t)c.max_lazy) {
            uint32_t f;
            if (base != dfl_window_base(strstart)) {
                // end of input: zlib slid the window one position early; the tables assume the regular schedule
                uint32_t q;
                f = dfl_longest(d, strstart, base, (uint32_t)c.max_chain, (uint32_t)c.nice_length, 0xffffffffu, &q);
                if (prev_length >= (uint32_t)c.good_length) f = q;
            } else {
                f = dfl_f_at(fv, strstart, fc);
                if (prev_length >= (uint32_t)c.good_length && (f & DFL_QDIFF)) {  // quartered chain: second table or on demand
                    if (fv.qx) f = dfl_q_at(fv, strstart);
                    else dfl_longest(d, strstart, base, (uint32_t)c.max_chain, (uint32_t)c.nice_length, 0xffffffffu, &f);
                }
                f &= ~DFL_QDIFF;
            }
            const uint32_t len = f >> 16, dist = f & 0xffff;
            if (len > prev_length) {
                match_length = len; match_start = strstart - dist;
                if (len == DFL_MIN_MATCH && dist > DFL_TOO_FAR) match_length = DFL_MIN_MATCH - 1;
            }
            // otherwise zlib's longest_match returns prev_length (or no search happens): either way the branch
            // below is taken exactly as with MIN_MATCH-1
        }
        if (prev_length >= DFL_MIN_MATCH && match_length <= prev_length) {
            const uint32_t lc = (uint32_t)dfl_length_code(prev_length - DFL_MIN_MATCH) + 257;
            const uint32_t dcd = (uint32_t)dfl_dist_code(strstart - 1 - prev_match - 1);
            lfreq[lc * lstride]++;
            dfreq[dcd * dstride]++;
            const bool bflush = ++sym_count == DFL_SYMS_PER_BLOCK;
            strstart += prev_length - 1;
            match_available = 0;
            match_length = DFL_MIN_MATCH - 1;
            dfl_rec_emit(rec, lc | (dcd << 9), strstart);
            if (bflush) DFL_FLUSH(false);
            if (canon && strstart >= sync_from) {
                const uint32_t k = dfl_canon_find(*canon, strstart - s.lx);
                if (k != DFL_NONE) { *sync_k = k; synced = true; break; }
            }
        } else if (match_available) {
            const uint32_t lit = ld8(s, strstart - 1);
            lfreq[lit * lstride]++;
            const bool bflush = ++sym_count == DFL_SYMS_PER_BLOCK;
            dfl_rec_emit(rec, lit | (DFL_LIT << 9), strstart);
            if (bflush) DFL_FLUSH(false);
            strstart++;
        } else {
            match_available = 1;
            strstart++;
        }
    }
    if (done) {
        if (match_available) {
            const uint32_t lit = ld8(s, strstart - 1);
            lfreq[lit * lstride]++; ++sym_count; match_available = 0;
            dfl_rec_emit(rec, lit | (DFL_LIT << 9), strstart);
        }
        DFL_FLUSH(true);
    }
#undef DFL_FLUSH
    st.strstart = strstart; st.match_start = match_start; st.match_length = match_length;
    st.match_available = match_available; st.sym_count = sym_count; st.block_start = block_start; st.bits = bits;
    st.base = base; st.read = read;
    return done ? 1 : synced ? 2 : 0;
}


// ------------------------------------------------------------------------------------------------
// the parse of a sequence alone, in parallel
// ------------------------------------------------------------------------------------------------
// The serial parse of a 5 Mbp sequence is ~1.4 M dependent loop iterations: 0.46 s on one thread, however many GPUs
// share the corpus (dfl_prep_kernel).  But right after a match the state of deflate_slow is just the position (see
// "canonical symbol stream" above), so the parse started ANYWHERE with that state falls in with the true parse at the
// first position where both end a match, and emits the same symbols from there on.  The sequence is therefore cut into
// chunks of DFL_CHUNK bytes, one thread each:
//   scan   thread k parses from its chunk start s_k to s_{k+1} + DFL_CHUNK_OV and notes, as two bitmaps, where its
//          matches end inside [s_k, s_k + OV) and inside [s_{k+1}, s_{k+1} + OV);
//   sync   y_{k+1} = the first position of [s_{k+1}, s_{k+1} + OV) where chunk k (true there: y_k < s_k + OV << s_{k+1})
//          and chunk k+1 both end a match; y_0 = 0;
//   count  thread k parses [y_k, y_{k+1}) and counts its symbols; a scan over the chunks gives every chunk its place;
//   emit   thread k parses [y_k, y_{k+1}) again and writes its symbols there.
// Everything stays below E = n - DFL_TAIL, where zlib's window schedule is the regular one the F tables assume; the
// blocks (every 16 383 symbols), the size, the checkpoint and the last DFL_TAIL bytes are then done per sequence by
// dfl_alone_kernel, exactly as a pair stream does them (dfl_canon_blocks + the serial parser for the tail).  A
// sequence where two neighbouring chunks never meet inside the overlap (long periodic runs: match ends of period 258
// that are out of phase) takes the serial kernel instead.
constexpr uint32_t DFL_CHUNK = 8192, DFL_CHUNK_OV = 1024, DFL_CHUNK_WORDS = DFL_CHUNK_OV / 32;
constexpr uint32_t DFL_PAR_MIN = 16 * DFL_CHUNK;            // shorter sequences: serial kernel
constexpr uint32_t DFL_NOWIN = 0x80000000u;                 // a window start no position (< 2^31) is within OV of

SNACC_HD uint32_t dfl_chunk_end(uint32_t n) { return n - DFL_TAIL; }                         // E
SNACC_HD uint32_t dfl_chunk_count(uint32_t n) { return dfl_chunk_end(n) / DFL_CHUNK; }       // the last chunk is [s, E): up to 2 chunks long

struct DflLite {
    int mode;                          // 0 scan, 1 count, 2 emit
    uint32_t head_lo, tail_lo;         // scan: windows [head_lo, +OV), [tail_lo, +OV) (DFL_NOWIN: none)
    uint32_t *head, *tail;             //       their bitmaps (DFL_CHUNK_WORDS words each, zeroed by the caller)
    uint32_t until;                    // count / emit: stop right after the match that ends here (DFL_NONE: run to `stop`)
    uint32_t count;                    // symbols seen (count / emit)
    uint32_t *end; uint16_t *code; uint32_t cap;     // emit: destination of symbol 0 and the slots left
};

// deflate_slow over F in the regular window schedule from the loop top at `from` (which follows a match, or is the
// stream start), without tallies and block flushes.  Returns false when an emit ran out of slots.
static __host__ __device__ bool dfl_lite_parse(const DflStream &d, const uint32_t *F, const uint32_t *Q, const DflConfig &c,
                                                uint32_t from, uint32_t stop, DflLite &o)
{
    uint32_t strstart = from, match_start = 0, match_length = DFL_MIN_MATCH - 1, match_available = 0;
    for (;;) {
        if (strstart >= stop) break;
        const uint32_t prev_length = match_length, prev_match = match_start;
        match_length = DFL_MIN_MATCH - 1;
        if (prev_length < (uint32_t)c.max_lazy) {
            uint32_t f = SNACC_LDG(F + strstart);
            if (prev_length >= (uint32_t)c.good_length && (f & DFL_QDIFF)) {
                if (Q) f = SNACC_LDG(Q + strstart);
                else dfl_longest(d, strstart, dfl_window_base(strstart), (uint32_t)c.max_chain, (uint32_t)c.nice_length, 0xffffffffu, &f);
            }
            f &= ~DFL_QDIFF;
            const uint32_t len = f >> 16, dist = f & 0xffff;
            if (len > prev_length) {
                match_length = len; match_start = strstart - dist;
                if (len == DFL_MIN_MATCH && dist > DFL_TOO_FAR) match_length = DFL_MIN_MATCH - 1;
            }
        }
        if (prev_length >= DFL_MIN_MATCH && match_length <= prev_length) {
            const uint32_t dist1 = strstart - 1 - prev_match - 1;
            strstart += prev_length - 1;
            match_available = 0;
            match_length = DFL_MIN_MATCH - 1;
            if (o.mode == 0) {
                if (strstart - o.head_lo < DFL_CHUNK_OV) o.head[(strstart - o.head_lo) >> 5] |= 1u << ((strstart - o.head_lo) & 31);
                if (strstart - o.tail_lo < DFL_CHUNK_OV) o.tail[(strstart - o.tail_lo) >> 5] |= 1u << ((strstart - o.tail_lo) & 31);
            } else {
                if (o.mode == 2) {
                    if (o.count >= o.cap) return false;
                    o.end[o.count] = strstart;
                    o.code[o.count] = (uint16_t)(((uint32_t)dfl_length_code(prev_length - DFL_MIN_MATCH) + 257) | ((uint32_t)dfl_dist_code(dist1) << 9));
                }
                ++o.count;
                if (strstart == o.until) break;
            }
        } else if (match_available) {
            if (o.mode == 2) {
                if (o.count >= o.cap) return false;
                o.end[o.count] = strstart;
                o.code[o.count] = (uint16_t)(ld8(d.s, strstart - 1) | (DFL_LIT << 9));
            }
            if (o.mode) ++o.count;
            strstart++;
        } else {
            match_available = 1;
            strstart++;
        }
    }
    return true;
}

// y_k of chunk k >= 1 from the two bitmaps that look at [s_k, s_k + OV): DFL_NONE when the chunks never meet there
SNACC_HD uint32_t dfl_chunk_sync(const uint32_t *tail_prev, const uint32_t *head, uint32_t s_k)
{
    for (uint32_t w = 0; w < DFL_CHUNK_WORDS; ++w) {
        const uint32_t m = tail_prev[w] & head[w];
        if (m) return s_k + w * 32 + (uint32_t)SNACC_FFS32(m) - 1;
    }
    return DFL_NONE;
}

#if defined(DFL_CHECK_COMPACT)
static int64_t dfl_compact_checked = 0, dfl_compact_mismatch = 0;     // host emulation only (tests/host_emu.cu)
#endif
// After dfl_parse returned 2 at canonical symbol k_sync: account every block of the pair stream that ends
// before the tail from the cumulative histograms and leave `st` at the loop top that follows the last
// canonical match ending at or before ly - DFL_TAIL.  Returns 1 when it advanced, 0 when there was nothing
// to skip, -1 when a block would consider the stored form (the job then takes the full serial parse).
// accA/accB: two scratch rows of DFL_L_CODES + DFL_D_CODES counters.
// (k_sync = DFL_NONE: the stream IS the canonical one from its first symbol -- the sequence alone, dfl_alone_kernel;
// t_end_out: number of canonical symbols accounted for.)
template <class TallyT>
static __host__ __device__ int dfl_canon_blocks(const DflCanon &cn, uint32_t lx, uint32_t n, uint32_t k_sync, DflParseState &st,
                                                TallyT *lfreq, int lstride, TallyT *dfreq, int dstride, DflTrees &tr,
                                                uint32_t *accA, uint32_t *accB, DflCompactTrees *ct = nullptr,
                                                uint32_t *t_end_out = nullptr)
{
    const uint32_t ly = n - lx, lim = ly - DFL_TAIL;
    uint32_t lo = 0, hi = cn.n_sym;                        // first symbol that ends beyond lim
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (SNACC_LDG(cn.end + mid) <= lim) lo = mid + 1; else hi = mid;
    }
    if (lo == 0) return 0;
    uint32_t kt = lo - 1;
    const uint32_t t_first = k_sync + 1;                   // (DFL_NONE + 1 = 0)
    if (kt < t_first) return 0;
    while (kt > t_first && (SNACC_LDG(cn.code + kt) >> 9) == DFL_LIT) --kt;
    if ((SNACC_LDG(cn.code + kt) >> 9) == DFL_LIT) return 0;
    uint32_t t = t_first;
    const uint32_t t_end = kt + 1;
    if (t_end_out) *t_end_out = t_end;
    uint32_t *a = accA, *b = accB;
    dfl_cum_at(cn, t, a);
    for (;;) {
        const uint32_t need = DFL_SYMS_PER_BLOCK - st.sym_count;
        const bool flush = t + need <= t_end;
        const uint32_t t2 = flush ? t + need : t_end;
        dfl_cum_at(cn, t2, b);
        for (int k = 0; k < DFL_L_CODES; ++k) lfreq[k * lstride] += (TallyT)(b[k] - a[k]);
        for (int k = 0; k < DFL_D_CODES; ++k) dfreq[k * dstride] += (TallyT)(b[DFL_L_CODES + k] - a[DFL_L_CODES + k]);
        st.sym_count += t2 - t;
        if (flush) {
            const uint32_t e2 = lx + SNACC_LDG(cn.end + t2 - 1);
            bool cand = false;
#if defined(DFL_CHECK_COMPACT) && !defined(__CUDA_ARCH__)
            {   // host emulation: the compacted trees must give exactly what the full ones give
                uint64_t b0 = st.bits, b1 = st.bits; bool c0 = false, c1 = false;
                dfl_flush_block(tr, lfreq, lstride, dfreq, dstride, e2 - st.block_start, true, false, b0, &c0);
                if (ct && dfl_flush_block_compact(*ct, lfreq, lstride, dfreq, dstride, e2 - st.block_start, true, false, b1, &c1)) {
                    ++dfl_compact_checked;
                    if (b0 != b1 || c0 != c1) ++dfl_compact_mismatch;
                }
            }
#endif
            if (!ct || !dfl_flush_block_compact(*ct, lfreq, lstride, dfreq, dstride, e2 - st.block_start, true, false, st.bits, &cand))
                dfl_flush_block(tr, lfreq, lstride, dfreq, dstride, e2 - st.block_start, true, false, st.bits, &cand);
            if (cand) return -1;
            for (int k = 0; k < DFL_L_CODES; ++k) lfreq[k * lstride] = 0;
            for (int k = 0; k < DFL_D_CODES; ++k) dfreq[k * dstride] = 0;
            lfreq[256 * lstride] = 1; st.sym_count = 0; st.block_start = e2;
        }
        uint32_t *sw = a; a = b; b = sw;
        t = t2;
        if (!flush) break;
    }
    st.strstart = lx + SNACC_LDG(cn.end + t_end - 1);
    st.match_available = 0; st.match_length = DFL_MIN_MATCH - 1; st.match_start = 0;
    st.base = dfl_window_base(st.strstart);                // a regular loop top: strstart <= n - DFL_TAIL
    const uint64_t want = (uint64_t)st.base + 2 * DFL_WSIZE;
    st.read = want < n ? (uint32_t)want : n;
    return 1;
}

// The whole pair stream x.y from the checkpoint of x (already in st / lfreq / dfreq).  Returns 0 when the job
// has to take the full serial parse (cn = null) instead, 1 when it was parsed serially, 2 when blocks were
// taken from the canonical stream.
template <class TallyT>
static __host__ __device__ int dfl_pair_stream(const DflStream &d, const DflFView &fv, const DflConfig &c, DflParseState &st,
                                                TallyT *lfreq, int lstride, TallyT *dfreq, int dstride, DflTrees &tr,
                                                const DflCanon *cn, uint32_t *accA, uint32_t *accB, DflCompactTrees *ct = nullptr)
{
    const uint32_t lx = d.s.lx, n = d.s.n;
    const bool use = cn && cn->n_sym != 0 && n - lx >= DFL_CANON_MIN;
    uint32_t k_sync = 0;
    int r = dfl_parse(d, fv, c, st, lfreq, lstride, dfreq, dstride, tr, 0xffffffffu, (DflRec *)nullptr, use ? cn : nullptr,
                      lx + DFL_JY, &k_sync);
    if (r == 2) {
        const int b = dfl_canon_blocks(*cn, lx, n, k_sync, st, lfreq, lstride, dfreq, dstride, tr, accA, accB, ct);
        if (b < 0) return 0;
        dfl_parse(d, fv, c, st, lfreq, lstride, dfreq, dstride, tr, 0xffffffffu);
        return b ? 2 : 1;
    }
    return 1;
}


// resume a pair stream from the checkpoint of its x (taken at the first loop top >= jx0 of x alone)
SNACC_HD void dfl_resume(DflParseState &st, uint32_t n)
{
    // zlib has always read up to base + 64 KiB (or everything); x alone had stopped at its own end
    const uint64_t want = (uint64_t)st.base + 2 * DFL_WSIZE;
    st.read = want < n ? (uint32_t)want : n;
}
SNACC_HD uint32_t dfl_jx0(uint32_t lx) { return lx > DFL_JX ? lx - DFL_JX : 0; }
SNACC_HD uint32_t dfl_jlen(uint32_t lx, uint32_t ly) { return (lx - dfl_jx0(lx)) + tmin(ly, DFL_JY); }
constexpr uint32_t DFL_JSTRIDE = DFL_JX + DFL_JY;
static_assert(DFL_JSTRIDE % 8 == 0, "junction slices must start on 32-byte boundaries (DflFCache)");

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// A 3-byte index slice is one block: DFL_BROW words of bucket starts (DFL_HASH + 1 used), then the sorted positions.  It
// lives in the y-side pool (the whole index of a sequence of the y layout) or in the x-side pool (its tail slice).
constexpr uint32_t DFL_BROW = DFL_HASH + 8;

// Device state is split by role.  x side (every sequence): record, tail index, tail packs.  y side (only the sequences
// of the current y layout, DeflateState::ylist): whole index, F, head tables, canonical stream.  Per-sequence tables of
// the y side are addressed through poff (per-position arrays) and yslot (fixed-size rows).
struct DflCorpus {
    const uint8_t *corpus; const uint64_t *off; const uint32_t *len;   // padded byte corpus (api.cu)
    const uint64_t *poff;        // per y-side sequence: offset of its slice in the F / FQ arrays and the order6 window
    uint32_t *const *ix;         // per sequence: its current 3-byte index slice (bucket starts, then positions)
    const uint32_t *yslot;       // per y-side sequence: its row of head_order, head_visit and bstart6
    // whole 3-byte index slices of the y side, the one of sequence sq at poff[sq] + yslot[sq] * DFL_BROW: a sequence is
    // parsed alone only while it is in the y layout, and the kernels that do so address its index from here, as
    // arithmetic the compiler may redo instead of keeping a loaded pointer live through the parse
    uint32_t *yindex;
    // head of every y-side sequence (its first DFL_JY positions), for the junction of the pair streams it ends:
    uint16_t *head_order;        // per y slot DFL_JY entries: the indexed head positions sorted by (hash, position)
    uint16_t *head_visit;        // per y slot and level DFL_JY entries: how longest_match went in the sequence alone
    // tail of every sequence, for the junction of the pair streams it starts:
    uint16_t *tail_cnt;          // per sequence DFL_HASH entries: bucket entries at or after dfl_tail3_from(len)
    uint16_t *tail6_order;       // per sequence DFL_T6 entries   } 6-byte index of the tail (DflTail6)
    uint16_t *tail6_start;       // per sequence DFL_H6 + 1 entries }
    // transient 6-byte index of whole sequences (DflIndex6): order6 is a window buffer addressed like `order`
    uint32_t *order6;
    uint32_t *bstart6;           // per y slot DFL_HASH + 1 entries
    // first position of the 3-byte index: 0, or len - DFL_XTAIL for a sequence that is only ever the x of pair streams
    // here (its record came from another rank): the junction walks reach at most 264 + 32 768 positions back from its end
    const uint32_t *ifrom;
};
constexpr uint32_t DFL_XTAIL = 40960;

// (the table is rewritten by the host between launches only)
__device__ __forceinline__ uint32_t *dfl_ix(const DflCorpus &c, int32_t s)
{
    return reinterpret_cast<uint32_t *>(__ldg(reinterpret_cast<const unsigned long long *>(c.ix + s)));
}

SNACC_HD Stream dfl_make_stream(const DflCorpus &c, int32_t x, int32_t y)
{
    Stream s;
    s.x = c.corpus + c.off[x];
    s.lx = c.len[x];
    if (y >= 0) { s.y = c.corpus + c.off[y]; s.n = s.lx + c.len[y]; }
    else        { s.y = s.x + s.lx;          s.n = s.lx; }
    return s;
}
// the pair stream x.y (y >= 0): each part's current index
__device__ __forceinline__ DflStream dfl_make(const DflCorpus &c, int32_t x, int32_t y)
{
    DflStream d;
    d.s = dfl_make_stream(c, x, y);
    d.pair = true;
    const uint32_t *ix = dfl_ix(c, x), *iy = dfl_ix(c, y);
    d.ix.bstart = ix; d.ix.order = ix + DFL_BROW;
    d.iy.bstart = iy; d.iy.order = iy + DFL_BROW;
    return d;
}
// sequence sq alone: only parsed while it is in the y layout, so its index is the whole one there
__device__ __forceinline__ DflStream dfl_make_alone(const DflCorpus &c, int32_t sq)
{
    DflStream d;
    d.s = dfl_make_stream(c, sq, -1);
    d.pair = false;
    const uint32_t *ix = c.yindex + c.poff[sq] + (size_t)c.yslot[sq] * DFL_BROW;
    d.ix.bstart = ix; d.ix.order = ix + DFL_BROW;
    d.iy = d.ix;
    return d;
}

// K3a: index of a sequence = its positions sorted by (hash, position): a stable LSD radix sort on the 15-bit hash in
// two passes (low 8 bits, high 7 bits).  The sort key is recomputed from the bytes, only positions move.
//   KIND 0: the 3-byte chain hash over positions [ifrom, len - 2) -> c.ix[sq];
//   KIND 1: the 6-byte hash over positions [0, len - 5) -> c.order6 / c.bstart6 (DflIndex6).
// A tile is 8192 consecutive keys handled by one CTA of 32 warps; warp w takes keys [256 w, 256 (w + 1)) of the tile in
// 8 rounds of 32, so (warp, round, lane) order is key order and ranks come out stable: inside a round from
// __match_any_sync, across rounds from the warp's running digit counts, across warps from a scan of those counts,
// across tiles from the scanned per-tile digit totals (dfl_radix_scan_kernel).
constexpr uint32_t DFL_RX_TILE = 8192, DFL_RX_THREADS = 1024, DFL_RX_ROUNDS = DFL_RX_TILE / DFL_RX_THREADS;
template <int KIND> SNACC_HD uint32_t dfl_index_count(uint32_t len) { return KIND == 0 ? (len >= 3 ? len - 2 : 0) : (len >= 6 ? len - 5 : 0); }
// first indexed position / number of index entries of sequence sq (the 6-byte index is always whole)
template <int KIND> __device__ __forceinline__ uint32_t dfl_index_first(const DflCorpus &c, int32_t sq) { return KIND == 0 ? c.ifrom[sq] : 0u; }
template <int KIND> __device__ __forceinline__ uint32_t dfl_index_n(const DflCorpus &c, int32_t sq)
{
    const uint32_t n = dfl_index_count<KIND>(c.len[sq]), f = dfl_index_first<KIND>(c, sq);
    return n > f ? n - f : 0u;
}
template <int KIND> __device__ __forceinline__ uint32_t dfl_index_hash(const uint8_t *p, uint32_t i)
{
    return KIND == 0 ? dfl_hash3(p[i], p[i + 1], p[i + 2]) : dfl_hash6w(ldu64(p + i));
}
SNACC_HD uint32_t dfl_rx_tiles(uint32_t n) { return (n + DFL_RX_TILE - 1) / DFL_RX_TILE; }

// SCATTER = false: digit totals of every tile -> hist[(seq slot * 256 + digit) * max_tiles + tile]
// SCATTER = true : hist holds the exclusive scan of those totals; keys go to their sorted place
// Scratch (src_all, and dst_all of pass 0) is addressed by poff; the 3-byte index lands in c.ix[sq], the 6-byte one in dst_all + poff.
template <int KIND, int PASS, bool SCATTER>
__global__ void __launch_bounds__(DFL_RX_THREADS)
dfl_radix_kernel(DflCorpus c, const int32_t *__restrict__ seqs, uint32_t max_tiles, uint32_t *__restrict__ hist,
                 const uint32_t *__restrict__ src_all, uint32_t *__restrict__ dst_all)
{
    __shared__ uint16_t wcnt[32][256];
    __shared__ uint32_t toff[256];
    const int32_t slot = blockIdx.y, sq = seqs[slot];
    const uint32_t n = dfl_index_n<KIND>(c, sq), first = dfl_index_first<KIND>(c, sq);
    const uint32_t tile = blockIdx.x;
    if (tile * DFL_RX_TILE >= n) return;
    const uint8_t *p = c.corpus + c.off[sq];
    const uint32_t *src = src_all + c.poff[sq];
    uint32_t *dst = (KIND == 0 && PASS == 1) ? dfl_ix(c, sq) + DFL_BROW : dst_all + c.poff[sq];
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (uint32_t i = threadIdx.x; i < 32 * 256; i += blockDim.x) (&wcnt[0][0])[i] = 0;
    __syncthreads();
    uint32_t pos[DFL_RX_ROUNDS], dg[DFL_RX_ROUNDS], lr[DFL_RX_ROUNDS];
#pragma unroll
    for (uint32_t r = 0; r < DFL_RX_ROUNDS; ++r) {
        const uint32_t idx = tile * DFL_RX_TILE + w * (32 * DFL_RX_ROUNDS) + r * 32 + lane;
        const bool ok = idx < n;
        pos[r] = ok ? (PASS == 0 ? first + idx : src[idx]) : 0;
        const uint32_t h = ok ? dfl_index_hash<KIND>(p, pos[r]) : 0;
        dg[r] = ok ? (PASS == 0 ? (h & 255u) : (h >> 8)) : 0x10000u + lane;
        const uint32_t peers = __match_any_sync(0xffffffffu, dg[r]);
        lr[r] = ok ? wcnt[w][dg[r]] + __popc(peers & ((1u << lane) - 1)) : 0;
        __syncwarp();
        if (ok && (peers >> lane) <= 1u) wcnt[w][dg[r]] += (uint16_t)__popc(peers);
        __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x < 256) {                               // exclusive scan over the warps, digit by digit
        uint32_t run = 0;
        for (uint32_t k = 0; k < 32; ++k) { const uint32_t v = wcnt[k][threadIdx.x]; wcnt[k][threadIdx.x] = (uint16_t)run; run += v; }
        const size_t hi = ((size_t)slot * 256 + threadIdx.x) * max_tiles + tile;
        if (SCATTER) toff[threadIdx.x] = hist[hi]; else hist[hi] = run;
    }
    if (!SCATTER) return;
    __syncthreads();
#pragma unroll
    for (uint32_t r = 0; r < DFL_RX_ROUNDS; ++r)
        if (dg[r] < 256u) dst[toff[dg[r]] + wcnt[w][dg[r]] + lr[r]] = pos[r];
}

// in-place exclusive scan of the 256 * max_tiles digit totals of every sequence slot (digit-major), one CTA per slot
__global__ void __launch_bounds__(1024)
dfl_radix_scan_kernel(uint32_t max_tiles, uint32_t *__restrict__ hist)
{
    __shared__ uint32_t part[1024];
    uint32_t *h = hist + (size_t)blockIdx.x * 256 * max_tiles;
    const uint32_t n = 256 * max_tiles, per = (n + 1023) / 1024;
    const uint32_t lo = tmin(n, threadIdx.x * per), hi = tmin(n, lo + per);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; ++i) sum += h[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    for (uint32_t o = 1; o < 1024; o <<= 1) {              // Hillis-Steele inclusive scan
        const uint32_t v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = part[threadIdx.x] - sum;
    for (uint32_t i = lo; i < hi; ++i) { const uint32_t v = h[i]; h[i] = run; run += v; }
}

// bucket starts from the sorted order: mark where the hash changes, then every unmarked (empty) bucket starts where the next
// one does
template <int KIND>
__global__ void __launch_bounds__(256)
dfl_index_bounds_kernel(DflCorpus c, const int32_t *__restrict__ seqs)
{
    const int32_t sq = seqs[blockIdx.y];
    const uint32_t n = dfl_index_n<KIND>(c, sq);
    const uint8_t *p = c.corpus + c.off[sq];
    const uint32_t *order = KIND == 0 ? dfl_ix(c, sq) + DFL_BROW : c.order6 + c.poff[sq];
    uint32_t *bstart = KIND == 0 ? dfl_ix(c, sq) : c.bstart6 + (size_t)c.yslot[sq] * (DFL_HASH + 1);
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const uint32_t h = dfl_index_hash<KIND>(p, order[k]);
        if (k == 0 || dfl_index_hash<KIND>(p, order[k - 1]) != h) bstart[h] = k;
    }
}
template <int KIND>
__global__ void __launch_bounds__(1024)
dfl_index_fill_kernel(DflCorpus c, const int32_t *__restrict__ seqs, int phase)
{
    // phase 0: all starts unmarked; phase 1 (after dfl_index_bounds_kernel): suffix minimum
    __shared__ uint32_t part[1024];
    const int32_t sq = seqs[blockIdx.x];
    const uint32_t n = dfl_index_n<KIND>(c, sq);
    uint32_t *bstart = KIND == 0 ? dfl_ix(c, sq) : c.bstart6 + (size_t)c.yslot[sq] * (DFL_HASH + 1);
    const uint32_t per = DFL_HASH / 1024;
    if (phase == 0) {
        for (uint32_t i = threadIdx.x; i < DFL_HASH; i += blockDim.x) bstart[i] = 0xffffffffu;
        if (threadIdx.x == 0) bstart[DFL_HASH] = n;
        return;
    }
    uint32_t m = 0xffffffffu;
    for (uint32_t k = 0; k < per; ++k) m = tmin(m, bstart[threadIdx.x * per + k]);
    part[threadIdx.x] = m;
    __syncthreads();
    for (uint32_t o = 1; o < 1024; o <<= 1) {              // inclusive suffix minimum
        const uint32_t v = threadIdx.x + o < 1024 ? part[threadIdx.x + o] : 0xffffffffu;
        __syncthreads();
        part[threadIdx.x] = tmin(part[threadIdx.x], v);
        __syncthreads();
    }
    uint32_t run = threadIdx.x + 1 < 1024 ? part[threadIdx.x + 1] : 0xffffffffu;
    run = tmin(run, n);
    for (int k = (int)per - 1; k >= 0; --k) {
        uint32_t &v = bstart[threadIdx.x * per + k];
        if (v == 0xffffffffu) v = run; else run = v;
    }
}

// K3b: F of every position of the listed sequences (each alone); thread per index entry so that the
// threads of a warp walk overlapping slices of the same bucket
__global__ void __launch_bounds__(256)
dfl_match_kernel(DflCorpus c, const int32_t *__restrict__ seqs, int32_t n_seqs, int level, uint32_t *__restrict__ F,
                 uint32_t *__restrict__ FQ)
{
    const DflConfig cfg = dfl_config(level);
    for (int32_t t = blockIdx.y; t < n_seqs; t += gridDim.y) {
        const int32_t sq = seqs[t];
        const DflStream d = dfl_make_alone(c, sq);
        const uint32_t len = d.s.n;
        const uint32_t nidx = len >= 3 ? len - 2 : 0;
        uint32_t *f = F + c.poff[sq];
        uint32_t *fq = FQ ? FQ + c.poff[sq] : nullptr;
        const DflIndex6 i6{c.order6 ? c.order6 + c.poff[sq] : nullptr, c.bstart6 + (size_t)c.yslot[sq] * (DFL_HASH + 1)};
        uint16_t *hvis = c.head_visit + (size_t)c.yslot[sq] * DFL_JY;
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
            if (k >= nidx) { f[k] = 0; if (fq) fq[k] = 0; continue; }       // the last two positions: no string, no search
            const uint32_t p = d.ix.order[k];
            uint32_t q, visit;
            f[p] = dfl_match_word(d, p, cfg, k, c.order6 ? &i6 : nullptr, &q, &visit);
            if (fq) fq[p] = q;
            if (p < DFL_JY) hvis[p] = (uint16_t)visit;
        }
    }
}

// K3b': head order of the listed sequences: the first min(len - 2, DFL_JY) positions sorted by (hash, position),
// taken bucket by bucket from the full index (a bucket's head positions are a prefix of it), and the tail counts of the
// x side.  head_order == nullptr: x-side index, tail counts only.  One CTA per sequence.
__global__ void __launch_bounds__(1024)
dfl_head_kernel(DflCorpus c, const int32_t *__restrict__ seqs, int32_t n_seqs)
{
    extern __shared__ uint32_t hcnt[];                   // DFL_HASH counters -> exclusive starts
    __shared__ uint32_t wsum[32];
    for (int32_t t = blockIdx.x; t < n_seqs; t += gridDim.x) {
        const int32_t sq = seqs[t];
        const uint32_t *bstart = dfl_ix(c, sq), *order = bstart + DFL_BROW;
        __syncthreads();
        const uint32_t tail_from = dfl_tail3_from(c.len[sq]);
        uint16_t *tc = c.tail_cnt + (size_t)sq * DFL_HASH;
        for (uint32_t h = threadIdx.x; h < DFL_HASH; h += blockDim.x) {
            const uint32_t lo = bstart[h], hi = bstart[h + 1];
            hcnt[h] = lo < hi ? dfl_lower_bound(order, lo, hi, DFL_JY) - lo : 0;
            tc[h] = (uint16_t)(lo < hi ? hi - dfl_lower_bound(order, lo, hi, tail_from) : 0);
        }
        if (c.ifrom[sq] || !c.head_order) continue;          // x-side index: no head order
        uint16_t *ho = c.head_order + (size_t)c.yslot[sq] * DFL_JY;
        __syncthreads();
        // exclusive scan over DFL_HASH counters: 32 per thread
        const uint32_t per = DFL_HASH / 1024;
        uint32_t sum = 0;
        for (uint32_t k = 0; k < per; ++k) sum += hcnt[threadIdx.x * per + k];
        uint32_t inc = sum;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o); if ((int)(threadIdx.x & 31) >= o) inc += u; }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = inc;
        __syncthreads();
        if (threadIdx.x < 32) {
            const uint32_t v = wsum[threadIdx.x];
            uint32_t w = v;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, w, o); if ((int)threadIdx.x >= o) w += u; }
            wsum[threadIdx.x] = w - v;
        }
        __syncthreads();
        uint32_t run = wsum[threadIdx.x >> 5] + inc - sum;
        for (uint32_t k = 0; k < per; ++k) { const uint32_t v = hcnt[threadIdx.x * per + k]; hcnt[threadIdx.x * per + k] = run; run += v; }
        __syncthreads();
        for (uint32_t h = threadIdx.x; h < DFL_HASH; h += blockDim.x) {
            const uint32_t lo = bstart[h], n = (h + 1 < DFL_HASH ? hcnt[h + 1] : tmin(DFL_JY, c.len[sq] >= 3 ? c.len[sq] - 2 : 0u)) - hcnt[h];
            for (uint32_t i = 0; i < n; ++i) ho[hcnt[h] + i] = (uint16_t)order[lo + i];
        }
    }
}

struct DflPair { int32_t x, y; };

// K3b'': 6-byte index of the tail of the listed sequences (DflTail6): stable counting sort by one warp, like
// the first version of the full index did.  Shared memory: DFL_H6 counters + one rank per tail position.
__global__ void __launch_bounds__(32)
dfl_tail6_kernel(DflCorpus c, const int32_t *__restrict__ seqs, int32_t n_seqs)
{
    extern __shared__ uint32_t t6_smem[];
    uint32_t *cnt = t6_smem;                                           // DFL_H6
    uint16_t *rank = reinterpret_cast<uint16_t *>(t6_smem + DFL_H6);   // DFL_T6
    const uint32_t lane = threadIdx.x;
    for (int32_t t = blockIdx.x; t < n_seqs; t += gridDim.x) {
        const int32_t sq = seqs[t];
        const uint32_t len = c.len[sq], t0 = dfl_tail6_t0(len), n6 = dfl_tail6_count(len);
        const uint8_t *p = c.corpus + c.off[sq] + t0;
        uint16_t *order = c.tail6_order + (size_t)sq * DFL_T6;
        uint16_t *start = c.tail6_start + (size_t)sq * (DFL_H6 + 1);
        for (uint32_t i = lane; i < DFL_H6; i += 32) cnt[i] = 0;
        __syncwarp();
        for (uint32_t b0 = 0; b0 < n6; b0 += 32) {
            const uint32_t i = b0 + lane;
            const bool ok = i < n6;
            const uint32_t h = ok ? dfl_hash6(ldu64(p + i)) : 0xffffffffu - lane;
            const uint32_t peers = __match_any_sync(0xffffffffu, h);
            if (ok) rank[i] = (uint16_t)(cnt[h] + __popc(peers & ((1u << lane) - 1)));
            __syncwarp();
            if (ok && (peers >> lane) <= 1u) cnt[h] += __popc(peers);
            __syncwarp();
        }
        uint32_t carry = 0;
        for (uint32_t b0 = 0; b0 < DFL_H6; b0 += 32) {
            const uint32_t v = cnt[b0 + lane];
            uint32_t inc = v;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o); if ((int)lane >= o) inc += u; }
            const uint32_t ex = carry + inc - v;
            start[b0 + lane] = (uint16_t)ex;
            cnt[b0 + lane] = ex;
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) start[DFL_H6] = (uint16_t)carry;
        __syncwarp();
        for (uint32_t i = lane; i < n6; i += 32) order[cnt[dfl_hash6(ldu64(p + i))] + rank[i]] = (uint16_t)i;
        __syncwarp();
    }
}

// K3c: junction F of a batch of pair streams: positions [jx0, lx + min(ly, DFL_JY)).  The last positions of x take
// the general walk.  The head positions of y are handled in (hash, position) order -- the lanes of a warp then
// walk the same bucket of x and their loads coalesce into broadcasts -- and continue the walk they had in y alone
// (dfl_longest_cont) instead of repeating it.
__global__ void __launch_bounds__(256)
dfl_junction_kernel(DflCorpus c, const DflPair *__restrict__ pairs, int32_t n_pairs, int level, const uint32_t *__restrict__ F,
                    const uint32_t *__restrict__ FQ, uint32_t *__restrict__ FJ, uint32_t *__restrict__ FJQ, int impl)
{
    const DflConfig cfg = dfl_config(level);
    for (int32_t b = blockIdx.y; b < n_pairs; b += gridDim.y) {
        const int32_t y = pairs[b].y;
        const DflStream d = dfl_make(c, pairs[b].x, y);
        const uint32_t lx = d.s.lx, ly = d.s.n - lx, jx0 = dfl_jx0(lx), jxl = lx - jx0, jyl = tmin(ly, DFL_JY);
        const uint32_t n_head = tmin(jyl, ly >= 3 ? ly - 2 : 0u);            // head positions that are in y's index
        uint32_t *f = FJ + (size_t)b * DFL_JSTRIDE;
        uint32_t *fq = FJQ ? FJQ + (size_t)b * DFL_JSTRIDE : nullptr;
        const uint32_t *fy = F + c.poff[y];
        const uint32_t *fqy = FQ ? FQ + c.poff[y] : nullptr;
        const uint16_t *ho = c.head_order + (size_t)c.yslot[y] * DFL_JY, *hv = c.head_visit + (size_t)c.yslot[y] * DFL_JY;
        const uint32_t u_end = jxl + jyl;
        const bool by_hash = impl != 3 || level != 9;
        const int32_t xi = pairs[b].x;
        const DflTail6 t6{c.tail6_order + (size_t)xi * DFL_T6, c.tail6_start + (size_t)xi * (DFL_H6 + 1), dfl_tail6_t0(lx)};
        const uint16_t *tcx = c.tail_cnt + (size_t)xi * DFL_HASH;
        // the 8 bytes at lx - k, k = 0..5 (dfl_longest_k6): loaded by six lanes, handed round by shuffle -- no block barrier,
        // the warps of a block finish a pair at very different times
        uint64_t edge[6];
        {
            const uint32_t ln = threadIdx.x & 31;
            const uint64_t mine = (ln < 6 && lx >= ln) ? ld64(d.s, lx - ln) : 0;
#pragma unroll
            for (int k = 0; k < 6; ++k) edge[k] = __shfl_sync(0xffffffffu, mine, k);
        }
        for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < u_end; u += gridDim.x * blockDim.x) {
            uint32_t q, w, pos;
            if (u < jxl) {
                pos = u;
                w = dfl_f_word(d, jx0 + u, cfg, 0xffffffffu, &q);
            } else if (u - jxl < n_head) {
                // with the 6-byte shortcut nearly every lane takes a handful of private candidates: position order keeps
                // the table reads and the result writes coalesced; the chain walk wants (hash, position) order instead
                const uint32_t yq = by_hash ? ho[u - jxl] : u - jxl;
                pos = jxl + yq;
                w = dfl_junction_word(d, lx + yq, cfg, fy[yq], hv[yq], fqy != nullptr, fqy ? fqy[yq] : 0u, impl == 3 ? &t6 : nullptr,
                                      tcx, &q, edge);
            } else {
                pos = u; w = 0; q = 0;                                       // the last two positions of a short y: no string
            }
            f[pos] = w;
            if (fq) fq[pos] = q;
        }
    }
}

// K3d: the serial parse, one stream per thread.
//   kind 3  a sequence alone: size -> seq_size, checkpoint at its junction start (what a pair stream x.* resumes
//           from) -> ckpt, canonical symbol stream -> canon pool
//   kind 2  pair stream resumed from the checkpoint of x, remaining blocks of y from the canonical stream of y
//   kind 4  pair stream resumed from the checkpoint of x, full serial parse (fallback of kind 2)
struct DflCkpt {
    DflParseState st;
    uint16_t lfreq[DFL_L_CODES];
    uint16_t dfreq[DFL_D_CODES];
};
struct DflJob { int32_t x, y, kind, fj; int64_t out; };     // fj: slot of the pair in the junction batch

struct DflCanonPool {
    uint32_t *end; uint16_t *code; uint32_t *cum;
    const uint64_t *soff;        // per sequence: first symbol slot
    const uint32_t *cap;         // per sequence: symbol slots
    const uint64_t *roff;        // per sequence: first cumulative row
    uint32_t *n_sym;             // per sequence: symbols recorded (0: none / overflow)
    int64_t *seq_size;           // per sequence: raw deflate size of the sequence alone
};
__device__ __forceinline__ DflCanon dfl_canon_of(const DflCanonPool &cp, int32_t s)
{
    DflCanon cn;
    cn.end = cp.end + cp.soff[s]; cn.code = cp.code + cp.soff[s];
    cn.cum = cp.cum + cp.roff[s] * DFL_CUM_W; cn.n_sym = cp.n_sym[s];
    return cn;
}

constexpr int DFL_PARSE_THREADS = 64;

__global__ void __launch_bounds__(DFL_PARSE_THREADS)
dfl_parse_kernel(DflCorpus c, const DflJob *__restrict__ jobs, int64_t n_jobs, int level, const uint32_t *__restrict__ F,
                 const uint32_t *__restrict__ FQ, const uint32_t *__restrict__ FJ, const uint32_t *__restrict__ FJQ,
                 DflCkpt *__restrict__ ckpt, DflCanonPool cp, DflTrees *__restrict__ scratch,
                 unsigned long long *__restrict__ counter, int64_t *__restrict__ out)
{
    __shared__ uint16_t s_l[DFL_L_CODES * DFL_PARSE_THREADS];
    __shared__ uint16_t s_d[DFL_D_CODES * DFL_PARSE_THREADS];
    extern __shared__ __align__(16) uint8_t s_compact[];              // DFL_PARSE_THREADS x DflCompactTrees
    const DflConfig cfg = dfl_config(level);
    const int T = DFL_PARSE_THREADS, tid = threadIdx.x;
    uint16_t *lf = s_l + tid, *df = s_d + tid;
    DflCompactTrees *ct = reinterpret_cast<DflCompactTrees *>(s_compact) + tid;
    DflTrees &tr = scratch[(size_t)blockIdx.x * T + tid];
    uint32_t accA[DFL_L_CODES + DFL_D_CODES], accB[DFL_L_CODES + DFL_D_CODES];
    for (;;) {
        const long long j = (long long)atomicAdd(counter, 1ull);
        if (j >= n_jobs) break;
        const DflJob jb = jobs[j];
        const DflStream d = dfl_make(c, jb.x, jb.y);
        const uint32_t lx = d.s.lx;
        DflFView fv;
        fv.fx = F + c.poff[jb.x]; fv.lx = lx;
        fv.qx = FQ ? FQ + c.poff[jb.x] : nullptr; fv.qy = fv.qj = fv.qx;
        fv.fy = F + c.poff[jb.y];
        fv.fj = FJ + (size_t)jb.fj * DFL_JSTRIDE;
        if (FQ) { fv.qy = FQ + c.poff[jb.y]; fv.qj = FJQ + (size_t)jb.fj * DFL_JSTRIDE; }
        fv.jx0 = dfl_jx0(lx); fv.jend = fv.jx0 + dfl_jlen(lx, d.s.n - lx);
        const DflCkpt &ck = ckpt[jb.x];
        DflParseState st = ck.st;
        dfl_resume(st, d.s.n);
        for (int k = 0; k < DFL_L_CODES; ++k) lf[k * T] = ck.lfreq[k];
        for (int k = 0; k < DFL_D_CODES; ++k) df[k * T] = ck.dfreq[k];
        DflCanon cn;
        cn.n_sym = 0;
        if (jb.kind == 2) cn = dfl_canon_of(cp, jb.y);
        const int how = dfl_pair_stream(d, fv, cfg, st, lf, T, df, T, tr, jb.kind == 2 ? &cn : nullptr, accA, accB, ct);
        out[jb.out] = how ? (int64_t)(st.bits >> 3) : -2;
    }
}

// K3d': the parse of every listed sequence ALONE: its size, the checkpoint at its junction start (what a pair stream
// x.* resumes from) and its canonical symbol stream.  A serial chain of ~1.1 M dependent steps for 5 Mbp, so the
// latency of each step is what counts: one CTA per sequence, thread 0 parses, the other warps stream F through a
// shared-memory ring one chunk ahead of it; symbol counters and tree scratch live in shared memory as well.
constexpr int DFL_PREP_THREADS = 128;
struct DflPrepSmem {
    uint32_t ring[2 * DFL_PREP_CHUNK];
    DflTrees tr;
    uint16_t lf[DFL_L_CODES], df[DFL_D_CODES];
    uint32_t done;
};

__global__ void __launch_bounds__(DFL_PREP_THREADS)
dfl_prep_kernel(DflCorpus c, const int32_t *__restrict__ seqs, int32_t n_seqs, int level, const uint32_t *__restrict__ F,
                const uint32_t *__restrict__ FQ, DflCkpt *__restrict__ ckpt, DflCanonPool cp)
{
    extern __shared__ __align__(16) uint8_t prep_raw[];
    DflPrepSmem &sm = *reinterpret_cast<DflPrepSmem *>(prep_raw);
    const DflConfig cfg = dfl_config(level);
    const uint32_t tid = threadIdx.x, C = DFL_PREP_CHUNK;
    for (int32_t t = blockIdx.x; t < n_seqs; t += gridDim.x) {
        const int32_t sq = seqs[t];
        const DflStream d = dfl_make_alone(c, sq);
        const uint32_t n = d.s.n, n_pad = (n + 7) & ~7u, jx0 = dfl_jx0(n);
        const uint32_t *fsrc = F + c.poff[sq];
        DflFView fv;
        DflParseState st;
        DflRec rec{cp.end + cp.soff[sq], cp.code + cp.soff[sq], cp.cap[sq], 0};
        bool ck_done = false;
        fv.fx = fv.fy = fv.fj = fsrc; fv.jx0 = fv.jend = fv.lx = n;
        fv.qx = FQ ? FQ + c.poff[sq] : nullptr; fv.qy = fv.qj = fv.qx;
        fv.ring = sm.ring;
        dfl_parse_fresh(st);
        __syncthreads();                                    // the previous sequence is done with the ring
        for (uint32_t i = tid; i < DFL_L_CODES; i += blockDim.x) sm.lf[i] = i == 256 ? 1 : 0;
        for (uint32_t i = tid; i < DFL_D_CODES; i += blockDim.x) sm.df[i] = 0;
        for (uint32_t i = tid * 4; i < tmin(C, n_pad); i += blockDim.x * 4)
            *reinterpret_cast<uint4 *>(sm.ring + i) = __ldg(reinterpret_cast<const uint4 *>(fsrc + i));
        __syncthreads();
        for (uint32_t lo = 0;; lo += C) {
            const uint32_t hi = lo + C;                      // F of [lo, hi) is in the ring
            if (tid >= 32) {                                 // next chunk into the other half
                for (uint32_t i = hi + (tid - 32) * 4; i < tmin(hi + C, n_pad); i += (blockDim.x - 32) * 4)
                    *reinterpret_cast<uint4 *>(sm.ring + (i & (2 * C - 1))) = __ldg(reinterpret_cast<const uint4 *>(fsrc + i));
            } else if (tid == 0) {
                const uint32_t stop_chunk = hi < n ? hi : 0xffffffffu;
                bool done = false;
                for (;;) {
                    const uint32_t stop = ck_done ? stop_chunk : tmin(stop_chunk, jx0);
                    if (dfl_parse(d, fv, cfg, st, sm.lf, 1, sm.df, 1, sm.tr, stop, &rec) == 1) { done = true; break; }
                    if (!ck_done && st.strstart >= jx0) {
                        DflCkpt &ck = ckpt[sq];
                        ck.st = st;
                        for (int k = 0; k < DFL_L_CODES; ++k) ck.lfreq[k] = sm.lf[k];
                        for (int k = 0; k < DFL_D_CODES; ++k) ck.dfreq[k] = sm.df[k];
                        ck_done = true;
                        continue;
                    }
                    break;                                   // the parse stands at or beyond the end of this chunk
                }
                sm.done = done ? 1u : 0u;
            }
            __syncthreads();
            if (sm.done) break;
        }
        if (tid == 0) {
            cp.n_sym[sq] = rec.n == DFL_NONE ? 0u : rec.n;
            cp.seq_size[sq] = (int64_t)(st.bits >> 3);
        }
    }
}

// ---- K3d'': the same products as dfl_prep_kernel for long sequences, in parallel (see "the parse of a sequence
// alone, in parallel").  Chunk k of the i-th listed sequence uses entry coff[i] + k of the per-chunk arrays.
struct DflChunkArgs {
    const int32_t *seqs; const uint64_t *coff; int32_t n_seqs;
    uint32_t *head, *tail;             // per chunk: DFL_CHUNK_WORDS words each
    uint32_t *ysync, *cnt, *off;       // per chunk: y_k, symbols of [y_k, y_{k+1}), their first slot
    int32_t *fail;                     // per listed sequence: chunks that never met / overflow / stored-block candidate
};

__global__ void __launch_bounds__(128)
dfl_chunk_scan_kernel(DflCorpus c, DflChunkArgs a, int level, const uint32_t *__restrict__ F, const uint32_t *__restrict__ FQ)
{
    const DflConfig cfg = dfl_config(level);
    for (int32_t i = blockIdx.y; i < a.n_seqs; i += gridDim.y) {
        const int32_t sq = a.seqs[i];
        const DflStream d = dfl_make_alone(c, sq);
        const uint32_t n = d.s.n, K = dfl_chunk_count(n), E = dfl_chunk_end(n);
        const uint32_t *f = F + c.poff[sq], *q = FQ ? FQ + c.poff[sq] : nullptr;
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
            DflLite o;
            o.mode = 0; o.until = DFL_NONE; o.count = 0; o.end = nullptr; o.code = nullptr; o.cap = 0;
            o.head = a.head + (a.coff[i] + k) * DFL_CHUNK_WORDS;
            o.tail = a.tail + (a.coff[i] + k) * DFL_CHUNK_WORDS;
            for (uint32_t w = 0; w < DFL_CHUNK_WORDS; ++w) o.head[w] = o.tail[w] = 0;
            const uint32_t s_k = k * DFL_CHUNK, s_next = s_k + DFL_CHUNK;
            const bool last = k + 1 == K;
            o.head_lo = k ? s_k : DFL_NOWIN;
            o.tail_lo = last ? DFL_NOWIN : s_next;
            const uint32_t stop = last ? (k ? tmin(s_k + DFL_CHUNK_OV, E) : 0u) : tmin(s_next + DFL_CHUNK_OV, E);
            dfl_lite_parse(d, f, q, cfg, s_k, stop, o);
        }
    }
}

template <int MODE>      // 1: sync points + symbol counts, 2: emit
__global__ void __launch_bounds__(128)
dfl_chunk_pass_kernel(DflCorpus c, DflChunkArgs a, int level, const uint32_t *__restrict__ F, const uint32_t *__restrict__ FQ,
                      DflCanonPool cp)
{
    const DflConfig cfg = dfl_config(level);
    for (int32_t i = blockIdx.y; i < a.n_seqs; i += gridDim.y) {
        if (MODE == 2 && a.fail[i]) continue;
        const int32_t sq = a.seqs[i];
        const DflStream d = dfl_make_alone(c, sq);
        const uint32_t n = d.s.n, K = dfl_chunk_count(n), E = dfl_chunk_end(n);
        const uint32_t *f = F + c.poff[sq], *q = FQ ? FQ + c.poff[sq] : nullptr;
        for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
            const uint64_t e = a.coff[i] + k;
            const bool last = k + 1 == K;
            uint32_t y_k, y_next;
            if (MODE == 1) {
                y_k = k ? dfl_chunk_sync(a.tail + (e - 1) * DFL_CHUNK_WORDS, a.head + e * DFL_CHUNK_WORDS, k * DFL_CHUNK) : 0u;
                y_next = last ? DFL_NONE : dfl_chunk_sync(a.tail + e * DFL_CHUNK_WORDS, a.head + (e + 1) * DFL_CHUNK_WORDS, (k + 1) * DFL_CHUNK);
                a.ysync[e] = y_k;
                if (y_k == DFL_NONE || (!last && y_next == DFL_NONE)) { a.fail[i] = 1; a.cnt[e] = 0; continue; }
            } else {
                y_k = a.ysync[e];
                y_next = last ? DFL_NONE : a.ysync[e + 1];
            }
            DflLite o;
            o.mode = MODE; o.until = y_next; o.count = 0;
            o.head = o.tail = nullptr; o.head_lo = o.tail_lo = DFL_NOWIN;
            o.end = nullptr; o.code = nullptr; o.cap = 0;
            if (MODE == 2) {
                o.end = cp.end + cp.soff[sq] + a.off[e]; o.code = cp.code + cp.soff[sq] + a.off[e]; o.cap = a.cnt[e];
            }
            dfl_lite_parse(d, f, q, cfg, y_k, E, o);
            if (MODE == 1) a.cnt[e] = o.count;
        }
    }
}

// every chunk's first slot; the sequence's symbol count (0 and fail when the symbols do not fit)
__global__ void dfl_chunk_offsets_kernel(DflCorpus c, DflChunkArgs a, DflCanonPool cp)
{
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_seqs) return;
    const int32_t sq = a.seqs[i];
    const uint32_t K = dfl_chunk_count(c.len[sq]);
    uint64_t acc = 0;
    for (uint32_t k = 0; k < K; ++k) { a.off[a.coff[i] + k] = (uint32_t)acc; acc += a.cnt[a.coff[i] + k]; }
    if (acc > cp.cap[sq]) a.fail[i] = 1;
    cp.n_sym[sq] = a.fail[i] ? 0u : (uint32_t)acc;
}

// blocks, size, checkpoint and tail of every listed sequence whose canonical stream stands (up to E) and whose
// cumulative histograms are built: what a pair stream does after its synchronisation point, from symbol 0
constexpr int DFL_ALONE_THREADS = 32;
struct DflAloneSmem {
    DflTrees tr;
    uint32_t accA[DFL_L_CODES + DFL_D_CODES], accB[DFL_L_CODES + DFL_D_CODES];
    uint16_t lf[DFL_L_CODES], df[DFL_D_CODES];
};
__global__ void __launch_bounds__(DFL_ALONE_THREADS)
dfl_alone_kernel(DflCorpus c, DflChunkArgs a, int level, const uint32_t *__restrict__ F, const uint32_t *__restrict__ FQ,
                 DflCkpt *__restrict__ ckpt, DflCanonPool cp)
{
    extern __shared__ __align__(16) uint8_t alone_raw[];
    DflAloneSmem &sm = *reinterpret_cast<DflAloneSmem *>(alone_raw);
    const DflConfig cfg = dfl_config(level);
    for (int32_t i = blockIdx.x; i < a.n_seqs; i += gridDim.x) {
        if (a.fail[i]) continue;
        const int32_t sq = a.seqs[i];
        __syncthreads();
        for (uint32_t k = threadIdx.x; k < DFL_L_CODES; k += blockDim.x) sm.lf[k] = k == 256 ? 1 : 0;
        for (uint32_t k = threadIdx.x; k < DFL_D_CODES; k += blockDim.x) sm.df[k] = 0;
        __syncthreads();
        if (threadIdx.x) continue;
        const DflStream d = dfl_make_alone(c, sq);
        const uint32_t n = d.s.n, jx0 = dfl_jx0(n);
        DflFView fv;
        fv.fx = fv.fy = fv.fj = F + c.poff[sq]; fv.jx0 = fv.jend = fv.lx = n;
        fv.qx = FQ ? FQ + c.poff[sq] : nullptr; fv.qy = fv.qj = fv.qx;
        const DflCanon cn = dfl_canon_of(cp, sq);
        DflParseState st;
        dfl_parse_fresh(st);
        uint32_t t_end = 0;
        const int b = dfl_canon_blocks(cn, 0, n, DFL_NONE, st, sm.lf, 1, sm.df, 1, sm.tr, sm.accA, sm.accB,
                                       (DflCompactTrees *)nullptr, &t_end);
        if (b <= 0) { a.fail[i] = 1; cp.n_sym[sq] = 0; continue; }       // (a block zlib might store: the serial kernel decides)
        DflRec rec{cp.end + cp.soff[sq], cp.code + cp.soff[sq], cp.cap[sq], t_end};
        bool ck_done = false;
        for (;;) {
            const uint32_t stop = ck_done ? 0xffffffffu : jx0;
            if (dfl_parse(d, fv, cfg, st, sm.lf, 1, sm.df, 1, sm.tr, stop, &rec) == 1) break;
            if (!ck_done && st.strstart >= jx0) {
                DflCkpt &ck = ckpt[sq];
                ck.st = st;
                for (int k = 0; k < DFL_L_CODES; ++k) ck.lfreq[k] = sm.lf[k];
                for (int k = 0; k < DFL_D_CODES; ++k) ck.dfreq[k] = sm.df[k];
                ck_done = true;
            }
        }
        cp.n_sym[sq] = rec.n == DFL_NONE ? 0u : rec.n;
        cp.seq_size[sq] = (int64_t)(st.bits >> 3);
    }
}

// K3e: cumulative symbol histograms of the canonical streams.  Step 1: histogram of every complete chunk of
// DFL_CUM_G symbols into row chunk+1; step 2: running sum down the rows (row 0 = zeros).
__global__ void __launch_bounds__(64)
dfl_cum_chunk_kernel(DflCanonPool cp, const int32_t *__restrict__ seqs, int32_t n_seqs)
{
    __shared__ uint32_t h[DFL_CUM_W];
    for (int32_t t = blockIdx.y; t < n_seqs; t += gridDim.y) {
        const int32_t sq = seqs[t];
        const uint32_t n_sym = cp.n_sym[sq];
        const uint16_t *code = cp.code + cp.soff[sq];
        uint32_t *cum = cp.cum + cp.roff[sq] * DFL_CUM_W;
        for (uint32_t chunk = blockIdx.x; (chunk + 1) * DFL_CUM_G <= n_sym; chunk += gridDim.x) {
            for (uint32_t i = threadIdx.x; i < DFL_CUM_W; i += blockDim.x) h[i] = 0;
            __syncthreads();
            for (uint32_t k = threadIdx.x; k < DFL_CUM_G; k += blockDim.x) {
                const uint32_t cd = code[chunk * DFL_CUM_G + k];
                atomicAdd(&h[cd & 511], 1u);
                if ((cd >> 9) != DFL_LIT) atomicAdd(&h[DFL_L_CODES + (cd >> 9)], 1u);
            }
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < DFL_CUM_W; i += blockDim.x) cum[(size_t)(chunk + 1) * DFL_CUM_W + i] = h[i];
            __syncthreads();
        }
    }
}
__global__ void __launch_bounds__(DFL_CUM_W)
dfl_cum_scan_kernel(DflCanonPool cp, const int32_t *__restrict__ seqs, int32_t n_seqs)
{
    for (int32_t t = blockIdx.x; t < n_seqs; t += gridDim.x) {
        const int32_t sq = seqs[t];
        const uint32_t rows = cp.n_sym[sq] / DFL_CUM_G;          // rows 1 .. rows hold chunk histograms
        uint32_t *cum = cp.cum + cp.roff[sq] * DFL_CUM_W + threadIdx.x;
        uint32_t acc = 0;
        cum[0] = 0;
        for (uint32_t r = 1; r <= rows; ++r) { acc += cum[(size_t)r * DFL_CUM_W]; cum[(size_t)r * DFL_CUM_W] = acc; }
    }
}
__global__ void dfl_gather_sizes_kernel(const int64_t *__restrict__ seq_size, const int32_t *__restrict__ xs, int64_t n,
                                        int64_t *__restrict__ out)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = seq_size[xs[k]];
}
#endif  // __CUDACC__

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// host-side orchestration (called from api.cu with the context lock held)
// ------------------------------------------------------------------------------------------------
// Device state of the deflate codecs, split by the role a sequence plays (DflCorpus):
//   x side, every sequence: its record (checkpoint + size alone), its tail 3-byte index (the whole index with
//     deflate_tail_index 0), tail counts and tail 6-byte pack -- what a pair stream x.* needs of x;
//   y side, only the sequences of `ylist` (the current y layout): whole index, F (+ FQ), head order and visits, 6-byte
//     index starts and the canonical symbol stream -- what a pair stream *.y needs of y, and what the parse of a
//     sequence alone needs to produce its record.
// deflate_run plans the y layouts of a call from free device memory: everything in one layout when it fits (the state
// then stays resident for later calls), else bands of y sequences, each prepared, used and dropped in turn.
struct DeflateState {
    int32_t n_seqs = 0;
    // ---- x side ----
    int x_whole = 0;                               // the x index pool holds whole indexes (made with deflate_tail_index 0)
    std::vector<uint64_t> h_xoff; uint64_t x_total = 0;
    uint64_t *d_xoff = nullptr;                    // per sequence: offset of its positions in the x sort scratch window
    uint32_t *d_xindex = nullptr;                  // x index slices: sequence i at h_xoff[i] + i * DFL_BROW
    uint16_t *d_tail_cnt = nullptr, *d_tail6_order = nullptr, *d_tail6_start = nullptr;
    uint32_t *d_ifrom = nullptr; std::vector<uint32_t> h_ifrom;     // first position of every 3-byte index (DflCorpus::ifrom)
    uint32_t *d_cap = nullptr;                     // canonical stream capacity of every sequence (symbols)
    uint32_t **d_ix = nullptr; std::vector<uint32_t *> h_ix;       // where each sequence's 3-byte index is (DflCorpus::ix)
    std::vector<uint8_t> xindexed;                 // x index slice built
    std::vector<uint8_t> have_ckpt[2];             // x-side record present (own parse or imported from another rank)
    DflCkpt *d_ckpt[2] = {nullptr, nullptr};
    int64_t *d_seq_size[2] = {nullptr, nullptr};
    uint32_t *d_nsym[2] = {nullptr, nullptr};
    // per-sequence addressing of the y side (x-side allocations, rewritten with every layout)
    uint64_t *d_poff = nullptr, *d_soff = nullptr, *d_roff = nullptr; uint32_t *d_yslot = nullptr;
    // ---- y side ----
    std::vector<int32_t> ylist;
    std::vector<uint32_t> h_yslot; std::vector<uint64_t> h_poff;
    uint64_t y_total = 0, sym_total = 0, row_total = 0;
    uint32_t *d_yindex = nullptr, *d_bstart6 = nullptr;     // y index slices: sequence i at h_poff[i] + h_yslot[i] * DFL_BROW
    uint16_t *d_head_order = nullptr, *d_head_visit[2] = {nullptr, nullptr};
    uint32_t *d_F[2] = {nullptr, nullptr};         // level 9, level 6
    uint32_t *d_FQ = nullptr;                      // level 6 only: quartered-chain table
    uint32_t *d_sym_end[2] = {nullptr, nullptr}; uint16_t *d_sym_code[2] = {nullptr, nullptr};
    uint32_t *d_cum[2] = {nullptr, nullptr};
    std::vector<uint8_t> yindexed, have_F[2], have_prep[2];
    // ---- working memory ----
    uint32_t *d_rx_hist = nullptr; size_t rx_cap = 0;   // radix-sort digit totals (dfl_build_index)
    uint32_t *d_order6 = nullptr; uint64_t order6_cap = 0;   // 6-byte index window
    uint32_t *d_xtmp = nullptr; uint64_t xtmp_cap = 0;       // sort scratch of x index builds
    DflTrees *d_scratch2[2] = {nullptr, nullptr}; size_t scratch_n[2] = {0, 0};
    uint32_t *d_FJ2[2] = {nullptr, nullptr}, *d_FJQ2[2] = {nullptr, nullptr}; size_t fj_pairs[2] = {0, 0};
    DflPair *d_pairs2[2] = {nullptr, nullptr}; DflJob *d_jobs2[2] = {nullptr, nullptr};
    cudaStream_t stream2 = nullptr; cudaEvent_t ev_j[2] = {nullptr, nullptr}, ev_p[2] = {nullptr, nullptr};
    cudaEvent_t ev_t[2] = {nullptr, nullptr};      // timing of the junction kernel
    unsigned long long *d_counter2 = nullptr;
    // ---- device bytes held, by kind: 0 x side, 1 y side, 2 preparation scratch (released at the end of every call),
    //      3 pair-batch buffers (junction tables, parse scratch, job lists; kept for the next call of the same shape) ----
    std::unordered_map<void *, std::pair<size_t, int>> held;
    size_t live[4] = {0, 0, 0, 0}, peak = 0;
    // ---- switches and statistics ----
    int use_index6 = 1;                            // 0: dfl_match_kernel always walks the 3-byte chain (tests)
    int use_parallel_prep = 1;                     // 0: every sequence alone is parsed by the serial kernel (tests, A/B)
    int use_tail_index = 1;                        // 0: x-role sequences get the whole 3-byte index too (tests, A/B)
    int use_canon = 1;                             // 0: every pair stream takes the full serial parse (tests)
    int junction_impl = 3;                         // 2: no 6-byte-index shortcut in the junction walk (tests)
    int64_t band_bytes = 0;                        // > 0: cap of the y layout of a band (tests); 0: plan from free memory
    int64_t parallel_prep_seqs = 0;                // sequences the chunked path finished in the last call
    int64_t serial_jobs = 0;                       // pair jobs of the last call that fell back to it
    int64_t bands = 0;                             // y layouts the last call went through
    int64_t prepared_seqs = 0;                     // full preparations (index, F, parse alone) the last call made
    double main_ms = 0.0;
};

template <typename T> static cudaError_t dfl_malloc(DeflateState &st, int kind, T **p, size_t bytes)
{
    *p = nullptr;
    const cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) return e;
    st.held[(void *)*p] = {bytes, kind};
    st.live[kind] += bytes;
    st.peak = std::max(st.peak, st.live[0] + st.live[1] + st.live[2] + st.live[3]);
    return e;
}
template <typename T> static void dfl_free(DeflateState &st, T *&p)
{
    if (!p) return;
    auto it = st.held.find((void *)p);
    if (it != st.held.end()) { st.live[it->second.second] -= it->second.first; st.held.erase(it); }
    cudaFree(p);
    p = nullptr;
}

// ---- bytes per sequence of each side (what the planner counts; the allocations below follow the same sums) ----
static inline uint64_t dfl_pad8(uint32_t len) { return ((uint64_t)len + 7) & ~7ull; }
// canonical stream: room for one symbol per 4 bytes (DNA needs one per ~9); a sequence that needs more simply has no
// canonical stream and its pair jobs take the serial parse
static inline uint32_t dfl_canon_cap(uint32_t len) { return (len / 4 + 1024 + DFL_CUM_G - 1) / DFL_CUM_G * DFL_CUM_G; }
static inline uint32_t dfl_xtail_from(uint32_t len) { return len > DFL_XTAIL ? len - DFL_XTAIL : 0u; }
static inline uint64_t dfl_xslot(uint32_t len, int whole) { return whole ? dfl_pad8(len) : std::min<uint64_t>(dfl_pad8(len), DFL_XTAIL); }
static inline uint64_t dfl_xbytes_fixed()
{
    return 4ull * DFL_BROW + 2ull * DFL_HASH + 2ull * DFL_T6 + 2ull * (DFL_H6 + 1)       // bstart, tail counts, tail pack
         + 8 + 4 + 4 + 8 + 8 + 8 + 8 + 4;                                     // xoff ifrom cap ix poff soff roff yslot
}
static inline uint64_t dfl_xbytes_level() { return sizeof(DflCkpt) + 8 + 4; }
static inline uint64_t dfl_ybytes(uint32_t len, int level)
{
    const uint64_t cap = dfl_canon_cap(len);
    return dfl_pad8(len) * 4 * (level == 9 ? 2 : 3)                                 // order, F (, FQ)
         + cap * 6 + (cap / DFL_CUM_G + 1) * DFL_CUM_W * 4                          // symbol ends + codes, cumulative rows
         + 4ull * (DFL_BROW + DFL_HASH + 1) + 4ull * DFL_JY                         // bucket starts (3-, 6-byte), head order + visits
         + (uint64_t)dfl_chunk_count(len) * (2 * DFL_CHUNK_WORDS + 3) * 4;          // chunk scratch of the parallel parse
}

static inline void deflate_drop_y(DeflateState &st)
{
    dfl_free(st, st.d_yindex); dfl_free(st, st.d_bstart6); dfl_free(st, st.d_head_order);
    dfl_free(st, st.d_FQ);
    for (int l = 0; l < 2; ++l) {
        dfl_free(st, st.d_F[l]); dfl_free(st, st.d_head_visit[l]);
        dfl_free(st, st.d_sym_end[l]); dfl_free(st, st.d_sym_code[l]); dfl_free(st, st.d_cum[l]);
        std::fill(st.have_F[l].begin(), st.have_F[l].end(), 0);
        std::fill(st.have_prep[l].begin(), st.have_prep[l].end(), 0);
    }
    for (int32_t i : st.ylist) { st.h_yslot[i] = DFL_NONE; st.yindexed[i] = 0; }
    st.ylist.clear();
    st.y_total = st.sym_total = st.row_total = 0;
}
static inline void deflate_free_corpus(DeflateState &st)
{
    deflate_drop_y(st);
    dfl_free(st, st.d_xoff); dfl_free(st, st.d_xindex);
    dfl_free(st, st.d_tail_cnt); dfl_free(st, st.d_tail6_order); dfl_free(st, st.d_tail6_start);
    dfl_free(st, st.d_ifrom); dfl_free(st, st.d_cap); dfl_free(st, st.d_ix);
    dfl_free(st, st.d_poff); dfl_free(st, st.d_soff); dfl_free(st, st.d_roff); dfl_free(st, st.d_yslot);
    dfl_free(st, st.d_bstart6); dfl_free(st, st.d_order6); st.order6_cap = 0;
    dfl_free(st, st.d_rx_hist); st.rx_cap = 0;
    dfl_free(st, st.d_xtmp); st.xtmp_cap = 0;
    for (int l = 0; l < 2; ++l) {
        dfl_free(st, st.d_ckpt[l]); dfl_free(st, st.d_seq_size[l]); dfl_free(st, st.d_nsym[l]);
        st.have_F[l].clear(); st.have_prep[l].clear(); st.have_ckpt[l].clear();
    }
    st.h_xoff.clear(); st.h_ifrom.clear(); st.h_ix.clear(); st.xindexed.clear();
    st.h_yslot.clear(); st.h_poff.clear(); st.yindexed.clear();
    st.n_seqs = 0; st.x_total = 0;
}
// the pair-batch buffers (junction tables, parse scratch, job lists)
static inline void deflate_free_batches(DeflateState &st)
{
    for (int k = 0; k < 2; ++k) {
        dfl_free(st, st.d_scratch2[k]); dfl_free(st, st.d_FJ2[k]); dfl_free(st, st.d_FJQ2[k]);
        dfl_free(st, st.d_pairs2[k]); dfl_free(st, st.d_jobs2[k]);
        st.scratch_n[k] = st.fj_pairs[k] = 0;
    }
}
static inline void deflate_free_work(DeflateState &st)
{
    deflate_free_batches(st);
    for (int k = 0; k < 2; ++k) {
        if (st.ev_j[k]) cudaEventDestroy(st.ev_j[k]);
        if (st.ev_p[k]) cudaEventDestroy(st.ev_p[k]);
        if (st.ev_t[k]) cudaEventDestroy(st.ev_t[k]);
        st.ev_j[k] = st.ev_p[k] = st.ev_t[k] = nullptr;
    }
    if (st.stream2) cudaStreamDestroy(st.stream2);
    st.stream2 = nullptr;
    dfl_free(st, st.d_counter2);
}
static inline void deflate_invalidate(DeflateState &st)
{
    std::fill(st.xindexed.begin(), st.xindexed.end(), 0);
    std::fill(st.yindexed.begin(), st.yindexed.end(), 0);
    for (int l = 0; l < 2; ++l) {
        std::fill(st.have_F[l].begin(), st.have_F[l].end(), 0);
        std::fill(st.have_prep[l].begin(), st.have_prep[l].end(), 0);
        std::fill(st.have_ckpt[l].begin(), st.have_ckpt[l].end(), 0);
    }
}

template <typename T> static int dfl_upload(std::string &err, cudaStream_t stream, const std::vector<T> &h, T **d)
{
    *d = nullptr;
    if (h.empty()) return 0;
    DCK(cudaMalloc(d, sizeof(T) * h.size()));
    DCK(cudaMemcpyAsync(*d, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice, stream));
    return 0;
}

constexpr int DFL_PARSE_BLOCKS = 148 * 5;           // parse threads a batch is sized for (the kernel's CTAs loop over jobs)
constexpr size_t DFL_BATCH = (size_t)DFL_PARSE_BLOCKS * 64;   // pair streams per junction batch: one per parse thread (6.3 GB of
                                                    // junction F per buffer, two buffers; the parse is latency-bound, so
                                                    // its throughput is the number of streams in flight)
constexpr uint64_t DFL_ORDER6_CAP = 192ull << 20;   // entries of the 6-byte index window: 768 MB at most
constexpr int DFL_INDEX_GROUP = 64;                 // sequences per index build

// build the KIND index of the listed sequences (radix sort, bucket starts); tmp: one scratch entry per position,
// addressed like the F slices (c.poff)
template <int KIND>
static int dfl_build_index(DeflateState &st, const DflCorpus &c, const std::vector<int32_t> &list, const uint32_t *h_len,
                           uint32_t *tmp, cudaStream_t stream, int64_t *launches, std::string &err)
{
    if (list.empty()) return 0;
    uint32_t mx = 0;
    for (int32_t i : list) {
        const uint32_t cnt = dfl_index_count<KIND>(h_len[i]), first = KIND == 0 ? st.h_ifrom[i] : 0u;
        mx = std::max(mx, cnt > first ? cnt - first : 0u);
    }
    const uint32_t max_tiles = std::max(1u, dfl_rx_tiles(mx));
    const size_t need = list.size() * 256 * (size_t)max_tiles;
    if (st.rx_cap < need) {
        dfl_free(st, st.d_rx_hist); st.rx_cap = 0;
        DCK(dfl_malloc(st, 2, &st.d_rx_hist, sizeof(uint32_t) * need));
        st.rx_cap = need;
    }
    int32_t *d_list = nullptr;
    if (dfl_upload(err, stream, list, &d_list)) return -1;
    const dim3 grid(max_tiles, (unsigned)list.size());
    uint32_t *order = KIND == 0 ? nullptr : c.order6;                  // (KIND 0: the slices of c.ix)
    DCK(cudaMemsetAsync(st.d_rx_hist, 0, sizeof(uint32_t) * need, stream));
    dfl_radix_kernel<KIND, 0, false><<<grid, DFL_RX_THREADS, 0, stream>>>(c, d_list, max_tiles, st.d_rx_hist, tmp, tmp);
    dfl_radix_scan_kernel<<<(unsigned)list.size(), 1024, 0, stream>>>(max_tiles, st.d_rx_hist);
    dfl_radix_kernel<KIND, 0, true><<<grid, DFL_RX_THREADS, 0, stream>>>(c, d_list, max_tiles, st.d_rx_hist, tmp, tmp);
    DCK(cudaMemsetAsync(st.d_rx_hist, 0, sizeof(uint32_t) * need, stream));
    dfl_radix_kernel<KIND, 1, false><<<grid, DFL_RX_THREADS, 0, stream>>>(c, d_list, max_tiles, st.d_rx_hist, tmp, order);
    dfl_radix_scan_kernel<<<(unsigned)list.size(), 1024, 0, stream>>>(max_tiles, st.d_rx_hist);
    dfl_radix_kernel<KIND, 1, true><<<grid, DFL_RX_THREADS, 0, stream>>>(c, d_list, max_tiles, st.d_rx_hist, tmp, order);
    dfl_index_fill_kernel<KIND><<<(unsigned)list.size(), 1024, 0, stream>>>(c, d_list, 0);
    dfl_index_bounds_kernel<KIND><<<dim3(std::max(1u, std::min((mx + 255) / 256, 1024u)), (unsigned)list.size()), 256, 0, stream>>>(c, d_list);
    dfl_index_fill_kernel<KIND><<<(unsigned)list.size(), 1024, 0, stream>>>(c, d_list, 1);
    DCK(cudaGetLastError());
    *launches += 9;
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_list);
    return 0;
}

// x side of every sequence (allocated on first use, and again when the x index layout changes)
static int deflate_ensure_x(DeflateState &st, const Corpus &dc, int level, cudaStream_t stream, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    const int32_t ns = dc.n_seqs;
    const int whole = st.use_tail_index ? 0 : 1;
    if (st.n_seqs != ns || !st.d_xoff) {
        deflate_free_corpus(st);
        st.n_seqs = ns;
        std::vector<uint32_t> cap(ns);
        for (int32_t i = 0; i < ns; ++i) cap[i] = dfl_canon_cap(dc.h_len[i]);
        DCK(dfl_malloc(st, 0, &st.d_xoff, sizeof(uint64_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_tail_cnt, sizeof(uint16_t) * (size_t)ns * DFL_HASH));
        DCK(dfl_malloc(st, 0, &st.d_tail6_order, sizeof(uint16_t) * (size_t)ns * DFL_T6));
        DCK(dfl_malloc(st, 0, &st.d_tail6_start, sizeof(uint16_t) * (size_t)ns * (DFL_H6 + 1)));
        DCK(dfl_malloc(st, 0, &st.d_ifrom, sizeof(uint32_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_cap, sizeof(uint32_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_ix, sizeof(uint32_t *) * ns));
        DCK(dfl_malloc(st, 0, &st.d_poff, sizeof(uint64_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_soff, sizeof(uint64_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_roff, sizeof(uint64_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_yslot, sizeof(uint32_t) * ns));
        DCK(cudaMemcpyAsync(st.d_cap, cap.data(), sizeof(uint32_t) * ns, cudaMemcpyHostToDevice, stream));
        DCK(cudaMemsetAsync(st.d_ifrom, 0, sizeof(uint32_t) * ns, stream));
        DCK(cudaStreamSynchronize(stream));
        st.h_ifrom.assign(ns, 0); st.h_ix.assign(ns, nullptr); st.xindexed.assign(ns, 0);
        st.h_yslot.assign(ns, DFL_NONE); st.h_poff.assign(ns, 0); st.yindexed.assign(ns, 0);
        for (int l = 0; l < 2; ++l) { st.have_F[l].assign(ns, 0); st.have_prep[l].assign(ns, 0); st.have_ckpt[l].assign(ns, 0); }
        st.x_whole = -1;
    }
    if (st.x_whole != whole) {
        dfl_free(st, st.d_xindex);
        std::fill(st.xindexed.begin(), st.xindexed.end(), 0);
        st.h_xoff.assign(ns, 0);
        uint64_t t = 0;
        for (int32_t i = 0; i < ns; ++i) { st.h_xoff[i] = t; t += dfl_xslot(dc.h_len[i], whole); }
        st.x_total = t;
        DCK(dfl_malloc(st, 0, &st.d_xindex, sizeof(uint32_t) * (t + (uint64_t)ns * DFL_BROW + 16)));
        DCK(cudaMemcpyAsync(st.d_xoff, st.h_xoff.data(), sizeof(uint64_t) * ns, cudaMemcpyHostToDevice, stream));
        DCK(cudaStreamSynchronize(stream));
        st.x_whole = whole;
    }
    if (!st.d_ckpt[li]) {
        DCK(dfl_malloc(st, 0, &st.d_ckpt[li], sizeof(DflCkpt) * ns));
        DCK(dfl_malloc(st, 0, &st.d_seq_size[li], sizeof(int64_t) * ns));
        DCK(dfl_malloc(st, 0, &st.d_nsym[li], sizeof(uint32_t) * ns));
        DCK(cudaMemsetAsync(st.d_nsym[li], 0, sizeof(uint32_t) * ns, stream));
    }
    return 0;
}

// the per-level arrays of the current y layout
static int deflate_alloc_y_level(DeflateState &st, int level, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    if (st.ylist.empty() || st.d_F[li]) return 0;
    const size_t ny = st.ylist.size();
    DCK(dfl_malloc(st, 1, &st.d_F[li], sizeof(uint32_t) * (st.y_total + 16)));
    if (level != 9 && !st.d_FQ) DCK(dfl_malloc(st, 1, &st.d_FQ, sizeof(uint32_t) * (st.y_total + 16)));
    DCK(dfl_malloc(st, 1, &st.d_head_visit[li], sizeof(uint16_t) * ny * DFL_JY));
    DCK(dfl_malloc(st, 1, &st.d_sym_end[li], sizeof(uint32_t) * (st.sym_total + 16)));
    DCK(dfl_malloc(st, 1, &st.d_sym_code[li], sizeof(uint16_t) * (st.sym_total + 16)));
    DCK(dfl_malloc(st, 1, &st.d_cum[li], sizeof(uint32_t) * st.row_total * DFL_CUM_W));
    return 0;
}
// (a failed allocation -- the device is shared -- leaves no layout rather than a layout with missing arrays)
static int deflate_ensure_y_level(DeflateState &st, int level, std::string &err)
{
    if (deflate_alloc_y_level(st, level, err)) { deflate_drop_y(st); return -1; }
    return 0;
}

static int deflate_layout_arrays(DeflateState &st, const Corpus &dc, int level, const std::vector<int32_t> &list,
                                 cudaStream_t stream, std::string &err)
{
    deflate_drop_y(st);
    const int32_t ns = dc.n_seqs;
    std::vector<uint64_t> soff(ns, 0), roff(ns, 0);
    uint64_t t = 0, sy = 0, ro = 0;
    for (size_t k = 0; k < list.size(); ++k) {
        const int32_t i = list[k];
        const uint32_t cap = dfl_canon_cap(dc.h_len[i]);
        st.h_yslot[i] = (uint32_t)k;
        st.h_poff[i] = t; t += dfl_pad8(dc.h_len[i]);
        soff[i] = sy; sy += cap;
        roff[i] = ro; ro += cap / DFL_CUM_G + 1;
    }
    st.ylist = list;
    st.y_total = t; st.sym_total = sy; st.row_total = ro;
    DCK(cudaMemcpyAsync(st.d_poff, st.h_poff.data(), sizeof(uint64_t) * ns, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(st.d_soff, soff.data(), sizeof(uint64_t) * ns, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(st.d_roff, roff.data(), sizeof(uint64_t) * ns, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(st.d_yslot, st.h_yslot.data(), sizeof(uint32_t) * ns, cudaMemcpyHostToDevice, stream));
    DCK(cudaStreamSynchronize(stream));
    const size_t ny = list.size();
    DCK(dfl_malloc(st, 1, &st.d_yindex, sizeof(uint32_t) * (t + ny * DFL_BROW + 16)));
    DCK(dfl_malloc(st, 1, &st.d_bstart6, sizeof(uint32_t) * ny * (DFL_HASH + 1)));
    DCK(dfl_malloc(st, 1, &st.d_head_order, sizeof(uint16_t) * ny * DFL_JY));
    return deflate_alloc_y_level(st, level, err);
}
// a new y layout holding exactly `list` (ascending): the previous one is dropped; on failure there is no layout
static int deflate_set_layout(DeflateState &st, const Corpus &dc, int level, const std::vector<int32_t> &list,
                              cudaStream_t stream, std::string &err)
{
    if (deflate_layout_arrays(st, dc, level, list, stream, err)) { deflate_drop_y(st); return -1; }
    return 0;
}

// every sequence's 3-byte index: the whole one while it is in the y layout and built, else its x slice
static int deflate_upload_ix(DeflateState &st, cudaStream_t stream, std::string &err)
{
    for (int32_t i = 0; i < st.n_seqs; ++i)
        st.h_ix[i] = st.yindexed[i] ? st.d_yindex + st.h_poff[i] + (size_t)st.h_yslot[i] * DFL_BROW
                                    : st.d_xindex + st.h_xoff[i] + (size_t)i * DFL_BROW;
    DCK(cudaMemcpyAsync(st.d_ix, st.h_ix.data(), sizeof(uint32_t *) * st.n_seqs, cudaMemcpyHostToDevice, stream));
    DCK(cudaStreamSynchronize(stream));
    return 0;
}

static DflCorpus deflate_corpus(const DeflateState &st, const Corpus &dc, int li)
{
    return DflCorpus{dc.d_corpus, dc.d_off, dc.d_len, st.d_poff, st.d_ix, st.d_yslot, st.d_yindex,
                     st.d_head_order, st.d_head_visit[li],
                     st.d_tail_cnt, st.d_tail6_order, st.d_tail6_start, nullptr, st.d_bstart6, st.d_ifrom};
}

// the head order / tail counts and tail packs of sequences whose 3-byte index was just built
static int dfl_index_packs(const DflCorpus &c, const std::vector<int32_t> &list, cudaStream_t stream, int64_t *launches,
                           std::string &err)
{
    int32_t *d_list = nullptr;
    if (dfl_upload(err, stream, list, &d_list)) return -1;
    DCK(cudaFuncSetAttribute(dfl_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(DFL_HASH * 4)));
    dfl_head_kernel<<<(unsigned)std::min<size_t>(list.size(), 148), 1024, DFL_HASH * 4, stream>>>(c, d_list, (int32_t)list.size());
    DCK(cudaGetLastError());
    const int t6_smem = (int)(DFL_H6 * 4 + DFL_T6 * 2);
    DCK(cudaFuncSetAttribute(dfl_tail6_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, t6_smem));
    dfl_tail6_kernel<<<(unsigned)std::min<size_t>(list.size(), 148 * 2), 32, t6_smem, stream>>>(c, d_list, (int32_t)list.size());
    DCK(cudaGetLastError());
    *launches += 3;
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_list);
    return 0;
}

// x index slices of the listed sequences (their last DFL_XTAIL positions, or whole with deflate_tail_index 0): the
// junction walks of a pair stream x.y reach at most 264 + 32 768 positions back from the end of x
static int deflate_build_x(DeflateState &st, const Corpus &dc, int li, const std::vector<int32_t> &list,
                           cudaStream_t stream, int64_t *launches, std::string &err)
{
    if (list.empty()) return 0;
    NvtxRange nvtx_("snacc_b200: deflate x index (radix sort, tail packs)");
    // window: the slices of up to DFL_INDEX_GROUP x-tail sequences, at least one whole slice (deflate_tail_index 0)
    uint64_t sum = 0, big = 0;
    for (int32_t i : list) { const uint64_t n = dfl_xslot(dc.h_len[i], st.x_whole); sum += n; big = std::max(big, n); }
    const uint64_t cap = std::max(big, std::min<uint64_t>(sum, (uint64_t)DFL_INDEX_GROUP * DFL_XTAIL));
    if (st.xtmp_cap < cap) { dfl_free(st, st.d_xtmp); st.xtmp_cap = 0; DCK(dfl_malloc(st, 2, &st.d_xtmp, sizeof(uint32_t) * (cap + 16))); st.xtmp_cap = cap; }
    for (int32_t i : list) { st.h_ifrom[i] = st.x_whole ? 0u : dfl_xtail_from(dc.h_len[i]); st.xindexed[i] = 1; }
    if (deflate_upload_ix(st, stream, err)) return -1;
    DCK(cudaMemcpyAsync(st.d_ifrom, st.h_ifrom.data(), sizeof(uint32_t) * st.n_seqs, cudaMemcpyHostToDevice, stream));
    DflCorpus c = deflate_corpus(st, dc, li);
    for (int32_t i : list) if (st.yindexed[i]) { err = "deflate_build_x: sequence holds its whole index"; return -1; }
    c.poff = st.d_xoff;                                                // sort scratch: a window addressed like the x slices
    c.head_order = nullptr;                                            // tail counts only
    size_t a = 0;
    while (a < list.size()) {
        size_t b = a + 1;
        const uint64_t first = st.h_xoff[list[a]];
        while (b < list.size() && b - a < (size_t)DFL_INDEX_GROUP &&
               st.h_xoff[list[b]] + dfl_xslot(dc.h_len[list[b]], st.x_whole) - first <= st.xtmp_cap) ++b;
        std::vector<int32_t> part(list.begin() + a, list.begin() + b);
        if (dfl_build_index<0>(st, c, part, dc.h_len, st.d_xtmp - first, stream, launches, err)) return -1;
        a = b;
    }
    return dfl_index_packs(c, list, stream, launches, err);
}

// the full preparation of the listed sequences of the y layout that lack it: whole index, F of this level and the
// parse of the sequence alone (size, checkpoint, canonical symbol stream)
static int deflate_prepare_y(DeflateState &st, const Corpus &dc, int level, const std::vector<int32_t> &list,
                             cudaStream_t stream, int64_t *launches, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    std::vector<int32_t> need_idx, need_f, need_prep;
    for (int32_t i : list) {
        if (!st.yindexed[i]) { need_idx.push_back(i); st.have_F[0][i] = st.have_F[1][i] = 0; }
        if (!st.have_F[li][i] || !st.yindexed[i]) { need_f.push_back(i); st.have_prep[li][i] = 0; }
        if (!st.have_prep[li][i]) need_prep.push_back(i);
    }
    if (need_prep.empty()) return 0;
    st.prepared_seqs += (int64_t)need_prep.size();
    uint32_t *FQ = level != 9 ? st.d_FQ : nullptr;
    if (!need_idx.empty()) {
        NvtxRange nvtx_("snacc_b200: deflate index (radix sort, head/tail packs)");
        for (int32_t i : need_idx) { st.yindexed[i] = 1; st.h_ifrom[i] = 0; }
        if (deflate_upload_ix(st, stream, err)) return -1;
        DCK(cudaMemcpyAsync(st.d_ifrom, st.h_ifrom.data(), sizeof(uint32_t) * st.n_seqs, cudaMemcpyHostToDevice, stream));
        const DflCorpus c = deflate_corpus(st, dc, li);
        // the F slices of this level double as sort scratch; they are recomputed right below
        for (size_t a0 = 0; a0 < need_idx.size(); a0 += DFL_INDEX_GROUP) {
            std::vector<int32_t> part(need_idx.begin() + a0, need_idx.begin() + std::min(need_idx.size(), a0 + DFL_INDEX_GROUP));
            if (dfl_build_index<0>(st, c, part, dc.h_len, st.d_F[li], stream, launches, err)) return -1;
        }
        if (dfl_index_packs(c, need_idx, stream, launches, err)) return -1;
    }
    const DflCorpus c = deflate_corpus(st, dc, li);
    if (!need_f.empty()) {
        NvtxRange nvtx_("snacc_b200: deflate match tables");
        // level 9: runs of sequences whose index slices fit the window buffer get a transient 6-byte index first
        // (dfl_match_word); level 6 always walks the chain (its limit of 128 binds everywhere on DNA)
        const bool i6 = st.use_index6 && level == 9;
        const uint64_t cap = std::min<uint64_t>(DFL_ORDER6_CAP, st.y_total);
        if (i6 && st.order6_cap < cap) {
            dfl_free(st, st.d_order6); st.order6_cap = 0;
            DCK(dfl_malloc(st, 2, &st.d_order6, sizeof(uint32_t) * (cap + 16))); st.order6_cap = cap;
        }
        size_t a = 0;
        while (a < need_f.size()) {
            size_t b = a + 1;
            const uint64_t first = st.h_poff[need_f[a]];
            auto end_of = [&](int32_t i) { return st.h_poff[i] + dfl_pad8(dc.h_len[i]); };
            while (b < need_f.size() && b - a < 64 && (!i6 || end_of(need_f[b]) - first <= st.order6_cap)) ++b;
            const bool fits = i6 && end_of(need_f[b - 1]) - first <= st.order6_cap;   // (a single sequence longer than the buffer: no index)
            std::vector<int32_t> part(need_f.begin() + a, need_f.begin() + b);
            int32_t *d_list = nullptr;
            if (dfl_upload(err, stream, part, &d_list)) return -1;
            DflCorpus cm = c;
            if (fits) {
                cm.order6 = st.d_order6 - first;                               // addressed like F: + poff[sq]
                if (dfl_build_index<1>(st, cm, part, dc.h_len, st.d_F[li], stream, launches, err)) return -1;
            }
            uint32_t mx = 0;
            for (int32_t i : part) mx = std::max(mx, dc.h_len[i]);
            dim3 grid(std::max(1u, std::min((mx + 255) / 256, 4096u)), (unsigned)part.size());
            dfl_match_kernel<<<grid, 256, 0, stream>>>(cm, d_list, (int32_t)part.size(), level, st.d_F[li], FQ);
            DCK(cudaGetLastError());
            ++*launches;
            DCK(cudaStreamSynchronize(stream));
            cudaFree(d_list);
            for (int32_t i : part) st.have_F[li][i] = 1;
            a = b;
        }
    }
    DflCanonPool cp{st.d_sym_end[li], st.d_sym_code[li], st.d_cum[li], st.d_soff, st.d_cap, st.d_roff, st.d_nsym[li],
                    st.d_seq_size[li]};
    NvtxRange nvtx_("snacc_b200: deflate sequence parses (sizes, checkpoints, canonical streams)");
    // long sequences: chunks in parallel (dfl_chunk_*_kernel), then cumulative rows, then dfl_alone_kernel; the
    // others -- and whatever the parallel path gives up on -- take the serial kernel
    std::vector<int32_t> par, ser;
    for (int32_t i : need_prep) (st.use_parallel_prep && dc.h_len[i] >= DFL_PAR_MIN ? par : ser).push_back(i);
    auto run_serial = [&](const std::vector<int32_t> &list) -> int {
        if (list.empty()) return 0;
        int32_t *d_list = nullptr;
        if (dfl_upload(err, stream, list, &d_list)) return -1;
        DCK(cudaFuncSetAttribute(dfl_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DflPrepSmem)));
        dfl_prep_kernel<<<(unsigned)std::min<size_t>(list.size(), 148 * 5), DFL_PREP_THREADS, sizeof(DflPrepSmem), stream>>>(
            c, d_list, (int32_t)list.size(), level, st.d_F[li], FQ, st.d_ckpt[li], cp);
        DCK(cudaGetLastError());
        ++*launches;
        DCK(cudaStreamSynchronize(stream));
        cudaFree(d_list);
        return 0;
    };
    auto run_cum = [&](const std::vector<int32_t> &list) -> int {
        if (list.empty()) return 0;
        int32_t *d_list = nullptr;
        if (dfl_upload(err, stream, list, &d_list)) return -1;
        uint32_t max_rows = 1;
        for (int32_t i : list) max_rows = std::max(max_rows, dc.h_len[i] / 4 / DFL_CUM_G + 8);
        dim3 grid(std::min(max_rows, 2048u), (unsigned)std::min<size_t>(list.size(), 64));
        dfl_cum_chunk_kernel<<<grid, 64, 0, stream>>>(cp, d_list, (int32_t)list.size());
        dfl_cum_scan_kernel<<<(unsigned)std::min<size_t>(list.size(), 148 * 4), DFL_CUM_W, 0, stream>>>(
            cp, d_list, (int32_t)list.size());
        DCK(cudaGetLastError());
        *launches += 2;
        DCK(cudaStreamSynchronize(stream));
        cudaFree(d_list);
        return 0;
    };
    if (!par.empty()) {
        // per-chunk scratch of the listed sequences (2 x 128 B of bitmaps + 12 B per 8 KiB chunk)
        std::vector<uint64_t> coff(par.size() + 1, 0);
        uint32_t max_k = 1;
        for (size_t k = 0; k < par.size(); ++k) {
            const uint32_t K = dfl_chunk_count(dc.h_len[par[k]]);
            coff[k + 1] = coff[k] + K; max_k = std::max(max_k, K);
        }
        const uint64_t tot = coff.back();
        int32_t *d_list = nullptr; uint64_t *d_coff = nullptr; uint32_t *d_w = nullptr; int32_t *d_fail = nullptr;
        if (dfl_upload(err, stream, par, &d_list)) return -1;
        auto free_all = [&]() { cudaFree(d_list); cudaFree(d_coff); dfl_free(st, d_w); cudaFree(d_fail); };
        if (cudaMalloc(&d_coff, sizeof(uint64_t) * coff.size()) != cudaSuccess ||
            dfl_malloc(st, 2, &d_w, sizeof(uint32_t) * tot * (2 * DFL_CHUNK_WORDS + 3)) != cudaSuccess ||
            cudaMalloc(&d_fail, sizeof(int32_t) * par.size()) != cudaSuccess) { free_all(); err = "cudaMalloc (chunk scratch) failed"; return -1; }
        cudaMemcpyAsync(d_coff, coff.data(), sizeof(uint64_t) * coff.size(), cudaMemcpyHostToDevice, stream);
        cudaMemsetAsync(d_fail, 0, sizeof(int32_t) * par.size(), stream);
        DflChunkArgs a{d_list, d_coff, (int32_t)par.size(), d_w, d_w + tot * DFL_CHUNK_WORDS, d_w + tot * 2 * DFL_CHUNK_WORDS,
                       d_w + tot * (2 * DFL_CHUNK_WORDS + 1), d_w + tot * (2 * DFL_CHUNK_WORDS + 2), d_fail};
        dim3 grid((max_k + 127) / 128, (unsigned)std::min<size_t>(par.size(), 65535));
        dfl_chunk_scan_kernel<<<grid, 128, 0, stream>>>(c, a, level, st.d_F[li], FQ);
        dfl_chunk_pass_kernel<1><<<grid, 128, 0, stream>>>(c, a, level, st.d_F[li], FQ, cp);
        dfl_chunk_offsets_kernel<<<(unsigned)((par.size() + 63) / 64), 64, 0, stream>>>(c, a, cp);
        dfl_chunk_pass_kernel<2><<<grid, 128, 0, stream>>>(c, a, level, st.d_F[li], FQ, cp);
        *launches += 4;
        std::vector<int32_t> fail(par.size(), 0);
        if (cudaGetLastError() != cudaSuccess ||
            cudaMemcpyAsync(fail.data(), d_fail, sizeof(int32_t) * par.size(), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
            cudaStreamSynchronize(stream) != cudaSuccess) { free_all(); err = "deflate chunk kernels failed"; return -1; }
        std::vector<int32_t> ok;
        for (size_t k = 0; k < par.size(); ++k) (fail[k] ? ser : ok).push_back(par[k]);
        if (run_serial(ser) || run_cum(need_prep)) { free_all(); return -1; }
        ser.clear();
        if (!ok.empty()) {
            // the sequences that stand: compact list (fail flags restart at 0)
            cudaMemcpyAsync(d_list, ok.data(), sizeof(int32_t) * ok.size(), cudaMemcpyHostToDevice, stream);
            cudaMemsetAsync(d_fail, 0, sizeof(int32_t) * ok.size(), stream);
            a.n_seqs = (int32_t)ok.size();
            cudaFuncSetAttribute(dfl_alone_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DflAloneSmem));
            dfl_alone_kernel<<<(unsigned)std::min<size_t>(ok.size(), 148 * 8), DFL_ALONE_THREADS, sizeof(DflAloneSmem), stream>>>(
                c, a, level, st.d_F[li], FQ, st.d_ckpt[li], cp);
            ++*launches;
            fail.assign(ok.size(), 0);
            if (cudaGetLastError() != cudaSuccess ||
                cudaMemcpyAsync(fail.data(), d_fail, sizeof(int32_t) * ok.size(), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
                cudaStreamSynchronize(stream) != cudaSuccess) { free_all(); err = "dfl_alone_kernel failed"; return -1; }
            std::vector<int32_t> redo;
            for (size_t k = 0; k < ok.size(); ++k) if (fail[k]) redo.push_back(ok[k]);
            st.parallel_prep_seqs += (int64_t)(ok.size() - redo.size());
            if (run_serial(redo) || run_cum(redo)) { free_all(); return -1; }
        }
        free_all();
    } else {
        if (run_serial(ser) || run_cum(need_prep)) return -1;
    }
    for (int32_t i : need_prep) { st.have_prep[li][i] = 1; st.have_ckpt[li][i] = 1; }
    return 0;
}

// The x-side product of a sequence -- what every pair stream x.* needs of x: the parse checkpoint at its junction
// start and the size of x alone -- as a flat record, so that ranks which prepared different sequences can exchange
// them (sharding.py: each rank parses its own band of sequences, one all-gather of these records).
struct DflPrefixRecord { DflCkpt ck; int64_t size; };

static int deflate_export_prefix(DeflateState &st, const Corpus &dc, int level, const int32_t *seqs, int64_t n,
                                 DflPrefixRecord *out, cudaStream_t stream, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    if (!st.d_ckpt[li] || st.n_seqs != dc.n_seqs) { err = "deflate_export_prefix: nothing prepared"; return -1; }
    for (int64_t k = 0; k < n; ++k) {
        const int32_t i = seqs[k];
        if (i < 0 || i >= dc.n_seqs || !st.have_ckpt[li][i]) { err = "deflate_export_prefix: sequence not prepared"; return -1; }
        DCK(cudaMemcpyAsync(&out[k].ck, st.d_ckpt[li] + i, sizeof(DflCkpt), cudaMemcpyDeviceToHost, stream));
        DCK(cudaMemcpyAsync(&out[k].size, st.d_seq_size[li] + i, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    }
    DCK(cudaStreamSynchronize(stream));
    return 0;
}

static int deflate_import_prefix(DeflateState &st, const Corpus &dc, int level, const int32_t *seqs, int64_t n,
                                 const DflPrefixRecord *in, cudaStream_t stream, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    if (deflate_ensure_x(st, dc, level, stream, err)) return -1;
    for (int64_t k = 0; k < n; ++k) {
        const int32_t i = seqs[k];
        if (i < 0 || i >= dc.n_seqs) { err = "deflate_import_prefix: sequence index out of range"; return -1; }
        if (st.have_ckpt[li][i]) continue;                      // this rank parsed it itself
        DCK(cudaMemcpyAsync(st.d_ckpt[li] + i, &in[k].ck, sizeof(DflCkpt), cudaMemcpyHostToDevice, stream));
        DCK(cudaMemcpyAsync(st.d_seq_size[li] + i, &in[k].size, sizeof(int64_t), cudaMemcpyHostToDevice, stream));
        st.have_ckpt[li][i] = 1;
    }
    DCK(cudaStreamSynchronize(stream));
    return 0;
}

// pair jobs (all, or the listed subset) through the junction / parse batches; sizes land at d_out[job]
static int deflate_pairs(DeflateState &st, const Corpus &dc, int level, const int32_t *xs, const int32_t *ys,
                         int64_t n_jobs, const std::vector<int64_t> *subset, int kind, size_t batch, int64_t *d_out,
                         cudaStream_t stream, int64_t *launches, std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    uint32_t *FQ = level != 9 ? st.d_FQ : nullptr;
    const int64_t total = subset ? (int64_t)subset->size() : n_jobs;
    if (!total) return 0;
    const int nbuf = total > (int64_t)batch ? 2 : 1;
    const int parse_blocks = (int)std::min<size_t>(DFL_PARSE_BLOCKS, (batch + DFL_PARSE_THREADS - 1) / DFL_PARSE_THREADS);
    for (int k = 0; k < nbuf; ++k) {
        if (st.scratch_n[k] < (size_t)parse_blocks * DFL_PARSE_THREADS) {
            dfl_free(st, st.d_scratch2[k]); st.scratch_n[k] = 0;
            DCK(dfl_malloc(st, 3, &st.d_scratch2[k], sizeof(DflTrees) * (size_t)parse_blocks * DFL_PARSE_THREADS));
            st.scratch_n[k] = (size_t)parse_blocks * DFL_PARSE_THREADS;
        }
        if (st.fj_pairs[k] < batch) {
            dfl_free(st, st.d_FJ2[k]); dfl_free(st, st.d_FJQ2[k]); dfl_free(st, st.d_pairs2[k]); dfl_free(st, st.d_jobs2[k]);
            st.fj_pairs[k] = 0;
            DCK(dfl_malloc(st, 3, &st.d_FJ2[k], sizeof(uint32_t) * batch * DFL_JSTRIDE));
            DCK(dfl_malloc(st, 3, &st.d_pairs2[k], sizeof(DflPair) * batch));
            DCK(dfl_malloc(st, 3, &st.d_jobs2[k], sizeof(DflJob) * batch));
            st.fj_pairs[k] = batch;
        }
        if (FQ && !st.d_FJQ2[k]) DCK(dfl_malloc(st, 3, &st.d_FJQ2[k], sizeof(uint32_t) * st.fj_pairs[k] * DFL_JSTRIDE));
    }
    DCK(cudaFuncSetAttribute(dfl_parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(DFL_PARSE_THREADS * sizeof(DflCompactTrees))));
    if (!st.stream2) {
        // the parse kernel is a few long-running, latency-bound CTAs: give it priority over the junction kernel's
        // many short blocks, which would otherwise keep every SM full until they are all done
        int prio_lo = 0, prio_hi = 0;
        DCK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        DCK(cudaStreamCreateWithPriority(&st.stream2, cudaStreamNonBlocking, prio_hi));
        for (int k = 0; k < 2; ++k) {
            DCK(cudaEventCreateWithFlags(&st.ev_j[k], cudaEventDisableTiming));
            DCK(cudaEventCreateWithFlags(&st.ev_p[k], cudaEventDisableTiming));
        }
        DCK(dfl_malloc(st, 3, &st.d_counter2, 2 * sizeof(unsigned long long)));
    }
    const DflCorpus c = deflate_corpus(st, dc, li);
    const DflCanonPool cp{st.d_sym_end[li], st.d_sym_code[li], st.d_cum[li], st.d_soff, st.d_cap, st.d_roff, st.d_nsym[li],
                          st.d_seq_size[li]};
    cudaEvent_t e0 = st.ev_t[0], e1 = st.ev_t[1];
    std::vector<DflJob> jobs;
    std::vector<DflPair> pairs;
    NvtxRange nvtx_("snacc_b200: deflate pair batches (junction tables + pair parses)");
    // measured: the junction kernel and the parse kernel running side by side (st.stream2) take 10 % longer
    // than one after the other -- each fills the SMs on its own (registers / shared memory) -- so the second
    // stream is only used when asked for; the double buffers still let the host prepare batch b+1 early
    cudaStream_t pstream = getenv("SNACC_DFL_OVERLAP") ? st.stream2 : stream;
    DCK(cudaEventRecord(st.ev_j[0], stream));                  // everything queued so far (prep) precedes the parses
    DCK(cudaStreamWaitEvent(st.stream2, st.ev_j[0], 0));
    int64_t nbatch = 0;
    for (int64_t b0 = 0; b0 < total; b0 += (int64_t)batch, ++nbatch) {
        const int k2 = (int)(nbatch & 1);
        const int64_t nb = std::min<int64_t>((int64_t)batch, total - b0);
        pairs.resize((size_t)nb); jobs.resize((size_t)nb);
        for (int64_t k = 0; k < nb; ++k) {
            const int64_t j = subset ? (*subset)[b0 + k] : b0 + k;
            pairs[k] = DflPair{xs[j], ys[j]};
            jobs[k] = DflJob{xs[j], ys[j], kind, (int32_t)k, j};
        }
        if (nbatch >= 2) DCK(cudaStreamWaitEvent(stream, st.ev_p[k2], 0));   // buffer k2 is free again
        DCK(cudaMemcpyAsync(st.d_pairs2[k2], pairs.data(), sizeof(DflPair) * nb, cudaMemcpyHostToDevice, stream));
        DCK(cudaMemcpyAsync(st.d_jobs2[k2], jobs.data(), sizeof(DflJob) * nb, cudaMemcpyHostToDevice, stream));
        DCK(cudaEventRecord(e0, stream));
        {
            dim3 grid((DFL_JSTRIDE + 255) / 256, (unsigned)std::min<int64_t>(nb, 4096));
            dfl_junction_kernel<<<grid, 256, 0, stream>>>(c, st.d_pairs2[k2], (int32_t)nb, level, st.d_F[li], FQ, st.d_FJ2[k2],
                                                          FQ ? st.d_FJQ2[k2] : nullptr, st.junction_impl);
        }
        if (cudaGetLastError() != cudaSuccess) { err = "junction kernel launch failed"; return -1; }
        DCK(cudaEventRecord(e1, stream));
        DCK(cudaEventRecord(st.ev_j[k2], stream));
        DCK(cudaStreamWaitEvent(pstream, st.ev_j[k2], 0));
        DCK(cudaMemsetAsync(st.d_counter2 + k2, 0, sizeof(unsigned long long), pstream));
        const int blocks = (int)std::min<size_t>(((size_t)nb + DFL_PARSE_THREADS - 1) / DFL_PARSE_THREADS, parse_blocks);
        dfl_parse_kernel<<<blocks, DFL_PARSE_THREADS, DFL_PARSE_THREADS * sizeof(DflCompactTrees), pstream>>>(c, st.d_jobs2[k2], nb, level, st.d_F[li], FQ, st.d_FJ2[k2],
                                                                      FQ ? st.d_FJQ2[k2] : nullptr, st.d_ckpt[li], cp,
                                                                      st.d_scratch2[k2], st.d_counter2 + k2, d_out);
        if (cudaGetLastError() != cudaSuccess) { err = "dfl_parse_kernel launch failed"; return -1; }
        DCK(cudaEventRecord(st.ev_p[k2], pstream));
        *launches += 2;
        // the host buffers are reused for the next batch: wait until this batch's uploads are done (the
        // kernels of the previous batch keep the GPU busy meanwhile)
        DCK(cudaEventSynchronize(st.ev_j[k2]));
        float ms = 0.f;
        DCK(cudaEventElapsedTime(&ms, e0, e1));
        st.main_ms += ms;                                  // the junction kernel is the dominant one
    }
    DCK(cudaStreamSynchronize(st.stream2));
    DCK(cudaStreamSynchronize(stream));
    if (kind != 2) return 0;
    // jobs whose shortcut met a block that might be stored (-2): full serial parse
    std::vector<int64_t> h_out((size_t)n_jobs), redo;
    DCK(cudaMemcpyAsync(h_out.data(), d_out, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, stream));
    DCK(cudaStreamSynchronize(stream));
    for (int64_t k = 0; k < total; ++k) {
        const int64_t j = subset ? (*subset)[k] : k;
        if (h_out[j] == -2) redo.push_back(j);
    }
    st.serial_jobs += (int64_t)redo.size();
    return redo.empty() ? 0 : deflate_pairs(st, dc, level, xs, ys, n_jobs, &redo, 4, batch, d_out, stream, launches, err);
}

// sizes of the raw deflate streams of the jobs (x alone when ys == nullptr) into d_out[0..n_jobs)
static int deflate_run(DeflateState &st, const Corpus &dc, int level, const int32_t *xs, const int32_t *ys,
                       const int32_t *d_xs, int64_t n_jobs, int64_t *d_out, cudaStream_t stream, int64_t *launches,
                       std::string &err)
{
    const int li = level == 9 ? 0 : 1;
    const int32_t ns = dc.n_seqs;
    st.main_ms = 0.0; st.serial_jobs = 0; st.bands = 0; st.prepared_seqs = 0; st.parallel_prep_seqs = 0;
    st.peak = st.live[0] + st.live[1] + st.live[2] + st.live[3];

    // ---- roles.  x of a pair stream or a single: its record (own parse or imported) and, for pair streams, an
    //      index; y of a pair stream: the full preparation; a sequence without a record gets the full preparation
    //      once to produce it ----
    const bool x_ready = st.n_seqs == ns && st.d_xoff && st.d_ckpt[li];     // (records outlive a new x index layout)
    std::vector<uint8_t> used(ns, 0);
    for (int64_t k = 0; k < n_jobs; ++k) { used[xs[k]] |= 1; if (ys) used[ys[k]] |= 2; }
    std::vector<int32_t> full, ylist_all, no_rec, xpair;
    for (int32_t i = 0; i < ns; ++i) {
        if (!used[i]) continue;
        const bool rec = x_ready && st.have_ckpt[li][i];
        if (!rec) no_rec.push_back(i);
        if (used[i] & 2) ylist_all.push_back(i);
        if ((used[i] & 2) || !rec) full.push_back(i);
        if (ys && (used[i] & 1)) xpair.push_back(i);
    }

    // ---- memory plan (device bytes; free memory read now: the device is shared) ----
    size_t free0 = 0, total0 = 0;
    DCK(cudaMemGetInfo(&free0, &total0));
    const size_t batch = ys ? std::min<size_t>(DFL_BATCH, (size_t)n_jobs) : 0;
    uint64_t x_need = 0;                                              // x side still to allocate
    if (!(st.n_seqs == ns && st.d_xoff)) x_need += (uint64_t)ns * dfl_xbytes_fixed();
    if (!(st.n_seqs == ns && st.d_xoff && st.x_whole == (st.use_tail_index ? 0 : 1)))
        for (int32_t i = 0; i < ns; ++i) x_need += 4 * dfl_xslot(dc.h_len[i], st.use_tail_index ? 0 : 1);
    if (!(st.n_seqs == ns && st.d_ckpt[li])) x_need += (uint64_t)ns * dfl_xbytes_level();
    uint32_t max_len = 0; uint64_t y_all = 0, y_max = 0;
    for (int32_t i : full) { const uint64_t b = dfl_ybytes(dc.h_len[i], level); y_all += b; y_max = std::max(y_max, b); max_len = std::max(max_len, dc.h_len[i]); }
    uint64_t work = 0;
    if (ys) {
        const uint64_t nbuf = (uint64_t)n_jobs > batch ? 2 : 1;
        const uint64_t threads = std::min<uint64_t>(DFL_PARSE_BLOCKS, (batch + DFL_PARSE_THREADS - 1) / DFL_PARSE_THREADS) * DFL_PARSE_THREADS;
        work += nbuf * (batch * ((uint64_t)DFL_JSTRIDE * 4 * (level == 9 ? 1 : 2) + sizeof(DflPair) + sizeof(DflJob)) + threads * sizeof(DflTrees));
        uint64_t sum = 0, big = 0;                                      // x index sort scratch, as deflate_build_x sizes it
        for (int32_t i : xpair) { const uint64_t v = dfl_xslot(dc.h_len[i], st.use_tail_index ? 0 : 1); sum += v; big = std::max(big, v); }
        work += 4 * (std::max(big, std::min<uint64_t>(sum, (uint64_t)DFL_INDEX_GROUP * DFL_XTAIL)) + 16);
    }
    if (!full.empty()) {
        if (st.use_index6 && level == 9) work += 4 * (std::min<uint64_t>(DFL_ORDER6_CAP, y_all) + 16);
        work += 4ull * DFL_INDEX_GROUP * 256 * std::max(1u, dfl_rx_tiles(max_len));
    }
    const uint64_t margin = (256ull << 20) + total0 / 100;           // allocator granularity, kernel stacks, the caller's epilogue
    // pair-batch buffers of another shape than this call's are released now: what stays is what the call reuses.  A call
    // without pair jobs leaves them alone and counts them as held.
    if (ys) {
        const size_t threads = std::min<size_t>(DFL_PARSE_BLOCKS, (batch + DFL_PARSE_THREADS - 1) / DFL_PARSE_THREADS) * DFL_PARSE_THREADS;
        const bool same = st.fj_pairs[0] == batch && st.scratch_n[0] == threads && (st.d_FJ2[1] != nullptr) == ((size_t)n_jobs > batch) &&
                          (st.d_FJ2[1] == nullptr || (st.fj_pairs[1] == batch && st.scratch_n[1] == threads)) &&
                          (st.d_FJQ2[0] != nullptr) == (level != 9);
        if (!same) deflate_free_batches(st);
    }
    // y layout (dropped when the call needs another), preparation scratch (none between calls), batch buffers (above)
    const uint64_t reusable = (uint64_t)st.live[1] + st.live[2] + (ys ? st.live[3] : 0);
    const uint64_t avail = free0 + reusable;
    const uint64_t fixed = x_need + work + margin;
    uint64_t y_budget = avail > fixed ? avail - fixed : 0;
    if (st.band_bytes > 0) y_budget = std::min<uint64_t>(y_budget, (uint64_t)st.band_bytes);
    if (!full.empty() && y_max > y_budget) {
        char b_[512];
        snprintf(b_, sizeof b_, "deflate: the x side of %d sequences, the working buffers and one y need %.3f GB of device memory "
                 "(%llu bytes; y layout capped at %llu bytes), %llu bytes are free",
                 ns, (double)(fixed + y_max) / 1e9, (unsigned long long)(fixed + y_max),
                 (unsigned long long)(st.band_bytes > 0 ? (uint64_t)st.band_bytes : avail), (unsigned long long)avail);
        err = b_;
        return SNACC_ERR_TOO_LARGE;
    }
    if (deflate_ensure_x(st, dc, level, stream, err)) return -1;
    if (!st.ev_t[0]) { DCK(cudaEventCreate(&st.ev_t[0])); DCK(cudaEventCreate(&st.ev_t[1])); }   // owned by the state: no leak on error paths

    bool in_layout = !st.ylist.empty();
    for (int32_t i : full) in_layout = in_layout && st.h_yslot[i] != DFL_NONE;
    if (in_layout) {
        // the layout holds the sequences (it may hold more): keep it only if all of it, with this level's arrays when they
        // are missing, fits the budget -- a kept layout is not released
        uint64_t lb = 0;
        if (!st.d_F[li])
            for (int32_t i : st.ylist) {
                const uint64_t cap = dfl_canon_cap(dc.h_len[i]);
                lb += dfl_pad8(dc.h_len[i]) * 4 * (level == 9 || st.d_FQ ? 1 : 2) + 2ull * DFL_JY + cap * 6 + (cap / DFL_CUM_G + 1) * DFL_CUM_W * 4;
            }
        in_layout = st.live[1] + lb <= y_budget;
    }
    bool banded = false;
    if (in_layout || y_all <= y_budget || full.empty()) {
        // ---- one band: the whole y state of the call in one layout, which stays resident for later calls ----
        st.bands = 1;
        if (!full.empty()) {
            if (!in_layout) { if (deflate_set_layout(st, dc, level, full, stream, err)) return -1; }
            else if (deflate_ensure_y_level(st, level, err)) return -1;
            if (deflate_prepare_y(st, dc, level, full, stream, launches, err)) return -1;
        }
        if (ys) {
            std::vector<int32_t> need_x;
            for (int32_t i : xpair) if (!st.yindexed[i] && !st.xindexed[i]) need_x.push_back(i);
            if (deflate_build_x(st, dc, li, need_x, stream, launches, err)) return -1;
            if (deflate_upload_ix(st, stream, err)) return -1;
            if (deflate_pairs(st, dc, level, xs, ys, n_jobs, nullptr, st.use_canon ? 2 : 4, batch, d_out, stream, launches, err)) return -1;
        }
    } else {
        // ---- bands: the y layout of each band holds what fits in y_budget; afterwards only the x side stays ----
        banded = true;
        deflate_drop_y(st);
        deflate_free_batches(st);
        auto cut = [&](const std::vector<int32_t> &list) {
            std::vector<std::vector<int32_t>> out;
            uint64_t acc = 0;
            for (int32_t i : list) {
                const uint64_t b = dfl_ybytes(dc.h_len[i], level);
                if (out.empty() || acc + b > y_budget) { out.emplace_back(); acc = 0; }
                out.back().push_back(i); acc += b;
            }
            return out;
        };
        // pass 0: the records of the sequences that have none
        for (const auto &part : cut(no_rec)) {
            ++st.bands;
            if (deflate_set_layout(st, dc, level, part, stream, err)) return -1;
            if (deflate_prepare_y(st, dc, level, part, stream, launches, err)) return -1;
        }
        deflate_drop_y(st);
        if (ys) {
            // pass 1: x index slices of every x, then the pair jobs band by band of their y, in the caller's job order
            std::vector<int32_t> need_x;
            for (int32_t i : xpair) if (!st.xindexed[i]) need_x.push_back(i);
            if (deflate_build_x(st, dc, li, need_x, stream, launches, err)) return -1;
            std::vector<int32_t> band_of(ns, -1);
            const auto bands = cut(ylist_all);
            for (size_t b = 0; b < bands.size(); ++b) for (int32_t i : bands[b]) band_of[i] = (int32_t)b;
            std::vector<std::vector<int64_t>> jobs_of(bands.size());
            for (int64_t k = 0; k < n_jobs; ++k) jobs_of[band_of[ys[k]]].push_back(k);
            for (size_t b = 0; b < bands.size(); ++b) {
                ++st.bands;
                if (deflate_set_layout(st, dc, level, bands[b], stream, err)) return -1;
                if (deflate_prepare_y(st, dc, level, bands[b], stream, launches, err)) return -1;
                if (deflate_upload_ix(st, stream, err)) return -1;
                if (deflate_pairs(st, dc, level, xs, ys, n_jobs, &jobs_of[b], st.use_canon ? 2 : 4, batch, d_out, stream, launches, err))
                    return -1;
            }
        }
    }
    if (!ys) {
        dfl_gather_sizes_kernel<<<(unsigned)((n_jobs + 255) / 256), 256, 0, stream>>>(st.d_seq_size[li], d_xs, n_jobs, d_out);
        if (cudaGetLastError() != cudaSuccess) { err = "dfl_gather_sizes_kernel launch failed"; return -1; }
        ++*launches;
    }
    DCK(cudaStreamSynchronize(stream));
    dfl_free(st, st.d_order6); st.order6_cap = 0;                  // preparation scratch: none between calls
    dfl_free(st, st.d_rx_hist); st.rx_cap = 0;
    dfl_free(st, st.d_xtmp); st.xtmp_cap = 0;
    if (banded) {
        // what stays is the x side: the caller's epilogue (snacc_ncd, a gather across ranks) needs the room
        deflate_drop_y(st);
        deflate_free_batches(st);
        if (deflate_upload_ix(st, stream, err)) return -1;
    }
    return 0;
}
#endif  // __CUDACC__

}  // namespace snacc
