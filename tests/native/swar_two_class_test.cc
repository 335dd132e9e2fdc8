// Host build of the two-class SWAR words (skywalking-banyandb_b200/csrc/lane_decode.cuh: swar_word / swar_masked_word with
// kTwoClass) and of the chunk walk around them in scan_kernels.cu (swar_chunk, delta_page_sum_masked): 2 KB chunks of 32 lanes x
// 64 bytes, a 16-byte aligned window around the page, masked first / last chunk, the previous lane's last word handed on, the
// last word of the previous chunk carried over, the two-class pass, the warp vote on the lanes' guards and the carried word, and
// the three-class pass again over a chunk that needs it.
//
// Pages hold 1- and 2-byte varints with 3- and 4-byte ones placed on purpose: at the page's first and last byte, across lane
// and chunk boundaries (two bytes at the end of one chunk, the rest in the next) and inside the masked head and tail chunks.
// Checked per page:
//   * sum and terminator count equal the plain definition (pages without a 4-byte varint), and `wide` is raised exactly when
//     the page holds a varint of 4 or more bytes;
//   * whichever pass produced them, every lane's n, T and R' equal those of the three-class word;
//   * a chunk is decoded again exactly when a class-2 byte (the third or later byte of a varint) lies in it or at the first
//     byte of the next chunk -- so a page of 1- and 2-byte varints never is.
// Built and run by tests/test_swar_two_class_native.py with g++.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "lane_decode.cuh"

using namespace bydb;

static int32_t zz(uint32_t u) { return static_cast<int32_t>(u >> 1) ^ -static_cast<int32_t>(u & 1u); }

struct Page {
    std::vector<uint8_t> win;  // the 16-byte aligned window: junk, the page body, junk
    std::vector<int64_t> d;    // the deltas
    uint32_t pstart = 0, pend = 0, total = 0;
    bool has_wide = false;     // a varint of 4 or more bytes
};

static void put_varint(Page &pg, std::mt19937_64 &rng, int L) {
    uint32_t u = static_cast<uint32_t>(rng()) & ((1u << (7 * L)) - 1u);
    if (L > 1 && (u >> (7 * (L - 1))) == 0) u |= 1u << (7 * (L - 1));  // canonical length
    if (L > 2 && rng() % 5 == 0) u &= ~0x3f80u;                        // a 0x80 continuation byte in the middle
    if (L > 1 && (u >> (7 * (L - 1))) == 0) u |= 1u << (7 * (L - 1));
    pg.d.push_back(zz(u));
    for (int k = 0; k < L; ++k) pg.win.push_back(static_cast<uint8_t>(((u >> (7 * k)) & 0x7f) | (k < L - 1 ? 0x80 : 0)));
    if (L >= 4) pg.has_wide = true;
}

// A page of ~n_bytes of 1- and 2-byte varints; when `place`, long varints (3 bytes, or 4 when `wide`) start at chosen window
// offsets: the page's first byte, lane and chunk edges, inside the head and tail chunk, and the page ends on one.
static Page make_page(std::mt19937_64 &rng, uint32_t n_bytes, bool place, bool wide) {
    Page pg;
    pg.pstart = static_cast<uint32_t>(rng() % 16);
    pg.win.resize(pg.pstart);
    for (auto &x : pg.win) x = static_cast<uint8_t>(rng());  // bytes of a neighbouring page in front of this one
    const uint32_t end = pg.pstart + n_bytes;
    std::vector<uint32_t> at;
    if (place) {
        if (rng() % 2) at.push_back(pg.pstart);
        for (int i = 0; i < 6; ++i) {
            const uint32_t k = static_cast<uint32_t>(rng() % (end / 64 + 1));
            const uint32_t edge = (rng() % 2 ? 2048u * (k / 32 + 1) : 64u * (k + 1));
            at.push_back(edge - 1 - static_cast<uint32_t>(rng() % 3));  // 1, 2 or 3 bytes before a lane / chunk edge
        }
        at.push_back(pg.pstart + static_cast<uint32_t>(rng() % 300));          // head chunk
        if (end > 400) at.push_back(end - 1 - static_cast<uint32_t>(rng() % 300));  // tail chunk
        std::sort(at.begin(), at.end());
    }
    size_t ai = 0;
    while (pg.win.size() < end) {
        while (ai < at.size() && at[ai] < pg.win.size()) ++ai;
        int L = 1 + static_cast<int>(rng() % 2);
        if (ai < at.size()) {
            const uint32_t gap = at[ai] - static_cast<uint32_t>(pg.win.size());
            if (gap == 0) {
                L = wide && rng() % 3 == 0 ? 4 : 3;
                ++ai;
            } else if (gap == 1) {
                L = 1;
            }
        }
        put_varint(pg, rng, L);
    }
    if (place) put_varint(pg, rng, 3);  // the page ends on a long varint
    pg.pend = static_cast<uint32_t>(pg.win.size());
    while (pg.win.size() % 16) pg.win.push_back(static_cast<uint8_t>(rng()));
    pg.total = static_cast<uint32_t>(pg.win.size());
    pg.win.resize(pg.win.size() + 2048, 0xAB);  // never read by the kernel; junk keeps the emulation honest
    return pg;
}

// chunks (of the window) that must be decoded again: a class-2 byte in the chunk or at the next chunk's first byte
static std::vector<bool> want_redo(const Page &pg, uint32_t nchunks) {
    std::vector<bool> r(nchunks, false);
    for (uint32_t i = pg.pstart + 2; i < pg.pend; ++i) {
        if ((pg.win[i - 1] & 0x80) && (pg.win[i - 2] & 0x80)) {
            r[i / 2048] = true;
            if (i % 2048 == 0) r[i / 2048 - 1] = true;
        }
    }
    return r;
}

struct LaneWords {
    uint32_t w[32][16];
    uint64_t valid[32];
    uint32_t lastw[32];  // the lane's last word as the kernel hands it on (bytes outside the page zeroed)
};

static void load_chunk(const Page &pg, uint32_t c, bool interior, LaneWords &lw) {
    for (int lane = 0; lane < 32; ++lane) {
        const uint32_t o = c * 2048 + lane * 64;
        for (int k = 0; k < 16; ++k) {
            lw.w[lane][k] = 0;
            if (o + 4 * k < pg.total) memcpy(&lw.w[lane][k], &pg.win[o + 4 * k], 4);
        }
        int lo_i = static_cast<int>(pg.pstart) - static_cast<int>(o), hi_i = static_cast<int>(pg.pend) - static_cast<int>(o);
        lo_i = lo_i < 0 ? 0 : (lo_i > 64 ? 64 : lo_i);
        hi_i = hi_i < 0 ? 0 : (hi_i > 64 ? 64 : hi_i);
        lw.valid[lane] = interior ? ~0ull : (hi_i >= 64 ? ~0ull : ((1ull << hi_i) - 1ull)) & ~(lo_i >= 64 ? ~0ull : ((1ull << lo_i) - 1ull));
        lw.lastw[lane] = lw.w[lane][15] & expand4(static_cast<uint32_t>(lw.valid[lane] >> 60));
    }
}

template <bool kTwoClass>
static void swar_pass(const LaneWords &lw, int lane, bool interior, uint32_t pw, SwarLane &sl) {
    swar_begin(sl, pw);
    for (int k = 0; k < 16; ++k) {
        if (interior) swar_word<false, kTwoClass>(sl, lw.w[lane][k], 0u);
        else swar_word<true, kTwoClass>(sl, lw.w[lane][k], expand4(static_cast<uint32_t>(lw.valid[lane] >> (4 * k))));
    }
}

static bool all_rows_check(const Page &pg, const char *what) {
    const int64_t n = static_cast<int64_t>(pg.d.size()) + 1;
    int64_t want = 0, pre = 0;
    for (int64_t x : pg.d) {
        pre += x;
        want += pre;
    }
    const uint32_t nchunks = (pg.total + 2047) / 2048;
    const std::vector<bool> redo_want = want_redo(pg, nchunks);
    int64_t S = 0;
    uint32_t tb = 0, carry_w = 0;
    bool wide = false;
    static LaneWords lw;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const bool interior = c * 2048 >= pg.pstart && (c + 1) * 2048 <= pg.pend;
        load_chunk(pg, c, interior, lw);
        SwarLane two[32], three[32];
        bool vote = swar_opens_class2(carry_w);
        for (int lane = 0; lane < 32; ++lane) {
            const uint32_t pw = lane == 0 ? carry_w : lw.lastw[lane - 1];
            swar_pass<true>(lw, lane, interior, pw, two[lane]);
            swar_pass<false>(lw, lane, interior, pw, three[lane]);
            vote = vote || (two[lane].guard & 0x80808080u) != 0;
            if (two[lane].prev_w != lw.lastw[lane]) {
                std::printf("FAIL %s: lane %d of chunk %u ends on %08x, hands on %08x\n", what, lane, c, two[lane].prev_w, lw.lastw[lane]);
                return false;
            }
        }
        if (vote != redo_want[c]) {
            std::printf("FAIL %s: chunk %u of %u redone=%d, class-2 byte in it or at the next one's start=%d (pstart %u pend %u)\n", what, c,
                        nchunks, vote, static_cast<int>(redo_want[c]), pg.pstart, pg.pend);
            return false;
        }
        carry_w = lw.lastw[31];
        uint32_t lb = 0;
        for (int lane = 0; lane < 32; ++lane) {
            const SwarLane &sl = vote ? three[lane] : two[lane];
            int32_t T, Rp, T3, Rp3;
            const uint32_t nl = swar_end(sl, T, Rp), n3 = swar_end(three[lane], T3, Rp3);
            if (nl != n3 || T != T3 || Rp != Rp3) {
                std::printf("FAIL %s: chunk %u lane %d gives (%u, %d, %d), three-class word (%u, %d, %d)\n", what, c, lane, nl, T, Rp, n3, T3, Rp3);
                return false;
            }
            if (vote) wide = wide || (sl.wide & 0x80808080u) != 0;
            const int64_t A = (n - 1) - static_cast<int64_t>(tb) - static_cast<int64_t>(lb);
            S += (A + 1) * static_cast<int64_t>(T) - static_cast<int64_t>(Rp);
            lb += nl;
        }
        tb += lb;
    }
    if (wide != pg.has_wide) {
        std::printf("FAIL %s: page with a 4-byte varint=%d, wide=%d\n", what, pg.has_wide, wide);
        return false;
    }
    if (!pg.has_wide && (tb != pg.d.size() || S != want)) {
        std::printf("FAIL %s: values=%zu pstart=%u terminators=%u S=%lld want=%lld\n", what, pg.d.size(), pg.pstart, tb, static_cast<long long>(S),
                    static_cast<long long>(want));
        return false;
    }
    return true;
}

template <bool kTwoClass>
static void masked_pass(const LaneWords &lw, int lane, bool interior, uint32_t pw, uint64_t aw, SwarMasked &sl) {
    swar_masked_begin(sl, pw, static_cast<uint32_t>(aw), static_cast<uint32_t>(aw >> 32));
    for (int k = 0; k < 16; ++k) {
        if (interior) swar_masked_word<false, kTwoClass>(sl, lw.w[lane][k], 0u);
        else swar_masked_word<true, kTwoClass>(sl, lw.w[lane][k], expand4(static_cast<uint32_t>(lw.valid[lane] >> (4 * k))));
    }
}

static bool masked_check(const Page &pg, std::mt19937_64 &rng, int density_pct, const char *what) {
    const int n_values = static_cast<int>(pg.d.size());
    const int64_t first = static_cast<int64_t>(rng() % 2000001) - 1000000;
    std::vector<uint8_t> act(n_values + 1 + 128, 0);
    for (size_t r = 0; r < static_cast<size_t>(n_values) + 1;) {
        const size_t run = 1 + rng() % 40;
        const bool on = static_cast<int>(rng() % 100) < density_pct;
        for (size_t k = 0; k < run && r < static_cast<size_t>(n_values) + 1; ++k) act[r++] = on;
    }
    int64_t want = 0, A_total = 0, v = first;
    for (int r = 0; r <= n_values; ++r) {
        if (r > 0) v += pg.d[r - 1];
        if (act[r]) {
            want += v;
            A_total++;
        }
    }
    const uint32_t nchunks = (pg.total + 2047) / 2048;
    const std::vector<bool> redo_want = want_redo(pg, nchunks);
    int64_t S = 0;
    uint32_t row_base = 1, atb = 0, carry_w = 0;
    bool wide = false;
    static LaneWords lw;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const bool interior = c * 2048 >= pg.pstart && (c + 1) * 2048 <= pg.pend;
        load_chunk(pg, c, interior, lw);
        // pass 1: the lanes' terminators -> their first rows and activity bits
        uint32_t nall[32], lb = 0;
        uint64_t aw[32];
        for (int lane = 0; lane < 32; ++lane) {
            nall[lane] = 0;
            for (int k = 0; k < 16; ++k) nall[lane] += count_terminators(lw.w[lane][k], interior ? 0xffffffffu : expand4(static_cast<uint32_t>(lw.valid[lane] >> (4 * k))));
            const uint32_t row0 = row_base + lb;
            aw[lane] = 0;
            for (uint32_t i = 0; i < nall[lane] && i < 64 && row0 + i < act.size(); ++i) aw[lane] |= static_cast<uint64_t>(act[row0 + i]) << i;
            lb += nall[lane];
        }
        // pass 2
        SwarMasked two[32], three[32];
        bool vote = swar_opens_class2(carry_w);
        for (int lane = 0; lane < 32; ++lane) {
            const uint32_t pw = lane == 0 ? carry_w : lw.lastw[lane - 1];
            masked_pass<true>(lw, lane, interior, pw, aw[lane], two[lane]);
            masked_pass<false>(lw, lane, interior, pw, aw[lane], three[lane]);
            vote = vote || (two[lane].guard & 0x80808080u) != 0;
        }
        if (vote != redo_want[c]) {
            std::printf("FAIL %s: chunk %u of %u redone=%d, class-2 byte in it or at the next one's start=%d\n", what, c, nchunks, vote,
                        static_cast<int>(redo_want[c]));
            return false;
        }
        carry_w = lw.lastw[31];
        uint32_t alb = 0;
        for (int lane = 0; lane < 32; ++lane) {
            const SwarMasked &sl = vote ? three[lane] : two[lane];
            int32_t T, Rp, T3, Rp3;
            const uint32_t na = swar_masked_end(sl, T, Rp), n3 = swar_masked_end(three[lane], T3, Rp3);
            if (na != n3 || T != T3 || Rp != Rp3) {
                std::printf("FAIL %s: chunk %u lane %d gives (%u, %d, %d), three-class word (%u, %d, %d)\n", what, c, lane, na, T, Rp, n3, T3, Rp3);
                return false;
            }
            if (vote) wide = wide || (sl.wide & 0x80808080u) != 0;
            const int64_t A1a = (A_total - act[0]) - static_cast<int64_t>(atb) - static_cast<int64_t>(alb) + 1;
            S += A1a * static_cast<int64_t>(T) - static_cast<int64_t>(Rp);
            alb += na;
        }
        atb += alb;
        row_base += lb;
    }
    if (wide != pg.has_wide) {
        std::printf("FAIL %s: page with a 4-byte varint=%d, wide=%d\n", what, pg.has_wide, wide);
        return false;
    }
    const int64_t got = A_total * first + S;
    if (!pg.has_wide && (row_base != static_cast<uint32_t>(n_values) + 1 || got != want || static_cast<int64_t>(atb) + act[0] != A_total)) {
        std::printf("FAIL %s: values=%d pstart=%u density=%d rows=%u got=%lld want=%lld\n", what, n_values, pg.pstart, density_pct, row_base,
                    static_cast<long long>(got), static_cast<long long>(want));
        return false;
    }
    return true;
}

int main() {
    std::mt19937_64 rng(20261017);
    long pages = 0, redone_pages = 0;
    for (int it = 0; it < 1500; ++it) {
        const uint32_t n_bytes = it < 40 ? static_cast<uint32_t>(it) : 1 + static_cast<uint32_t>(rng() % 12000);
        const int kind = it % 3;  // 0: 1- and 2-byte varints only, 1: with 3-byte ones, 2: with 3- and 4-byte ones
        const Page pg = make_page(rng, n_bytes, kind > 0, kind == 2);
        const uint32_t nchunks = (pg.total + 2047) / 2048;
        const std::vector<bool> rw = want_redo(pg, nchunks);
        bool any = false;
        for (bool b : rw) any = any || b;
        if (kind == 0 && any) {
            std::printf("FAIL generator: a page of 1- and 2-byte varints holds a class-2 byte\n");
            return 1;
        }
        redone_pages += any;
        if (!all_rows_check(pg, "all rows")) return 1;
        static const int kDensity[] = {0, 1, 12, 50, 90, 100};
        if (!masked_check(pg, rng, kDensity[it % 6], "masked")) return 1;
        ++pages;
    }
    if (redone_pages < pages / 3) {
        std::printf("FAIL generator: only %ld of %ld pages hold a class-2 byte\n", redone_pages, pages);
        return 1;
    }
    std::printf("OK %ld pages, %ld with chunks decoded again\n", pages, redone_pages);
    return 0;
}
