// libbz2_order.cu -- where libbz2 1.0.8's block sort leaves rotation 0 of a periodic block (host code).
//
// With BZ2B200_LIBBZ2 the stored origin pointer must be the row libbz2 stores: the index at which its sorted pointer
// array holds rotation 0.  A block that is not periodic has one such row, the rank of rotation 0, and the GPU sort
// gives it.  A periodic block (u^k) has k equal rotations, and libbz2 stores whichever of their rows its sort happened to
// put rotation 0 in.  For such blocks that sort is fallbackSort: below 10000 bytes libbz2 calls it directly, and from
// 10000 bytes on mainSort compares equal rotations over their whole length (n / 8 units of its 9 n work budget per
// comparison), runs out of budget and libbz2 starts over with fallbackSort.  (Not always: a block with a few long
// periods can cost mainSort few enough comparisons to finish, and then mainSort's order decides -- not reproduced, see
// DESIGN.md §10.)  fallbackSort is deterministic -- a Manber-Myers doubling whose buckets are split
// by a 3-way quicksort with a fixed linear-congruential pivot choice and an insertion sort below 10 entries -- and it is
// restated here step for step: the order of equal rotations is an artefact of exactly these steps.
//
// The walk is serial (a data-dependent quicksort), so it runs on the host, only for blocks whose class of rotation 0 has
// more than one member (k_bwt_out counts them on the device) and only in this mode.  The interior blocks of a long run of
// one byte value are all the same block, so the last answer is kept with its block (DESIGN.md §10).
#include <stdint.h>
#include <string.h>
#include <vector>

namespace {

typedef int32_t Int32;
typedef uint32_t UInt32;

constexpr Int32 SMALL_THRESH = 10;
constexpr Int32 STACK_SIZE = 100;

inline void simple_sort(UInt32 *fmap, const UInt32 *eclass, Int32 lo, Int32 hi) {
    if (lo == hi) return;
    if (hi - lo > 3) {
        for (Int32 i = hi - 4; i >= lo; i--) {
            UInt32 tmp = fmap[i], ec = eclass[tmp];
            Int32 j;
            for (j = i + 4; j <= hi && ec > eclass[fmap[j]]; j += 4) fmap[j - 4] = fmap[j];
            fmap[j - 4] = tmp;
        }
    }
    for (Int32 i = hi - 1; i >= lo; i--) {
        UInt32 tmp = fmap[i], ec = eclass[tmp];
        Int32 j;
        for (j = i + 1; j <= hi && ec > eclass[fmap[j]]; j++) fmap[j - 1] = fmap[j];
        fmap[j - 1] = tmp;
    }
}

inline void vswap(UInt32 *fmap, Int32 p1, Int32 p2, Int32 n) {
    while (n > 0) { UInt32 t = fmap[p1]; fmap[p1] = fmap[p2]; fmap[p2] = t; p1++; p2++; n--; }
}

// returns false if the explicit stack would overflow (libbz2 asserts there; it cannot happen for n <= 900000)
bool qsort3(UInt32 *fmap, const UInt32 *eclass, Int32 loSt, Int32 hiSt) {
    Int32 stackLo[STACK_SIZE], stackHi[STACK_SIZE];
    UInt32 r = 0;
    Int32 sp = 0;
    stackLo[sp] = loSt; stackHi[sp] = hiSt; sp++;
    while (sp > 0) {
        if (sp >= STACK_SIZE - 1) return false;
        sp--;
        Int32 lo = stackLo[sp], hi = stackHi[sp];
        if (hi - lo < SMALL_THRESH) { simple_sort(fmap, eclass, lo, hi); continue; }
        r = ((r * 7621) + 1) % 32768;                       // the pivot: first, middle or last by r % 3
        UInt32 r3 = r % 3, med;
        if (r3 == 0) med = eclass[fmap[lo]];
        else if (r3 == 1) med = eclass[fmap[(lo + hi) >> 1]];
        else med = eclass[fmap[hi]];
        Int32 unLo = lo, ltLo = lo, unHi = hi, gtHi = hi, n, m;
        for (;;) {
            for (;;) {
                if (unLo > unHi) break;
                n = (Int32)eclass[fmap[unLo]] - (Int32)med;
                if (n == 0) { UInt32 t = fmap[unLo]; fmap[unLo] = fmap[ltLo]; fmap[ltLo] = t; ltLo++; unLo++; continue; }
                if (n > 0) break;
                unLo++;
            }
            for (;;) {
                if (unLo > unHi) break;
                n = (Int32)eclass[fmap[unHi]] - (Int32)med;
                if (n == 0) { UInt32 t = fmap[unHi]; fmap[unHi] = fmap[gtHi]; fmap[gtHi] = t; gtHi--; unHi--; continue; }
                if (n < 0) break;
                unHi--;
            }
            if (unLo > unHi) break;
            UInt32 t = fmap[unLo]; fmap[unLo] = fmap[unHi]; fmap[unHi] = t; unLo++; unHi--;
        }
        if (gtHi < ltLo) continue;
        n = (ltLo - lo < unLo - ltLo) ? ltLo - lo : unLo - ltLo;
        vswap(fmap, lo, unLo - n, n);
        m = (hi - gtHi < gtHi - unHi) ? hi - gtHi : gtHi - unHi;
        vswap(fmap, unLo, hi - m + 1, m);
        n = lo + unLo - ltLo - 1;
        m = hi - (gtHi - unHi) + 1;
        if (n - lo > hi - m) {                               // the larger part is pushed first, popped last
            stackLo[sp] = lo; stackHi[sp] = n; sp++;
            stackLo[sp] = m; stackHi[sp] = hi; sp++;
        } else {
            stackLo[sp] = m; stackHi[sp] = hi; sp++;
            stackLo[sp] = lo; stackHi[sp] = n; sp++;
        }
    }
    return true;
}

#define SET_BH(zz) bh[(zz) >> 5] |= ((UInt32)1 << ((zz) & 31))
#define CLEAR_BH(zz) bh[(zz) >> 5] &= ~((UInt32)1 << ((zz) & 31))
#define ISSET_BH(zz) (bh[(zz) >> 5] & ((UInt32)1 << ((zz) & 31)))
#define WORD_BH(zz) bh[(zz) >> 5]
#define UNALIGNED_BH(zz) ((zz) & 0x01f)

}  // namespace

// Row of rotation 0 after libbz2's fallbackSort of block[0, n); -1 if its stack would overflow.
long long bz_libbz2_fallback_origin(const uint8_t *block, uint32_t n) {
    if (n == 0) return 0;
    const Int32 nblock = (Int32)n;
    std::vector<UInt32> fmap(n), eclass(n), bhtab(2 + n / 32 + 4, 0);
    UInt32 *bh = bhtab.data();
    Int32 ftab[257];
    for (Int32 i = 0; i < 257; i++) ftab[i] = 0;
    for (Int32 i = 0; i < nblock; i++) ftab[block[i]]++;
    for (Int32 i = 1; i < 257; i++) ftab[i] += ftab[i - 1];
    for (Int32 i = 0; i < nblock; i++) {                     // 1-byte radix sort, each bucket filled from its end
        Int32 j = block[i], k = ftab[j] - 1;
        ftab[j] = k;
        fmap[k] = (UInt32)i;
    }
    for (Int32 i = 0; i < 256; i++) SET_BH(ftab[i]);
    for (Int32 i = 0; i < 32; i++) { SET_BH(nblock + 2 * i); CLEAR_BH(nblock + 2 * i + 1); }   // block-end sentinels
    Int32 H = 1;
    for (;;) {
        Int32 j = 0;
        for (Int32 i = 0; i < nblock; i++) {
            if (ISSET_BH(i)) j = i;
            Int32 k = (Int32)fmap[i] - H;
            if (k < 0) k += nblock;
            eclass[k] = (UInt32)j;
        }
        Int32 nNotDone = 0, r = -1;
        for (;;) {
            Int32 k = r + 1;                                 // the next bucket of more than one entry: [l, r]
            while (ISSET_BH(k) && UNALIGNED_BH(k)) k++;
            if (ISSET_BH(k)) {
                while (WORD_BH(k) == 0xffffffffu) k += 32;
                while (ISSET_BH(k)) k++;
            }
            Int32 l = k - 1;
            if (l >= nblock) break;
            while (!ISSET_BH(k) && UNALIGNED_BH(k)) k++;
            if (!ISSET_BH(k)) {
                while (WORD_BH(k) == 0x00000000u) k += 32;
                while (!ISSET_BH(k)) k++;
            }
            r = k - 1;
            if (r >= nblock) break;
            if (r > l) {
                nNotDone += (r - l + 1);
                if (!qsort3(fmap.data(), eclass.data(), l, r)) return -1;
                Int32 cc = -1;
                for (Int32 i = l; i <= r; i++) {
                    Int32 cc1 = (Int32)eclass[fmap[i]];
                    if (cc != cc1) { SET_BH(i); cc = cc1; }
                }
            }
        }
        H *= 2;
        if (H > nblock || nNotDone == 0) break;
    }
    for (Int32 i = 0; i < nblock; i++)
        if (fmap[i] == 0) return i;
    return -1;
}

#undef SET_BH
#undef CLEAR_BH
#undef ISSET_BH
#undef WORD_BH
#undef UNALIGNED_BH
