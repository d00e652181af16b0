"""Shared-memory bank count of the NTT tile rounds (multi_stark_b200/csrc/ntt.cu), on the CPU.

Restates the kernels' thread -> (item, slot) -> tile-row map and the XOR-swizzled tile layout (kXt = 4 u64 per row, no
padding), and counts, for every warp-wide 64-bit shared-memory load or store of every round of every tile size, the
wavefronts it needs: the largest number of distinct 32-bit words that fall into one of the 32 banks. A warp moving 256 bytes
needs at least 2. Exits non-zero if any access needs more than the minimum.

    python tools/smem_banks.py [-v]
"""
import sys

KXT = 4


def sw2(row):
    return ((row >> 2) ^ (row >> 4) ^ (row >> 6) ^ (row >> 8)) & 3


def tile_at(row, q):
    return (row ^ sw2(row)) * KXT + q


def round_bits(tb, k):
    r1 = min(tb, 4)
    rem = tb - r1
    r2 = min(rem, 4)
    return [r1, r2, rem - r2][k]


def rounds(tb, dit):
    """(RB, S0) of each round in execution order, as tile_pass runs them."""
    b = [round_bits(tb, k) for k in range(3)]
    dif = [(b[0], tb - b[0])]
    if b[1]:
        dif.append((b[1], b[2]))
    if b[2]:
        dif.append((b[2], 0))
    if dit and tb == 7:  # 4, 3 from the low bits up
        return [(4, 0), (3, 4)]
    return dif[::-1] if dit else dif


def tile_threads(tb):
    rows = 1 << (tb - 4) if tb >= 4 else 1
    return min(max(rows * KXT, 32), 64 * KXT)


def wavefronts(elems):
    banks = {}
    for e in elems:
        for word in (2 * e, 2 * e + 1):
            banks.setdefault(word % 32, set()).add(word)
    return max(len(s) for s in banks.values())


def round_accesses(tb, rb, s0):
    """Per (warp, g-loop iteration, slot m): the element indices the active lanes touch."""
    items = 1 << (tb - rb)
    blk_bits = tb - rb - s0
    nthr = tile_threads(tb)
    nrows = nthr // KXT
    for warp in range(0, nthr, 32):
        it = 0
        while True:
            lanes = []
            for t in range(warp, min(warp + 32, nthr)):
                g = (t // KXT) + it * nrows
                if g >= items:
                    continue
                off, blk = (g >> blk_bits, g & ((1 << blk_bits) - 1)) if s0 else (0, g)
                lanes.append(((blk << (s0 + rb)) + off, t % KXT))
            if not lanes:
                break
            for m in range(1 << rb):
                yield [tile_at(row0 | (m << s0), q) for row0, q in lanes]
            it += 1


def main():
    verbose = "-v" in sys.argv
    bad = 0
    print("tb  dir  round(RB@S0)  shared ld/st  accesses  worst wavefronts (min 2 for a full warp)")
    for tb in range(5, 11):  # tiles of <= 4 bits are one register round: no shared memory
        for dit in (False, True):
            rs = rounds(tb, dit)
            for i, (rb, s0) in enumerate(rs):
                ops = ("ld" if i > 0 else "") + ("st" if i + 1 < len(rs) else "")
                if not ops:
                    continue
                worst, n = 0, 0
                for elems in round_accesses(tb, rb, s0):
                    need = (len(elems) * 8 + 127) // 128
                    worst = max(worst, wavefronts(elems) / need)
                    n += 1
                flag = "" if worst == 1 else "  CONFLICT"
                bad += worst != 1
                if verbose or flag:
                    print("%2d  %s  %2d@%d  %-4s  %5d  x%.2f%s" % (tb, "DIT" if dit else "DIF", rb, s0, ops, n, worst, flag))
    print("bank conflicts: %s" % ("none" if not bad else "%d rounds" % bad))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
