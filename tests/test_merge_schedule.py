"""CPU model of the MMA schedule of the resident-weight 64 -> 64 strip kernel (femasr_b200/csrc/tc_gemm.cu, the merged tap-row schedule):
the merged form (one MMA of N = 64 x rows per input strip, kw, k-step and product) must hand every accumulator exactly the
contributions of the unmerged form, in the same order, and read them from the right weight plane of the merged layout.
Mirrors the index arithmetic of the kernel; the GPU proof is scripts/ab_digest.py (bit-identical outputs)."""
MR, KW, KSTEPS = 4, 3, 4


def unmerged(products):
    """[(accumulator row r, (kh, kw, k, product))] in issue order: per strip, per output row, per kw, per k, per product."""
    seq = []
    for sr in range(MR + 2):
        r_lo, r_hi = max(sr - 2, 0), min(sr, MR - 1)
        for r in range(r_lo, r_hi + 1):
            kh = sr - r
            for kw in range(KW):
                for k in range(KSTEPS):
                    for prod in products:
                        seq.append((r, (kh, kw, k, prod), "overwrite" if (kh, kw, k) == (0, 0, 0) and prod == products[0] else "acc"))
    return seq


def merged(products):
    """The kernel's loop: per strip, per kw, per k, per product ONE MMA over rows r_lo..r_hi (the fresh row's very first
    product split off).  Weight planes per kw group: plane p holds kh = 2 - p; a merged MMA starts at b_first."""
    seq = []
    for sr in range(MR + 2):
        r_lo, r_hi = max(sr - 2, 0), min(sr, MR - 1)
        fresh = sr < MR
        rows = r_hi - r_lo + 1
        b_first = 2 - (sr - r_lo)
        for kw in range(KW):
            for k in range(KSTEPS):
                for pi, prod in enumerate(products):
                    if fresh and kw == 0 and k == 0 and pi == 0:
                        groups = ([(r_lo, rows - 1, b_first, "acc")] if rows > 1 else []) + [(r_hi, 1, 2, "overwrite")]
                    else:
                        groups = [(r_lo, rows, b_first, "acc")]
                    for r0, n, plane0, mode in groups:
                        for j in range(n):                      # D columns [64 j, 64 j + 64) <-> B rows of plane plane0 + j
                            kh = 2 - (plane0 + j)
                            seq.append((r0 + j, (kh, kw, k, prod), mode))
    return seq


def per_acc(seq):
    out = {}
    for r, what, mode in seq:
        out.setdefault(r, []).append((what, mode))
    return out


def test_merged_schedule_equals_unmerged_per_accumulator():
    for products in (("lo8", "hi"), ("lo_hi", "hi_lo", "hi_hi")):          # F8 mode, three fp16 products
        a, b = per_acc(unmerged(products)), per_acc(merged(products))
        assert a.keys() == b.keys() == set(range(MR))
        for r in range(MR):
            assert a[r] == b[r], f"row {r}"
            assert a[r][0][1] == "overwrite" and all(m == "acc" for _w, m in a[r][1:])
            assert len(a[r]) == 3 * KW * KSTEPS * len(products)               # three tap rows per output row


def test_merged_mma_count_is_half():
    n_un = len(unmerged(("lo8", "hi")))
    mm = 0
    for sr in range(MR + 2):
        fresh = sr < MR
        rows = min(sr, MR - 1) - max(sr - 2, 0) + 1
        mm += KW * KSTEPS * 2 + (1 if fresh and rows > 1 else 0)
    assert n_un == 288 and mm == 144 + 3          # 144 + the three split-off first products of rows 1..3
