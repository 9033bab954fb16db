"""TEST INFRASTRUCTURE -- CPU restatement of parse_bampe(pairing='name') (include/tecount.h, tec_bulk_begin(ctx, 2, qual)).

Not a crash site of the reference but a file layout: te_count.py:76-79 pairs record 2i with record 2i+1, which is only
right for a name-collated BAM.  Rule: a record takes part when it is primary and carries exactly one mate flag (0x1 set,
0x100 and 0x800 clear, exactly one of 0x40 / 0x80); within one exact QNAME the k-th read1 in file order pairs with the
k-th read2 in file order; records left over have no mate.  The pairs, each written read1 then read2, go through the
unchanged paired-end oracle (oracle/te_oracle.py, oracle/te_oracle_c.py).  Tests only; the product never imports it.
"""
from collections import defaultdict, deque


def name_role(flag):
    """1 read1, 2 read2, 0 excluded from pairing by name."""
    if not flag & 0x1 or flag & 0x900:
        return 0
    m = flag & 0xC0
    return 1 if m == 0x40 else 2 if m == 0x80 else 0


def collate_by_name(records):
    """records: dicts with at least 'name' and 'flag' (the SAM flag), in file order.  Returns (collated, n_excluded,
    n_no_mate): collated = [read1, read2, read1, read2, ...] in the order the second mate of each pair appears (bulk
    counting does not depend on the order of pairs)."""
    waiting = defaultdict(lambda: (deque(), deque()))
    collated = []
    excluded = 0
    for r in records:
        role = name_role(int(r.get("flag", 0)))
        if not role:
            excluded += 1
            continue
        mine, other = waiting[r["name"]] if role == 1 else waiting[r["name"]][::-1]
        if other:
            mate = other.popleft()
            collated += [mate, r] if role == 2 else [r, mate]
        else:
            mine.append(r)
    no_mate = sum(len(a) + len(b) for a, b in waiting.values())
    return collated, excluded, no_mate
