"""What pipeline.quantify_regions leaves on a region, as plain comparable data with the type of every value (tests of the
sharded pipeline compare two runs with it)."""


def value(v):
    """(type, value); an object with slots (AnchorHit) or a __dict__ (Allele) as its fields, each with its type."""
    if hasattr(v, "__slots__"):
        return type(v), [(k, type(getattr(v, k)), getattr(v, k)) for k in v.__slots__]
    if hasattr(v, "__dict__"):
        return type(v), [(k, type(x), x) for k, x in sorted(vars(v).items())]
    return type(v), v


def region_state(rr):
    reads = [(name, [(k, value(v)) for k, v in sorted(vars(rd).items())]) for name, rd in rr.read_dict.items()]
    alleles = getattr(rr, "allele_list", "unset")
    return dict(attrs=sorted(vars(rr)), reads=reads, cores=list(rr.read_core_seq_dict.items()),
                buffer_len=getattr(rr, "buffer_len", None),
                alleles=[value(a) for a in alleles] if isinstance(alleles, list) else alleles,
                removed=getattr(rr, "num_removed_reads", "unset"))


def first_difference(a, b):
    """A short description of where two lists of region states differ (None when they are equal)."""
    if len(a) != len(b):
        return f"{len(a)} regions against {len(b)}"
    for r, (x, y) in enumerate(zip(a, b)):
        for k in x:
            if x[k] != y[k]:
                if k == "reads":
                    for (n1, a1), (n2, a2) in zip(x[k], y[k]):
                        if (n1, a1) != (n2, a2):
                            return f"region {r}: read {n1} / {n2}: {[t for t in a1 if t not in a2]} vs {[t for t in a2 if t not in a1]}"
                return f"region {r}: {k} differs ({len(x[k]) if isinstance(x[k], list) else x[k]!r:.200})"
    return None
