"""The GPU coverage lists of tests/test_gpu_coverage.py against the library source: every B7_* switch the library reads is
run by an execution variant or excluded with a reason, and every bucket of the dimension / width dispatch ladders is
reached by the dimensions and widths those tests use.  A new switch or a new bucket fails here until it is covered."""
import os
import re

import test_gpu_coverage as cov

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bot7_b200", "csrc")
MAX_DIMS = 40                                   # b7_gp_fit accepts 1 <= d < 40


def _src(name):
    with open(os.path.join(CSRC, name)) as fh:
        return fh.read()


def _all_sources():
    return {n: _src(n) for n in sorted(os.listdir(CSRC)) if n.endswith((".cu", ".cuh", ".h"))}


def _buckets(thresholds, top):
    """(lo, hi] ranges of an `if (x <= t)` ladder whose last case takes everything up to `top`."""
    edges = [0] + sorted(thresholds) + [top]
    return [(edges[i], edges[i + 1]) for i in range(len(edges) - 1) if edges[i + 1] > edges[i]]


def test_every_knob_is_run_or_excluded():
    read = set()
    for text in _all_sources().values():
        read |= set(re.findall(r'getenv\("(B7_[A-Z0-9_]+)"\)', text))
    assert len(read) >= 15                                           # the parse found the switches
    run = {k for _, env, _, _ in cov.VARIANTS for k in env}
    assert not run & set(cov.EXCLUDED_KNOBS), "a knob is both run and excluded"
    assert all(reason.strip() for reason in cov.EXCLUDED_KNOBS.values())
    missing = read - run - set(cov.EXCLUDED_KNOBS)
    assert not missing, f"B7_* switches read by the library with no execution variant and no exclusion: {sorted(missing)}"
    stale = (run | set(cov.EXCLUDED_KNOBS)) - read
    assert not stale, f"listed switches the library no longer reads: {sorted(stale)}"


def test_variant_table_is_well_formed():
    ids = [v[0] for v in cov.VARIANTS]
    assert len(ids) == len(set(ids))
    import gpu_variant_worker as W
    for vid, env, workloads, expect in cov.VARIANTS:
        assert set(workloads) <= set(W.WORKLOADS), vid
        assert all(k.startswith("B7_") and isinstance(v, str) for k, v in env.items()), vid
        assert expect in ("same", "oracle") or (expect.startswith("same_as:") and expect.split(":", 1)[1] in ids), vid
        assert env or vid in cov.PROFILED, f"{vid}: a variant must change something"


def test_every_dimension_bucket_is_swept():
    ladders = {"cov.cu": r"if \(d <= (\d+)\) return launch_dt<(\d+)>", "posterior_i8.cu": r"if \(d <= (\d+)\) B7_COV_SLICES\((\d+)\)"}
    for name, pat in ladders.items():
        pairs = [(int(a), int(b)) for a, b in re.findall(pat, _src(name))]
        assert len(pairs) >= 6 and all(a == b for a, b in pairs), name       # the parse found the ladder; DT = threshold
        for lo, hi in _buckets([a for a, _ in pairs], MAX_DIMS - 1):
            hit = [d for d in cov.SWEEP_D if lo < d <= hi]
            assert hit, f"{name}: no swept d in the DT bucket ({lo}, {hi}]"
    assert max(cov.SWEEP_D) == MAX_DIMS - 1 and min(cov.SWEEP_D) == 1


def test_every_blr_width_bucket_is_run():
    text = _src("blr.cu")
    dp_cases = [int(a) for a, b in re.findall(r"case (\d+): return launch_moments_dp<(\d+)>", text)]
    assert len(dp_cases) >= 7 and "default: return launch_moments_dp<64>" in text
    dp_hit = {(D + 7) // 8 * 8 for D in cov.BLR_D}
    for dp in dp_cases + [64]:
        assert dp in dp_hit, f"launch_moments_dp<{dp}> not reached by BLR_D {cov.BLR_D}"
    assert max(cov.BLR_D) == 64                                     # the head's limit, kMaxD
    mlp_cases = [int(a) for a, b in re.findall(r"case (\d+): rc = launch_mlp_layer<(\d+)>", text)]
    assert len(mlp_cases) >= 7 and "default: rc = launch_mlp_layer<64>" in text
    # input widths of the layers: the grid's dims, then each hidden width
    widths = [cov.BLR_INPUT_DIMS] + list(cov.BLR_HIDDEN)
    hit = {(h + 7) // 8 for h in widths}
    for c in mlp_cases:
        assert c in hit, f"launch_mlp_layer case {c} not reached by widths {widths}"
    assert any((h + 7) // 8 > max(mlp_cases) for h in widths), "the default case of the mlp width switch is not reached"
    assert len(cov.BLR_D) == len(cov.BLR_HIDDEN)
