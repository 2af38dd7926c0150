"""Differential fuzz on FRESH seeds (none of these cases has a committed golden):
  CPU: the oracle against the unmodified reference binary (its STDOUT on these cases is stored as digests in
       tests/golden/reference_outputs.json) — pins the restatement on inputs nobody looked at: random CIGARs (D/N/=/X/H/P,
       P-then-I, leading deletions), missing NM/SM tags, filtered flags, reads without a library, -q/-b/-i/-p/-d.
  GPU: the engine against the oracle on the same cases, raw accumulators bit-for-bit, with and without the deep-site kernel
       forced onto the small tiles."""
import numpy as np
import pytest

import cases
import edge_cases

SEEDS = (101, 102, 103, 104, 105, 106)


def _case(seed):
    rng = np.random.default_rng(seed)
    safe = bool(seed % 2)
    return edge_cases.fuzz_case(seed, L=int(rng.integers(300, 700)), n_reads=int(rng.integers(150, 380)), name=f"fresh{seed}",
                                per_lib_safe=safe, n_libs=int(rng.integers(1, 6)), overhang=bool(seed % 3), force_perlib=not safe)


@pytest.mark.parametrize("seed", SEEDS)
def test_oracle_equals_reference_binary_on_fresh_fuzz(seed):
    case = _case(seed)
    for fname, fl in case["flag_sets"].items():
        want, _, _ = cases.run_oracle(case, fl, site_list=True)
        cases.assert_reference_output(f"fuzz {seed} {fname}", want.encode("latin-1"))


@pytest.mark.gpu
@pytest.mark.parametrize("deep", (False, True), ids=("pileup", "deep-forced"))
@pytest.mark.parametrize("seed", SEEDS)
def test_engine_equals_oracle_on_fresh_fuzz(seed, deep, monkeypatch):
    if deep:
        monkeypatch.setenv("BRC_DEEP_MIN_READS", "1")
    case = _case(seed)
    # single-base site-list lines as well as the whole contig: the small tiles are what the deep-site kernel takes
    L = case["contigs"][0][1]
    rng = np.random.default_rng(seed + 1000)
    case = dict(case, regions=[(0, 1, L)] + [(0, int(p), int(p)) for p in np.sort(rng.integers(2, L - 2, 25))])
    for fname, fl in case["flag_sets"].items():
        otext, odump, owarn = cases.run_oracle(case, fl, site_list=True)
        etext, edump, ewarn, _ = cases.run_engine(case, fl, site_list=True, want_dump=True)
        assert edump == odump, fname
        assert etext == otext, fname
        assert (ewarn[0], ewarn[1], ewarn[3]) == owarn, fname
