"""The oracle's matchAll on reads longer than 2048 bases, up to the 65535 bases the product accepts, against a brute-force
numpy restatement that tests every window of the text: seed of at most `s` mismatches, whole read of at most `e`, inside one
record and free of N.  Scores are recomputed in float64, added in read order like the reference, then cast to float32."""
import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import synth
from util import brute_match_all, canon_hits


def long_read_case(seed, seedl):
    """A 160 kbp text of three records with an N run and a near-identical repeat, and reads of 2080..65535 bases planted in
    it with substitutions, on both strands, with a quality byte per base drawn from 0..255.  Some reads must not match:
    too many substitutions, substitutions in the seed, a window across a record boundary, a window over the N run."""
    rng = np.random.RandomState(seed)
    n = 160_000
    sym = rng.randint(0, 4, n).astype(np.uint8)
    seg = sym[5_000:9_200].copy()
    seg[[150, 2_222, 3_999]] ^= 1                          # the repeat: 3 substitutions away from the original
    sym[75_000:79_200] = seg
    sym[100_000:100_064] = 4
    text = synth.Text(sym, [(" a", 0), (" b", 70_000), (" c", 140_000)])
    clean = np.where(sym > 3, 1, sym).astype(np.uint8)

    seqs, quals, plan = [], [], []

    def plant(L, pos, inv, nsub, in_seed=0, valid=True):
        r = clean[pos:pos + L].copy()
        seed_at = L - seedl if inv else 0                 # where the seed lies in the text window
        rest = np.setdiff1d(np.arange(L), np.arange(seed_at, seed_at + seedl))
        where = list(rng.choice(rest, nsub, replace=False)) + list(seed_at + rng.choice(seedl, in_seed, replace=False))
        for j in where:
            r[j] = (r[j] + 1 + rng.randint(0, 3)) & 3
        if inv:
            r = synth.revcomp_mapped(r)
        seqs.append(r)
        quals.append(rng.randint(0, 256, L).astype(np.uint8))
        plan.append((valid, in_seed, nsub + in_seed))

    plant(2080, 1_000, 0, 3)
    plant(2081, 1_000, 0, 4)
    plant(2081, 30_000, 1, 2, in_seed=1)
    plant(4099, 5_000, 0, 2)                              # also hits the repeat with 3 more substitutions
    plant(4099, 4_990, 1, 1)
    plant(10_000, 141_000, 1, 9)
    plant(65_535, 2_000, 0, 8)
    plant(65_535, 3_000, 1, 12, in_seed=2)
    plant(65_535, 4_000, 0, 13)                           # more than e substitutions
    plant(2081, 20_000, 0, 0, in_seed=3)                  # more than s substitutions in the seed
    plant(4099, 68_000, 0, 0, valid=False)                # window across the record boundary at 70000
    plant(4099, 98_000, 1, 0, valid=False)                # window over the N run
    return text, synth.reads_from_list(seqs, quals), plan


@pytest.mark.parametrize("seedl,s,e", [(32, 2, 12), (12, 2, 15), (64, 1, 9)])
def test_oracle_long_reads_vs_brute_force(seedl, s, e):
    text, reads, plan = long_read_case(7 + seedl, seedl)
    ll = O.build_ll()
    got = canon_hits(O.match_all(text, reads, seedl=seedl, seedkmax=s, totalkmax=e, scores=True, ll=ll))
    want = brute_match_all(text, reads, seedl, s, e, ll)
    assert got.shape == want.shape and np.array_equal(got, want)
    # exactly the reads whose planted window passes both tests match (the reference's limit used to be seedl + 2048 bases)
    want_reads = {r for r, (valid, ks, k) in enumerate(plan) if valid and ks <= s and k <= e}
    assert set(got[:, 0].tolist()) == want_reads and len(want_reads) >= 6
    assert (np.diff(reads.offsets.astype(np.int64))[sorted(want_reads)] == 65535).any()
