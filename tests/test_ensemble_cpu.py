"""Host-side logic of ensemble sampling: member key derivation, the chunk plan and the per-rank member ranges."""
import wsr

dmod = wsr.sub("models.diffusion_models.diffusion")
par = wsr.sub("parallel")


def test_member_keys():
    seed = 123456789
    assert dmod.member_key(seed, 0) == seed                        # member 0 is the plain single-GPU run
    assert dmod.member_key(seed, 3) == dmod.rank_stream_seed(seed, 3)
    keys = [dmod.member_key(seed, m) for m in range(256)]
    assert len(set(keys)) == 256 and all(0 <= k < 2 ** 62 for k in keys)
    assert dmod.member_key(seed + 1, 1) != keys[1]
    # splitmix64(seed + m * golden) masked to 62 bits, written out
    m64 = (1 << 64) - 1
    z = (seed + 5 * 0x9E3779B97F4A7C15) & m64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m64
    assert dmod.member_key(seed, 5) == (z ^ (z >> 31)) & ((1 << 62) - 1)


def test_chunk_plan():
    assert dmod.ensemble_chunks(10, 8, 64) == [(0, 8), (8, 2)]
    assert dmod.ensemble_chunks(16, 4, 64) == [(0, 16)]
    assert dmod.ensemble_chunks(5, 100, 64) == [(0, 1), (1, 1), (2, 1), (3, 1), (4, 1)]       # at least one member per chunk
    assert dmod.ensemble_chunks(3, 2, 4, member_offset=6) == [(6, 2), (8, 1)]
    for n, b, cap in ((37, 3, 64), (8, 8, 64), (1, 2, 64)):
        chunks = dmod.ensemble_chunks(n, b, cap)
        assert sum(c for _, c in chunks) == n
        assert [f for f, _ in chunks] == [sum(c for _, c in chunks[:i]) for i in range(len(chunks))]


def test_member_ranges_per_rank():
    for n, world in ((16, 2), (7, 3), (2, 4)):
        ranges = [par.shard_bounds(n, r, world) for r in range(world)]
        assert ranges[0][0] == 0 and ranges[-1][1] == n
        assert all(ranges[i][1] == ranges[i + 1][0] for i in range(world - 1))
        sizes = [hi - lo for lo, hi in ranges]
        assert max(sizes) - min(sizes) <= 1
