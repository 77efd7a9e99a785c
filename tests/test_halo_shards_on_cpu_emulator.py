"""The sharded halo exchange (ddc_halo_exchange_shards_f64) on a machine without a GPU.

tests/emu_halo_shards.cpp (built by tests/halo_emu.py) runs the product's own k_halo_open / k_halo_push / k_halo_close (ddc_kernels.cuh
compiled as host C++) for G emulated ranks, phase by phase, each rank pushing into the others' buffers as it would
over NVLink, and k_halo_exchange on one buffer beside them.  Interiors hold the global cell index, so every ghost
cell is checked for WHICH cell arrived (tests/halo_global.py); the sharded result must also equal the single-buffer
kernel bit for bit, over three exchanges whose interiors change in between.  Says nothing about speed."""
import itertools

import numpy as np
import pytest

import halo_emu
import halo_global as hg

RANKS = (1, 2, 3, 5)
SEEDS = ("0", "11", "4242")  # DDC_EMU_SCHED_SEED: "0" index order, otherwise random block / thread schedules


def decomposition(oracle, seed, px, py):
    rng = np.random.default_rng(seed)
    nx, ny = int(rng.integers(6, 40)), int(rng.integers(6, 40))
    P = int(rng.integers(2, 14)) if seed % 4 else 3  # every fourth case has fewer parts than the largest rank count
    mask = (rng.random((ny, nx)) > rng.uniform(0.1, 0.6)).astype(np.int32)
    return oracle.partition(mask, P, px, py, use_hist=True), nx, ny


def run(oracle, d, nx, ny, px, py, G, periodic, steps=3, stall=-1):
    off = hg.tile_offsets(d.boxes)
    tiles_in = np.stack([hg.initial_tiles(d.boxes, off, nx, 1000.0 * k) for k in range(steps)])
    out, single, err = halo_emu.emu_halo_shards(d, G, periodic, tiles_in, stall)
    return off, tiles_in, out, single, err


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_sharded_exchange_matches_single_buffer_and_expected(oracle, monkeypatch, G, sched):
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for case, (px, py) in enumerate(itertools.product((False, True), repeat=2)):
        for seed in (case, case + 4, case + 8):
            d, nx, ny = decomposition(oracle, seed, px, py)
            for periodic in (0, 1):
                ctx = (G, sched, seed, px, py, periodic, d.P)
                off, _, out, single, err = run(oracle, d, nx, ny, px, py, G, periodic)
                assert err.tolist() == [0] * G, ctx
                for k in range(out.shape[0]):
                    want = hg.expected_tiles(d.boxes, off, nx, ny, px, py, periodic, 1000.0 * k)
                    assert np.array_equal(single[k], want), ctx + (k, "single-buffer kernel")
                    assert out[k].tobytes() == single[k].tobytes(), ctx + (k, "sharded != single buffer")


def test_more_ranks_than_parts(oracle):
    """ranks without parts still take part in both barriers; the parts' ghosts are complete"""
    d, nx, ny = decomposition(oracle, 0, True, True)
    assert d.P == 3
    for G in (5, 8, 16):
        off, _, out, single, err = run(oracle, d, nx, ny, True, True, G, 1)
        assert err.tolist() == [0] * G
        assert out[-1].tobytes() == single[-1].tobytes()
        assert np.array_equal(out[-1], hg.expected_tiles(d.boxes, off, nx, ny, True, True, 1, 2000.0))


def test_one_part_is_a_no_op(oracle):
    d = oracle.partition(np.ones((9, 7), dtype=np.int32), 1)
    off = hg.tile_offsets(d.boxes)
    tiles_in = np.stack([hg.initial_tiles(d.boxes, off, 7)])
    out, single, err = halo_emu.emu_halo_shards(d, 2, 1, tiles_in)
    assert np.array_equal(out[0], tiles_in[0]) and np.array_equal(single[0], tiles_in[0])


def test_neighbour_lists_are_symmetric(oracle):
    """k_halo_push walks the lists of the SOURCE parts and finds its entry in the receiver's opposite-edge list: q is
    in p's edge-e list iff p is in q's opposite-edge list, with the same periodic flag and the same halo size"""
    for seed in range(24):
        px, py = bool(seed & 1), bool(seed & 2)
        d, _, _ = decomposition(oracle, seed, px, py)
        for per in range(2):
            for e in range(4):
                lists = {}
                for ee in (e, e ^ 1):
                    counts = d.nbr.counts[per][ee]
                    firsts = np.concatenate([[0], np.cumsum(counts)])
                    lists[ee] = {(p, int(q)): int(h) for p in range(d.P)
                                 for q, h in zip(d.nbr.ids[per][ee][firsts[p]:firsts[p + 1]],
                                                 d.nbr.halos[per][ee][firsts[p]:firsts[p + 1]])}
                mirrored = {(q, p): h for (p, q), h in lists[e ^ 1].items()}
                assert lists[e] == mirrored, (seed, per, e)


def test_a_rank_that_never_arrives(oracle):
    """emulation only: one rank runs none of the kernels; every other rank reports the timeout and writes nothing"""
    d, nx, ny = decomposition(oracle, 5, True, False)
    G = 3
    for stall in range(G):
        off, tiles_in, out, single, err = run(oracle, d, nx, ny, True, False, G, 1, steps=1, stall=stall)
        assert err.tolist() == [0 if r == stall else 1 for r in range(G)], stall
        for r, (b, c) in enumerate(hg.shard_ranges(d.P, G)):
            if r != stall:  # (the stalled rank's buffer is not checked: its peers write nothing either)
                sl = slice(int(off[b]), int(off[b + c]))
                assert np.array_equal(out[0][sl], tiles_in[0][sl]), (stall, r)


@pytest.mark.parametrize("P,G", [(1, 1), (7, 1), (7, 2), (7, 3), (3, 5), (16, 8), (4096, 8), (16384, 8), (1000, 3),
                                 (5, 16), (0, 4)])
def test_shard_parts(capi_lib, P, G):
    got = [capi_lib(P, G, r) for r in range(G)]
    assert got == hg.shard_ranges(P, G)
    assert got[0][0] == 0 and sum(c for _, c in got) == P  # covering ...
    for (b0, c0), (b1, _) in zip(got, got[1:]):
        assert b0 + c0 == b1  # ... contiguous ...
    assert max(c for _, c in got) - min(c for _, c in got) <= 1  # ... and balanced within one


@pytest.fixture(scope="module")
def capi_lib():
    from domain_decomp_b200 import capi
    return capi.shard_parts
