"""The table play kernels run 768 threads per CTA for large batches and 512 for small ones (play3_block_threads,
g2048_play3.cuh).  Keys derive from global env (playout) indices, so a batch launched whole -- large, 768 threads --
and the same batch launched in shards -- small, 512 threads -- must give the same per-env results, bit for bit, in the
plain form, the recording form and the playout form."""
import pytest
import torch

pytestmark = pytest.mark.gpu

MODE = 1  # partitionable
SHARDS = 8


@pytest.fixture(scope="module")
def E():
    from g2048 import engine

    assert torch.cuda.is_available()
    return engine


def _sizes():
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    big = 24 * sms * 768  # above 16 envs per lane of a 768-thread launch
    big -= big % SHARDS
    assert big // SHARDS < 16 * sms * 768  # every shard is a small launch
    return big, big // SHARDS


def _subs(E, seed, max_steps=2048):
    return E.chain_advance(E.words_tensor(list(E.key_words(seed)), "cuda"), MODE, 1 + 2 * max_steps)


@pytest.mark.parametrize("policy", [0, 1])
def test_play_whole_equals_shards(E, policy):
    n, part = _sizes()
    subs = _subs(E, 77 + policy)
    whole = E.play(policy, subs, n, 0, n, MODE)
    for key in ("final_boards", "lengths", "scores"):
        shards = torch.cat([E.play(policy, subs, n, lo, part, MODE)[key] for lo in range(0, n, part)])
        assert torch.equal(whole[key], shards), key


def test_recording_whole_equals_shards(E):
    n, part = _sizes()
    subs = _subs(E, 91)

    def flat(rec):
        lengths = rec["lengths"].to(torch.int64)
        off = torch.cumsum(lengths, 0) - lengths
        f = E.play_record_compact(rec, off, int(lengths.sum()))
        return rec, f

    rec, f = flat(E.play_record(0, subs, n, 0, n, MODE))
    assert E.play_stats_dict(rec["stats"])["episodes"] == n
    parts = [flat(E.play_record(0, subs, n, lo, part, MODE)) for lo in range(0, n, part)]
    for key in ("final_boards", "lengths", "scores"):
        assert torch.equal(rec[key], torch.cat([r[key] for r, _ in parts])), key
    for key in ("boards", "meta", "rewards", "max_rewards"):
        assert torch.equal(f[key], torch.cat([g[key] for _, g in parts])), key


def test_playouts_whole_equal_shards(E):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    k = 64
    n_boards = -(-24 * sms * 768 // (4 * k))  # 4 k playouts per board: above 16 per lane of a 768-thread launch
    n_boards += (-n_boards) % SHARDS
    subs = _subs(E, 5, max_steps=512)
    drul = E.play(1, subs, n_boards, 0, n_boards, MODE)["final_boards"]
    boards = drul & 0x00FF00FF00FF00FF  # end-of-game boards with half their tiles removed: mostly legal moves left
    whole = E.playout_values(0, boards, subs, k, MODE)["records"]
    part = n_boards // SHARDS
    shards = torch.cat([E.playout_values(0, boards[lo:lo + part], subs, k, MODE, board_lo=lo, n_boards_global=n_boards)["records"]
                        for lo in range(0, n_boards, part)])
    assert int(whole[..., 3].sum()) > 0
    assert torch.equal(whole, shards)
