"""The self-play move commit when trajectory slots run out: the persistent kernel (SelfPlayEngine.play with E0) and the
stepwise path (search + SearchEngine.selfplay_step) give the same finish-queue rows, park the same games and pack the
same record bytes, with and without an opening book, with restart=True and then restart=False.

Which games win the few spare slots depends on the order games finish in, which the persistent kernel's warp schedule
decides; so games are compared by (game index, deal), where deal k is the k-th game that index played."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, NIR, S, G, EXTRA, SEED, NSEED = 6, 4, 16, 6, 2, 4, 9


def _persistent(book):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    eng = SearchEngine(G, board_size=N, n_in_row=NIR, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=SEED, noise_seed=NSEED, openings=book)

    def run(traj, restart):             # more moves than the slots allow: the launch ends once every game is parked
        sp.play(moves_per_game=4 * eng.A, traj=traj, restart=restart)
    return eng, run


def _stepwise(book):
    """Lock-step moves through the stepwise kernels, each game's noise drawn from its own search counter as the
    persistent kernel draws it; a parked game's root is inactive and its action -1."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    eng = SearchEngine(G, board_size=N, n_in_row=NIR, num_simulations=S)
    sp = SelfPlayEngine(eng, lambda obs: eng.e0_eval(obs, SEED), noise_seed=NSEED, openings=book)
    A, ctr = eng.A, np.zeros(G, np.int64)
    gum = torch.empty((G, A), dtype=torch.float64, device=eng.device)

    def run(traj, restart):
        for _ in range(4 * A):
            for g in range(G):
                eng.fill_gumbel(gum[g], NSEED, (int(ctr[g]) * G + g) * A)
            pol, val, act, _ = sp.search(gumbel=gum)
            moved = act.cpu().numpy() >= 0
            if not moved.any():
                return
            eng.selfplay_step(pol, val, act, traj, restart)
            ctr[:] += moved
        raise AssertionError("games still playing")
    return eng, run


def _play(make, book):
    """Phase 0: restart=True until every game is parked; pack and recycle (release + unpark).  Phase 1: restart=False
    until every game has finished once more; pack, then release its slots.  Returns the free-slot counts along the way,
    {(game, deal): (phase, slot or None, length, winner, record bytes)} and the roots left after the last unpark."""
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng, run = make(book)
    traj = TrajectoryStore(eng, extra_slots=EXTRA)
    body = 64 + 21 * eng.A                       # the tail padding of a record is not record content
    free, games, deals = [], {}, np.zeros(G, np.int64)
    for phase, restart in enumerate((True, False)):
        run(traj, restart)
        free.append(traj.free_slots_left())
        pg = traj.pack_finished(recycle=restart)
        free.append(traj.free_slots_left())
        if not restart:
            traj.release(pg.table[:, 0])
            free.append(traj.free_slots_left())
        raw = pg.records.cpu().numpy()[:, :body].copy()
        raw[:, 0:4] = 0                          # game_seq: the position in this pack, i.e. the finish order
        raw[:, 52:56] = 0                        # slot: popped in finish order
        for i, (slot, g, length, winner) in enumerate(pg.table.tolist()):
            k = int(deals[g])
            deals[g] += 1
            games[(g, k)] = (phase, slot if k == 0 else None, length, winner, raw[pg.offsets[i]:pg.offsets[i + 1]])
    roots = [t.cpu().numpy() for t in eng.get_roots()]
    return free, games, deals, roots


@pytest.mark.parametrize("with_book", [False, True])
def test_commit_paths_agree_when_slots_run_out(with_book):
    from test_openings_gpu import _book
    book = _book(N, NIR) if with_book else None
    fp, pers, dp, rp = _play(_persistent, book)
    fs, step, ds, rs = _play(_stepwise, book)
    # phase 0 ends with G + EXTRA finished games and every slot held; the unpark deals all G parked games, leaving EXTRA
    # free.  Phase 1 parks every game after one game; releasing its G slots unparks all G.
    assert fp == fs == [0, EXTRA, EXTRA, EXTRA, EXTRA]
    for games in (pers, step):
        assert sum(1 for v in games.values() if v[0] == 0) == G + EXTRA
        assert sum(1 for v in games.values() if v[0] == 1) == G
        assert all(v[1] == g for (g, k), v in games.items() if k == 0)     # deal 0 records into slot g (gmz_traj_init)
    both = sorted(set(pers) & set(step))
    assert all((g, 0) in both and (g, 1) in both for g in range(G))
    for key in both:
        a, b = pers[key], step[key]
        assert a[1:4] == b[1:4], key                    # a deal-1 game may finish in phase 0 on one path, 1 on the other
        assert np.array_equal(a[4], b[4]), key
    labels = np.array([pers[(g, 0)][4][0, 56:60].view(np.int32)[0] for g in range(G)])
    assert (labels > 0).all() if with_book else (labels == 0).all()
    # the games dealt by the last unpark: the same root wherever the index has played as many games
    same = dp == ds
    assert same.any()
    for x, y in zip(rp, rs):
        assert np.array_equal(x[same], y[same])
