"""Small end-to-end run for compute-sanitizer: fused search, stepwise search, self-play packed into the device
replay ring, PER, tactics -- tiny sizes."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from datou_gomoku_muzero_b200.config import config
from datou_gomoku_muzero_b200.engine import SearchEngine
from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
from datou_gomoku_muzero_b200 import replay_buffer as rb
from datou_gomoku_muzero_b200.tactics import classify_boards
for N, S, G in ((6, 24, 10), (15, 40, 9), (19, 20, 5)):
    A = N * N
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    eng.reset_games()
    gum = torch.empty((G, A), dtype=torch.float64, device="cuda"); eng.fill_gumbel(gum, 1, 0)
    eng.search_e0(gum, 3, 16, trace=True); eng.finalize()
    eng.search_stepwise_e0(gum, 3, 16); eng.finalize()
    # packed records -> device replay ring + PER tree -> batch (float32 accumulation, dense logits)
    e32 = SearchEngine(G, board_size=N, num_simulations=S, accum_dtype="float32")
    sp32 = SelfPlayEngine(e32, "e0", seed=5, logit_div=0, noise_seed=6)
    t32 = TrajectoryStore(e32, extra_slots=8)
    ring = rb.DeviceReplayBuffer(64, N)
    sp32.play(moves_per_game=A, traj=t32, sink=ring.add_packed, chunk=7)
    if len(ring) >= 4:
        (obs, act, rew, pi, val), idx, w = ring.sample(4, rot_k=1, flip=True)
        ring.update_priorities(idx, val[:, 0] - 0.5)
    b, pl, lm, mc = eng.get_roots()
    classify_boards(b, pl, N)
    mz = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero")
    mz.reset_games()
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0
    e0 = TorchE0(N, seed=4)
    MuZeroDeviceSearch(mz, e0.initial, e0.recurrent).search(gum); mz.finalize()
    mz.search_e0(gum, 4, 0); mz.finalize()                      # fused MuZero-mode kernel, dense heads
config.ENABLE_PER = True
buf = rb.InMemoryReplayBuffer(37)
for i in range(50):
    buf.add(i)
batch, idx, w = buf.sample(8)
buf.update_priorities(idx, np.random.randn(8).astype(np.float32))
torch.cuda.synchronize()
print("sanity_small OK")
