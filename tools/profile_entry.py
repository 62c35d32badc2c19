"""Where does a full self_play_v1_gpu(search_backend="tree") iteration spend its time?  Prints the wall clock per block of
4 plies with the live-game count and the wave-batch bucket (4,096 games x 200 sims, warmed-up engine)."""
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from liuzhou_b200 import self_play as sp  # noqa: E402
from liuzhou_b200.net import ChessNet, InferenceNet  # noqa: E402
from liuzhou_b200.actor import SelfPlayActor  # noqa: E402

games, sims = int(sys.argv[1]) if len(sys.argv) > 1 else 4096, int(sys.argv[2]) if len(sys.argv) > 2 else 200
torch.manual_seed(20260314)
net = InferenceNet(ChessNet(), "cuda:0")
actor = SelfPlayActor(net, games, device="cuda:0", mcts_simulations=sims, tree_reuse=True)
kw = dict(temperature_init=1.0, temperature_final=0.1, temperature_threshold=10, add_dirichlet_noise=True,
          sample_moves=True, opening_random_n=0, soft_value_k=2.0)
sp._play_wave_tree(actor, sp.TreePlyRules(max_plies=3, **kw))
torch.cuda.synchronize()
prog = []
t0 = time.perf_counter()
rows, rec, stats = sp._play_wave_tree(actor, sp.TreePlyRules(max_plies=512, **kw), progress=prog)
torch.cuda.synchronize()
t1 = time.perf_counter()
print(f"total {t1 - t0:.2f} s, {rows.shape[0]} positions -> {rows.shape[0] / (t1 - t0):.0f} positions/s; plies {actor._finish_plies}")
prev_t, prev_ply = t0, 0
for ply, live, t in prog:
    print(f"ply {ply:4d} live {live:5d} bucket {actor.mcts.bucket_for(live):5d}: {(t - prev_t) / max(1, ply - prev_ply) * 1e3:7.1f} ms/ply")
    prev_t, prev_ply = t, ply
print(f"tail (drain, ply-major reorder): {(t1 - prev_t) * 1e3:.0f} ms")
