"""Play a match between two players on one GPU and print MatchResult.summary() and a JSON line.

A player is a network and search settings.  The network is a PolicyValueNet state_dict file (--net-a / --net-b,
loaded with torch.load(..., weights_only=True)) or random initial weights (--init-seed-a / --init-seed-b), of
--blocks-X x --hidden-X, in bf16 unless --fp32-X.  The search settings are key=value pairs: C and num_searches go to
the reference's args dict, the rest to BatchedMCTS (cuda_graph defaults to 1 here), e.g.

  python tools/arena.py --start STANDARD --pairs 512 --a "num_searches=400" --b "gumbel=1,num_searches=32"

All search and scoring logic is alphazero_4_player_chess_b200.arena's."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from alphazero_4_player_chess_b200.arena import Arena, Player  # noqa: E402
from alphazero_4_player_chess_b200.fen import START_FENS, start_record  # noqa: E402
from alphazero_4_player_chess_b200.net import InferenceNet, PolicyValueNet  # noqa: E402

FLAGS = {"cuda_graph", "batch_rotation", "gumbel", "gumbel_interior"}
FLOATS = {"C", "gumbel_scale"}


def parse_search(text: str):
    """'k=v,k=v' -> (args, BatchedMCTS keyword arguments)."""
    args, search = {"C": 3.0, "num_searches": 32}, {"cuda_graph": True}
    for item in filter(None, (s.strip() for s in text.split(","))):
        key, _, value = item.partition("=")
        key = key.strip()
        v = bool(int(value)) if key in FLAGS else float(value) if key in FLOATS else int(value)
        (args if key in ("C", "num_searches") else search)[key] = v
    return args, search


def network(R, path, init_seed, blocks, hidden, fp32):
    torch.manual_seed(init_seed)
    model = PolicyValueNet(R, blocks, hidden, device="cuda")
    if path:
        model.load_state_dict(torch.load(path, map_location="cuda", weights_only=True))
    return InferenceNet(model.eval(), bf16=not fp32)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--start", default="STANDARD", choices=sorted(START_FENS))
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--opening-plies", type=int, default=8)
    ap.add_argument("--max-game-length", type=int, default=200)
    ap.add_argument("--seed", type=int, default=0)
    for side in "ab":
        ap.add_argument(f"--{side}", default="", help="search settings, e.g. 'gumbel=1,num_searches=32'")
        ap.add_argument(f"--net-{side}", default=None, help="PolicyValueNet.state_dict() file")
        ap.add_argument(f"--init-seed-{side}", type=int, default=0, help="random initial weights without --net")
        ap.add_argument(f"--blocks-{side}", type=int, default=10)
        ap.add_argument(f"--hidden-{side}", type=int, default=128)
        ap.add_argument(f"--fp32-{side}", action="store_true", help="fp32 network instead of bf16")
        ap.add_argument(f"--name-{side}", default=side.upper())
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/arena.py needs a GPU")
    _, R = START_FENS[opt.start]
    players = []
    for side in "ab":
        o = {k: getattr(opt, f"{k}_{side}") for k in ("net", "init_seed", "blocks", "hidden", "fp32", "name")}
        args, search = parse_search(getattr(opt, side))
        net = network(R, o["net"], o["init_seed"], o["blocks"], o["hidden"], o["fp32"])
        players.append(Player(net, args, name=o["name"], **search))
    arena = Arena(R, opt.pairs, *players, start_record(opt.start), opening_plies=opt.opening_plies,
                  max_game_length=opt.max_game_length, seed=opt.seed)
    res = arena.play()
    print(res.summary())
    print(json.dumps({"start": opt.start, "opening_plies": opt.opening_plies, "max_game_length": opt.max_game_length,
                      "seed": opt.seed, "a": repr(players[0]), "b": repr(players[1]), **res.to_json()}))


if __name__ == "__main__":
    main()
