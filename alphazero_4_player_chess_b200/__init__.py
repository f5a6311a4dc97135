"""B200-native batched four-player-chess environment for the AlphaZero self-play hot path.

Public surface (everything runs in libfpc.so's sm_100a kernels behind the C-ABI of include/fpc.h; there is no CPU path):

  BatchedEnv      N games resident in HBM, tensors owned by PyTorch      (env.py; alphazero_cpp.Board batch calls)
  NativeEnv       the same store owned by the library, DLPack export      (native_env.py; fpc_env_*)
  BatchedMCTS     GPU-resident PUCT search, one warp per game's tree      (mcts.py; fpchess::Node + src/py/mcts.py)
  SelfPlay        device-resident self-play driver                        (selfplay.py; src/py/alphazero.py:81-179)
  Learner         replay store + optimiser loop, DDP across GPUs          (train.py; src/py/alphazero.py:181-276)
  Player, Arena, MatchResult   paired, team-swapped evaluation games between two players, score and Elo interval
                               (arena.py; no counterpart in the reference)
  PolicyValueNet, InferenceNet   the reference's ResNet in PyTorch        (net.py; src/py/net.py)
  GEOMETRIES, start_record, record_from_fen, Shard; perft.perft(R, record, depth) is the GPU perft
  dropin/alphazero_cpp  the pybind11 module with the reference's binding API (csrc/binding.cpp; build.build_binding())

Attributes are imported on first use so that `import alphazero_4_player_chess_b200` stays cheap (no torch import)."""
from __future__ import annotations

import importlib

_EXPORTS = {
    "BatchedEnv": ".env", "NativeEnv": ".native_env", "BatchedMCTS": ".mcts", "SelfPlay": ".selfplay",
    "Learner": ".train", "ReplayStore": ".train", "Player": ".arena", "Arena": ".arena", "MatchResult": ".arena",
    "PolicyValueNet": ".net", "InferenceNet": ".net",
    "GEOMETRIES": ".geometry", "Geometry": ".geometry", "start_record": ".fen", "record_from_fen": ".fen",
    "START_FENS": ".fen", "Shard": ".shard", "FpcError": "._lib",
}
__all__ = sorted(_EXPORTS)


def __getattr__(name: str):
    mod = _EXPORTS.get(name)
    if mod is None:
        raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
    return getattr(importlib.import_module(mod, __name__), name)
