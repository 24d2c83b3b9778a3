"""skill-chaining-with-graphs_b200 - B200-native hot path of skill chaining on Pinball.

Hand-written sm_100a CUDA kernels behind a C ABI (include/scg_b200.h, built in-tree as
libscg_b200.so) with a thin Python host layer that mirrors the interface of the CPU oracle
standing in for the reference (the reference ships no code: /root/reference/README.md:1-2):

    PinballMap, PinballEnv       env.reset / env.step                      (K1)
    FourierBasis, OptionSet, Option   initiation / act / update / fit_initiation   (K2, K3, K4)
    SkillChainAgent, AgentConfig      step / manage / run_episode / sync     (fused pipeline + NCCL)

The directory name contains hyphens, so it is imported through the alias package
`skill_chaining_with_graphs_b200` at the repository root.  There is no CPU fallback: every
operator raises if libscg_b200.so or a CUDA device is missing.
"""
from ._lib import LIB_PATH, EXPORTS, ScgError, load as load_library
from .pinball import PinballMap, PinballEnv, unpack_flags
from .option import FourierBasis, OptionSet, Option
from .agent import SkillChainAgent, AgentConfig, merge_episodes, merge_occupancy

__all__ = ["LIB_PATH", "EXPORTS", "ScgError", "load_library", "PinballMap", "PinballEnv", "unpack_flags",
           "FourierBasis", "OptionSet", "Option", "SkillChainAgent", "AgentConfig", "merge_episodes",
           "merge_occupancy"]
