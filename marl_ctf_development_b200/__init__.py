"""B200-native batched backend for the GridworldCtf step loop of g-nightingale/marl-ctf-development.

Public surface:
    GridworldCtfGPU   batched env (B envs per GPU), device tensors in / out
    GridworldCtf      single-env view with the reference's exact methods (drop-in for ppo.py / utils.py)
    FusedPolicy       CtfPolicy inference from packed observations (fused_policy.py)
    PolicyPool        several policies' inference on one env batch: one grouped trunk launch per forward (fused_policy.py)
    PackedPPO         PPO for a CtfPolicy from packed rollouts, advantages by the ctf_gae kernel (ppo.py)
    compressible_empty  torch.empty in compressible device memory, for caller-bound observation buffers
    compile_config    (AGENT_CONFIG, SCENARIO, kwargs) -> ctf_config_t
    experiment_env_config / experiment_names   the reference's nine experiment configs as data
"""
from .config import METRIC_NAMES, compile_config, env_dims  # noqa: F401
from .scenario_io import experiment_env_config, experiment_names, load_env_config  # noqa: F401


def __getattr__(name):
    # env.py imports torch; keep `import marl_ctf_development_b200` light for host-only users
    if name in ("GridworldCtfGPU", "GridworldCtf", "metrics_dict"):
        from . import env

        return getattr(env, name)
    if name == "compressible_empty":
        from .compressible import compressible_empty

        return compressible_empty
    if name in ("FusedPolicy", "PolicyPool"):
        from . import fused_policy

        return getattr(fused_policy, name)
    if name == "PackedPPO":
        from .ppo import PackedPPO

        return PackedPPO
    raise AttributeError(name)
