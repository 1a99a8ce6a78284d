"""Hydra-free loading of the reference's own task configs (``bez_isaacgym/cfg/task/*.yaml`` under ``cfg/config.yaml``).

The reference resolves its yaml files with Hydra + OmegaConf and four custom resolvers (``train.py:53-58``: ``eq``,
``contains``, ``if``, ``resolve_default``); neither package is needed for the handful of interpolations the task files use:
relative references to top-level keys of ``cfg/config.yaml`` (``${..physics_engine}``, ``${...num_envs}``, ``${....sim_device}``,
...) and the resolvers applied to them.  ``load_task_config`` parses a task yaml with PyYAML and resolves exactly those, so
``KickEnv(load_task_config(".../cfg/task/bez_kick.yaml", num_envs=4096), ...)`` takes the reference's file as it is.
"""
import re

import yaml

#: top-level defaults of the reference's cfg/config.yaml (:3-40)
TOP_LEVEL_DEFAULTS = dict(num_envs="", seed=42, physics_engine="physx", pipeline="gpu", sim_device="cuda:0", rl_device="cuda:0",
                          graphics_device_id=0, num_threads=4, solver_type=1, num_subscenes=4, test=False, checkpoint="",
                          multi_gpu=False, headless=False, experiment="", max_iterations="")

_REF = re.compile(r"\$\{(\.+)([A-Za-z_][A-Za-z0-9_.]*)\}")         # ${..key} / ${....task.env.numEnvs} / ${.name}


def _literal(text):
    text = text.strip()
    if len(text) >= 2 and text[0] == text[-1] and text[0] in "\"'":
        return text[1:-1]
    try:
        return yaml.safe_load(text)
    except yaml.YAMLError:
        return text


def _split_args(body):
    """Split resolver arguments on top-level commas (arguments may contain nested ${...})."""
    args, depth, cur = [], 0, ""
    for ch in body:
        if ch == "," and depth == 0:
            args.append(cur)
            cur = ""
            continue
        depth += ch == "{"
        depth -= ch == "}"
        cur += ch
    args.append(cur)
    return args


def _lookup(dots, path, top, siblings):
    """``${.name}`` is a sibling of the value being resolved; two or more dots climb to the composed root, where the top-level
    keys of cfg/config.yaml (and ``task`` for the train files) live."""
    node = siblings if len(dots) == 1 else top
    for part in path.split("."):
        node = node[part]
    return node


def _resolve(value, top, siblings=None):
    """Resolve one scalar: nested ${resolver:args} / relative ${..key} references, innermost first."""
    if not isinstance(value, str) or "${" not in value:
        return value
    text = value.strip()
    whole = _REF.fullmatch(text)
    if whole:
        return _resolve(_lookup(whole.group(1), whole.group(2), top, siblings or {}), top, siblings)
    if text.startswith("${") and text.endswith("}") and ":" in text:
        name, body = text[2:-1].split(":", 1)
        args = [_resolve(a.strip(), top, siblings) if "${" in a else _literal(a) for a in _split_args(body)]
        if name == "eq":                                   # train.py:53  lambda x, y: x.lower() == y.lower()
            return str(args[0]).lower() == str(args[1]).lower()
        if name == "contains":                             # train.py:54  lambda x, y: x.lower() in y.lower()
            return str(args[0]).lower() in str(args[1]).lower()
        if name == "if":                                   # train.py:55  lambda pred, a, b: a if pred else b
            return args[1] if args[0] else args[2]
        if name == "resolve_default":                      # train.py:58  lambda default, arg: default if arg == '' else arg
            return args[0] if args[1] == "" else args[1]
        raise ValueError(f"unknown resolver {name!r} in {value!r}")
    raise ValueError(f"cannot resolve {value!r}")


def _walk(node, top, siblings=None):
    if isinstance(node, dict):
        return {k: _walk(v, top, node) for k, v in node.items()}
    if isinstance(node, list):
        return [_walk(v, top, siblings) for v in node]
    return _resolve(node, top, siblings)


def load_task_config(path, **overrides):
    """Parse a reference task yaml and resolve its interpolations against ``cfg/config.yaml``'s top-level keys (``overrides``
    replace those: ``num_envs=``, ``pipeline=``, ``sim_device=``, ``rl_device=``, ...).  The result is the dict the reference's
    task constructors take; ``rl_device`` is added at the top level as ``VecTask`` expects."""
    top = dict(TOP_LEVEL_DEFAULTS)
    unknown = set(overrides) - set(top)
    if unknown:
        raise KeyError(f"unknown top-level config keys: {sorted(unknown)}")
    top.update(overrides)
    with open(path) as f:
        raw = yaml.safe_load(f)
    cfg = _walk(raw, top)
    cfg.setdefault("rl_device", top["rl_device"])
    cfg.setdefault("seed", top["seed"])
    return cfg


def load_train_config(path, task_cfg, **overrides):
    """Parse a reference train yaml (``cfg/train/*PPO.yaml``) against the composed root: cfg/config.yaml's top-level keys plus
    ``task`` (a dict from ``load_task_config``).  Returns the resolved ``params`` dict rl_games' ``Runner.load`` receives
    (``train.py:100-106``); ``agent_config`` extracts what ``learner.A2CAgent`` consumes."""
    top = dict(TOP_LEVEL_DEFAULTS)
    unknown = set(overrides) - set(top)
    if unknown:
        raise KeyError(f"unknown top-level config keys: {sorted(unknown)}")
    top.update(overrides)
    top["task"] = task_cfg
    with open(path) as f:
        raw = yaml.safe_load(f)
    return _walk(raw, top)


#: rl_games ``params.config`` keys that ``learner.A2CAgent`` understands
AGENT_KEYS = ("gamma", "tau", "learning_rate", "lr_schedule", "kl_threshold", "grad_norm", "truncate_grads", "e_clip", "horizon_length",
              "minibatch_size", "mini_epochs", "critic_coef", "clip_value", "entropy_coef", "bounds_loss_coef", "normalize_input",
              "normalize_value", "normalize_advantage", "value_bootstrap", "reward_shaper", "mixed_precision")


def agent_config(train_cfg):
    """``params.config`` of a resolved train yaml -> the ``config`` dict of ``learner.A2CAgent``."""
    c = train_cfg["params"]["config"]
    return {k: c[k] for k in AGENT_KEYS if k in c}


#: rl_games ``params.config`` keys of the training loop (``A2CBase.train``: meters, checkpoints, stop rules) that
#: ``learner.A2CAgent.train`` understands
TRAIN_LOOP_KEYS = ("games_to_track", "save_best_after", "save_frequency", "score_to_win", "max_epochs", "name")


def train_loop_config(train_cfg):
    """``params.config`` of a resolved train yaml -> the training-loop keys of ``learner.A2CAgent``'s ``config``.  The agent's
    ``track_outcomes`` (``learner.agent.OUTCOME_DEFAULTS``) and ``track_reward_terms`` (``learner.agent.REWARD_TERM_DEFAULTS``) are
    not read from the yaml: they are this project's own options, not rl_games settings, so callers pass them in the ``config`` dict
    themselves."""
    c = train_cfg["params"]["config"]
    return {k: c[k] for k in TRAIN_LOOP_KEYS if k in c}


#: rl_games ``params.config.player`` keys (``BasePlayer``) with their RECALLED defaults (v1.1.x); ``learner.PpoPlayerContinuous``
#: takes them as its ``config``
PLAYER_DEFAULTS = dict(games_num=2000, deterministic=True, print_stats=True, n_game_life=1)


def player_config(train_cfg):
    """``params.config.player`` of a resolved train yaml -> the ``config`` of ``learner.PpoPlayerContinuous``: ``games_num``,
    ``deterministic`` (rl_games' older spelling ``determenistic`` is accepted), ``print_stats``, ``n_game_life``, defaults
    filled in."""
    p = dict(train_cfg["params"]["config"].get("player") or {})
    if "deterministic" not in p and "determenistic" in p:
        p["deterministic"] = p["determenistic"]
    return {k: type(v)(p.get(k, v)) for k, v in PLAYER_DEFAULTS.items()}
