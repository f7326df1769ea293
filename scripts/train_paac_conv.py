#!/usr/bin/env python
"""Mirror of the reference's scripts/train_paac_conv.py (CLI flags :95-121, wiring :30-92):

    python scripts/train_paac_conv.py --height=84 --clip_norm=1                      # config 3: 32 emulators, 1 GPU
    torchrun --nproc-per-node 8 scripts/train_paac_conv.py -ec 8192 --clip_norm=1    # config 5: env batch sharded

Flag names and defaults are the reference's; additions: --n_locusts, --max_updates, --no_cuda_graph,
--reward_indexing, --mask_terminals, --bootstrap_truncated, --fresh_noise, --physics, --action_repeat.
'-d/--device' accepts the reference's '/gpu:0' spelling.
"""
import argparse
import copy
import logging
import os
import signal
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

logging.getLogger().setLevel(logging.INFO)


def bool_arg(string):
    value = string.lower()
    if value == 'true':
        return True
    elif value == 'false':
        return False
    raise argparse.ArgumentTypeError("Expected True or False, but got {}".format(string))


def physics_ranges(spec):
    """'F=0.3:0.7,L=5:15' -> {'F': (0.3, 0.7), 'L': (5.0, 15.0)} (BatchedSwarmEnv's physics ranges); '' -> None."""
    if not spec:
        return None
    out = {}
    for item in spec.split(","):
        try:
            name, rng = item.split("=")
            lo, hi = rng.split(":")
            out[name.strip()] = (float(lo), float(hi))
        except ValueError:
            raise argparse.ArgumentTypeError("expected NAME=LO:HI[,NAME=LO:HI...], got %r" % spec)
    return out


def get_network_and_environment_creator(args, random_seed=3):
    import golds_rl_gym_b200 as pkg
    ec = pkg.submodule("agents.paac.environment_creator")
    pv = pkg.submodule("agents.paac.policy_v_network")
    env_creator = ec.SwarmEnvironmentCreator(n_locusts=args.n_locusts, grid_size=args.height,
                                             noise="fresh" if getattr(args, "fresh_noise", False) else "frozen",
                                             physics=getattr(args, "physics", None),
                                             action_repeat=getattr(args, "action_repeat", 1))
    args.num_actions = env_creator.num_actions
    args.random_seed = random_seed
    network_conf = {
        'num_actions': args.num_actions,
        'entropy_regularisation_strength': args.entropy_regularisation_strength,
        'device': args.device, 'height': args.height, 'width': args.height, 'channels': 3,
        'filters': args.filters, 'conv_layers': 2, 'scale': args.scale, 'clip_norm': args.clip_norm,
        'clip_norm_type': args.clip_norm_type, 'static_size': args.static_size,
        'temporal_size': args.temporal_size, 'static_hidden_size': args.static_hidden_size,
        'rnn_hidden_size': args.temporal_hidden_size,
    }

    def network_creator(name='local_learning'):
        conf = copy.copy(network_conf)
        conf['name'] = name
        return pv.ConvSingleAgentPolicyNetwork(conf)

    return network_creator, env_creator


# (flags, default, type, dest) -- names and defaults are the reference's (train_paac_conv.py:95-121)
REFERENCE_FLAGS = [
    (('-d', '--device'), '/gpu:0', str, 'device'),
    (('--e',), 0.1, float, 'e'),
    (('--alpha',), 0.99, float, 'alpha'),
    (('-lr', '--initial_lr'), 0.0001, float, 'initial_lr'),
    (('-lra', '--lr_annealing_steps'), 80000000, int, 'lr_annealing_steps'),
    (('--entropy',), 0.02, float, 'entropy_regularisation_strength'),
    (('--clip_norm',), 40.0, float, 'clip_norm'),
    (('--clip_norm_type',), 'global', str, 'clip_norm_type'),
    (('--gamma',), 0.99, float, 'gamma'),
    (('--max_global_steps',), 80000000, int, 'max_global_steps'),
    (('--max_local_steps',), 5, int, 'max_local_steps'),
    (('--single_life_episodes',), False, bool_arg, 'single_life_episodes'),
    (('-ec', '--emulator_counts'), 32, int, 'emulator_counts'),
    (('-ew', '--emulator_workers'), 8, int, 'emulator_workers'),
    (('-df', '--debugging_folder'), 'logs/', str, 'debugging_folder'),
    (('-rs', '--random_start'), True, bool_arg, 'random_start'),
    (('--scale',), 1000., float, 'scale'),
    (('--height',), 84, int, 'height'),
    (('--filters',), 32, int, 'filters'),
    (('--rnn-length',), 5, int, 'rnn_length'),
    (('--static-size',), 2, int, 'static_size'),
    (('--temporal-size',), 2, int, 'temporal_size'),
    (('--static-hidden-size',), 32, int, 'static_hidden_size'),
    (('--temporal-hidden-size',), 32, int, 'temporal_hidden_size'),
]


def get_arg_parser():
    parser = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    for flags, default, kind, dest in REFERENCE_FLAGS:
        parser.add_argument(*flags, default=default, type=kind, dest=dest)
    # additions of this implementation
    parser.add_argument('--n_locusts', default=None, type=int, help="SwarmEnv.N_LOCUSTS (default 80)")
    parser.add_argument('--max_updates', default=None, type=int)
    parser.add_argument('--no_cuda_graph', action='store_true')
    parser.add_argument('--reward_indexing', default='reference', choices=['reference', 'per_agent'])
    parser.add_argument('--mask_terminals', action='store_true')
    parser.add_argument('--bootstrap_truncated', action='store_true',
                        help="with --mask_terminals: bootstrap a TimeLimit truncation from V of the terminal observation")
    parser.add_argument('--fresh_noise', action='store_true',
                        help="advance the env noise row every step (SURVEY Q1 fixed); default: the reference's frozen row")
    parser.add_argument('--physics', default=None, type=physics_ranges,
                        help="per-env physics redrawn at every reset of each training env, e.g. 'F=0.3:0.7,L=5:15' "
                             "(columns noise, gravity, wind, F, L, dt; unnamed ones keep the reference's constant)")
    parser.add_argument('--action_repeat', default=1, type=int,
                        help="env steps per decision, rewards summed (frame skip); gamma stays per decision")
    parser.add_argument('--eval_every', default=30.0, type=float,
                        help="seconds between evaluation episodes on Swarm-eval-v0 (policy_monitor.py); 0 = off")
    parser.add_argument('--net_precision', default='fp32', choices=['fp32', 'tf32', 'bf16'],
                        help="policy net arithmetic (the reference trains in FP32)")
    parser.add_argument('--obs', default='auto', choices=['auto', 'compact', 'expanded'],
                        help="observation the net consumes: compact = (grid, positions) with conv1 factorised")
    return parser


def main(args):
    import torch
    import torch.distributed as dist
    import golds_rl_gym_b200 as pkg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.device.startswith('/gpu:') and world == 1:
        local = int(args.device.split(':')[1])
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    network_creator, env_creator = get_network_and_environment_creator(args)
    paac = pkg.submodule("agents.paac.paac")
    learner = paac.GridPAACLearner(network_creator, env_creator, args, reward_indexing=args.reward_indexing,
                                   mask_terminals=args.mask_terminals, use_cuda_graph=not args.no_cuda_graph,
                                   compact_obs={"auto": "auto", "compact": True, "expanded": False}[args.obs],
                                   net_precision=args.net_precision, bootstrap_truncated=args.bootstrap_truncated)

    def on_signal(signum, frame):            # train_paac_conv.py:47-58
        learner.cleanup()
        sys.exit(0)
    signal.signal(signal.SIGINT, on_signal)
    signal.signal(signal.SIGTERM, on_signal)
    monitor = None
    if args.eval_every > 0 and int(os.environ.get("RANK", "0")) == 0:
        os.makedirs(args.debugging_folder, exist_ok=True)
        pm = pkg.submodule("agents.paac.policy_monitor")
        sp = pkg.submodule("agents.state_processors")
        monitor = pm.SwarmPolicyMonitor(global_policy_net=learner.network,
                                        state_processor=sp.SwarmStateProcessor(grid_size=args.height),
                                        out_dir=args.debugging_folder, fresh_noise=args.fresh_noise,
                                        action_repeat=args.action_repeat)
    fps = learner.train(max_updates=args.max_updates, monitor=monitor, eval_every=args.eval_every,
                        summary_dir=args.debugging_folder)     # scalars: global_norm, rl/reward (summaries.jsonl)
    if int(os.environ.get("RANK", "0")) == 0:
        logging.info("done: %d global steps, %.1f frames/s", learner.global_step, fps)
    learner.cleanup()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main(get_arg_parser().parse_args())
