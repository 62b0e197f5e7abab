"""Command line of the drop-in: the reference's flags with the reference's defaults and value checks
(reference main.py:5-14 flags, :21-53 checks, :56-70 dispatch), plus optional flags whose defaults keep the
reference behaviour.  `python main.py --dataset ml1m --epoch 50 --group 5 --learn sisa --delper 2 --deltype rand`
A request run applies a deletion request to a saved SISA state:
`python main.py --unlearn-from DIR --out OUT [--forget-users FILE] [--forget-ratings FILE] [--recommend N]`
"""
import argparse
import os

# flag -> (type, default, help, accepted values or predicate); Appendix A12: --layer parses integers
_FLAGS = {
    'dataset': (str, 'ml1m', 'dataset name', ('ml1m', 'toy')),
    'epoch': (int, 50, 'number of epochs', lambda v: v > 0),
    'worker': (int, 24, 'number of CPU workers', lambda v: v > 0),
    'verbose': (int, 1, 'verbose type', (0, 1, 2)),
    'group': (int, 2, 'number of groups', lambda v: v >= 0),
    'learn': (str, 'sisa', 'type of learning and unlearning', ('sisa',)),
    'delper': (int, 2, 'deleted user (or, with --deltype inter, rating) proportion', (2, 5)),
    'deltype': (str, 'rand', 'deletion type: rand = users, inter = single ratings', ('rand', 'inter')),
}
GROUP_TYPES = ('emb-ot', 'rating-ot')          # emb-ot: the grouping the reference's CLI reaches (main.py:64)


def _build_parser():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    for name, (typ, default, text, _) in _FLAGS.items():
        p.add_argument('--' + name, type=typ, default=default, help=text)
    p.add_argument('--layer', nargs='+', type=int, default=[64, 32], help='setting of layers')
    # not in the reference
    p.add_argument('--synth', action='store_true',
                   help='write a deterministic synthetic ML-1M-shaped data/ml1m/squ0_{train,test}.csv if absent')
    p.add_argument('--epoch-eval', default=None, choices=['faithful', 'final', 'none'],
                   help='per-epoch in-training evaluation fidelity of the SISA path')
    p.add_argument('--recommend', type=int, default=0, metavar='N',
                   help='also write every pass\'s top-N recommendations (rec{N}*.npy, seen items excluded); 0 = off')
    p.add_argument('--combine', default='mean', choices=['mean', 'fit'],
                   help='how the SISA shard models are combined for the final evaluation and the recommendations: '
                        'mean = the reference\'s plain mean, fit = a per-group least-squares combination refitted '
                        'on the retained data after every unlearn (combine.npy)')
    p.add_argument('--loss', default='mse', choices=['mse', 'bpr'],
                   help='training objective: mse = the reference\'s squared error on the rating, bpr = pairwise '
                        'ranking of each rated item over a sampled unrated one (implicit feedback, for --recommend); '
                        'BPR runs write under their own run name (..._bpr)')
    p.add_argument('--grouping', default='emb-ot', choices=GROUP_TYPES,
                   help='how users are grouped into shards: emb-ot = OT clustering of the user table of a --group 0 '
                        'run, rating-ot = OT clustering of the users\' rating rows of the training file (no earlier '
                        'run needed)')
    p.add_argument('--slices', type=int, default=1, metavar='R',
                   help='SISA slices per shard (1 .. 32): every shard trains in R stages and keeps the weights before '
                        'each, so an unlearn retrains a shard only from its first affected slice; 1 = unsliced')
    p.add_argument('--save-state', action='store_true',
                   help='every SISA pass also writes its model as state/ in its pass directory (Sisa.save_state)')
    p.add_argument('--unlearn-from', default=None, metavar='DIR',
                   help='request run: load the SISA state in DIR (a pass\'s state/) and unlearn the deletions of '
                        '--forget-users / --forget-ratings from it; dataset, shards, slices, epochs, combine and grouping '
                        'come from the state')
    p.add_argument('--out', default=None, metavar='OUT',
                   help='request run: the new, or empty, directory the unlearn pass and the updated state/ go to')
    p.add_argument('--forget-users', default=None, metavar='FILE',
                   help='request run: users to delete (.npy, or text with one id per line)')
    p.add_argument('--forget-ratings', default=None, metavar='FILE',
                   help='request run: ratings to delete (.npy [n, 2], or text with user,item per line)')
    return p


parser = _build_parser()

# request run: flag -> the manifest entry it must agree with when it is given
_FROM_STATE = {'dataset': 'dataset', 'group': 'K', 'slices': 'slices', 'epoch': 'epochs', 'combine': 'combine',
               'grouping': 'grouping', 'epoch_eval': 'epoch_eval', 'loss': 'loss'}
_NOT_WITH_REQUEST = ('delper', 'deltype', 'save_state')


def _given(argv):
    """{dest: value} of the flags given on the command line (defaults left out)."""
    p = _build_parser()
    for act in p._actions:
        act.default = argparse.SUPPRESS
    return vars(p.parse_args(argv))


def _checked(args):
    """The reference validates with bare asserts; keep AssertionError as the failure mode."""
    for name, (_, _, _, ok) in _FLAGS.items():
        v = getattr(args, name)
        assert ok(v) if callable(ok) else v in ok, f'--{name} {v!r} is not accepted'
    assert all(isinstance(w, int) for w in args.layer)
    assert 0 <= args.recommend <= 64, f'--recommend {args.recommend!r} is not accepted (0 .. 64)'
    assert 1 <= args.slices <= 32, f'--slices {args.slices!r} is not accepted (1 .. 32)'
    assert not (args.loss == 'bpr' and args.combine == 'fit'), \
        '--loss bpr cannot be combined with --combine fit (a least-squares fit on ratings; BPR scores are not ratings)'
    if args.slices > 1:
        assert args.epoch_eval != 'faithful', '--slices > 1 needs --epoch-eval final or none'
        assert args.group > 0, '--slices > 1 needs SISA shards (--group > 0)'
    request = (args.out, args.forget_users, args.forget_ratings)
    if args.unlearn_from is None:
        assert request == (None, None, None), '--out, --forget-users and --forget-ratings need --unlearn-from'
    else:
        assert args.out is not None, '--unlearn-from needs --out'
        assert args.forget_users is not None or args.forget_ratings is not None, \
            '--unlearn-from needs --forget-users or --forget-ratings'
    return args


def _check_against_state(given, man, state_dir):
    """A request run takes its settings from the state's manifest: a flag given with another value is an error."""
    for flag in _NOT_WITH_REQUEST:
        assert flag not in given, f'--{flag.replace("_", "-")} has no meaning with --unlearn-from'
    for flag, key in _FROM_STATE.items():
        if flag in given:
            assert given[flag] == man[key], (f'--{flag.replace("_", "-")} {given[flag]!r} conflicts with the state in '
                                             f'{state_dir}, which has {key} = {man[key]!r}')


def _request(a, argv):
    from .config import check_out_dir, run_request
    from .method import sisa_state as st
    man = st.read_manifest(a.unlearn_from)
    _check_against_state(_given(argv), man, a.unlearn_from)
    check_out_dir(a.out)
    users = st.parse_request_file(a.forget_users, 'users') if a.forget_users else ()
    pairs = st.parse_request_file(a.forget_ratings, 'ratings') if a.forget_ratings else ()
    return run_request(a.unlearn_from, a.out, users, pairs, a.recommend, a.verbose)


def main(argv=None):
    a = _checked(parser.parse_args(argv))
    if a.unlearn_from is not None:
        from . import dist as udist
        udist.init_from_env()
        return _request(a, argv)
    if a.epoch_eval:
        os.environ['ULTRARE_EPOCH_EVAL'] = a.epoch_eval
    elif a.slices > 1:                  # the sliced passes evaluate the final models only
        os.environ['ULTRARE_EPOCH_EVAL'] = "final"
    from . import dist as udist
    udist.init_from_env()
    from .config import InsParam, Instance
    if a.synth:
        from . import synth
        synth.ensure_dataset(a.dataset)
    param = InsParam(a.dataset, a.epoch, a.worker, a.layer, a.group, a.delper, a.deltype)
    param.loss = a.loss
    ins = Instance(param)
    ins.recommend_n = a.recommend
    ins.combine = a.combine
    ins.slices = a.slices
    ins.save_state = a.save_state
    if a.group == 0:
        ins.runFull(is_save=True, verbose=a.verbose)
        return ins
    ins.runGroup(is_save=True, learn_type=a.learn, group_type=a.grouping, n_group=a.group, verbose=a.verbose)
    return ins


if __name__ == '__main__':
    main()
