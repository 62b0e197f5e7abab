"""Command line of the drop-in: the reference's flags with the reference's defaults and value checks
(reference main.py:5-14 flags, :21-53 checks, :56-70 dispatch), plus optional flags whose defaults keep the
reference behaviour.  `python main.py --dataset ml1m --epoch 50 --group 5 --learn sisa --delper 2 --deltype rand`
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
GROUP_TYPES = ('emb-ot',)                      # the only grouping the reference's CLI reaches (main.py:64)


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
    return p


parser = _build_parser()


def _checked(args):
    """The reference validates with bare asserts; keep AssertionError as the failure mode."""
    for name, (_, _, _, ok) in _FLAGS.items():
        v = getattr(args, name)
        assert ok(v) if callable(ok) else v in ok, f'--{name} {v!r} is not accepted'
    assert all(isinstance(w, int) for w in args.layer)
    assert 0 <= args.recommend <= 64, f'--recommend {args.recommend!r} is not accepted (0 .. 64)'
    return args


def main(argv=None):
    a = _checked(parser.parse_args(argv))
    if a.epoch_eval:
        os.environ['ULTRARE_EPOCH_EVAL'] = a.epoch_eval
    from . import dist as udist
    udist.init_from_env()
    from .config import InsParam, Instance
    if a.synth:
        from . import synth
        synth.ensure_dataset(a.dataset)
    ins = Instance(InsParam(a.dataset, a.epoch, a.worker, a.layer, a.group, a.delper, a.deltype))
    ins.recommend_n = a.recommend
    ins.combine = a.combine
    if a.group == 0:
        ins.runFull(is_save=True, verbose=a.verbose)
        return ins
    for group_type in GROUP_TYPES:
        ins.runGroup(is_save=True, learn_type=a.learn, group_type=group_type, n_group=a.group, verbose=a.verbose)
    return ins


if __name__ == '__main__':
    main()
