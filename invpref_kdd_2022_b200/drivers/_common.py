"""Shared body of the five drivers' ``main()`` (reference e.g. Coat_InvPref_explicit.py:57-190,
MovieLens_InvPref.py:57-190): seed, build model / evaluator / trainer, train, pick the best epoch."""
from __future__ import annotations

import argparse
import json
import os

import numpy as np
import torch

from .. import dataloader as dl
from ..evaluate import ExplicitTestManager, ImplicitTestManager
from ..models import InvPrefExplicit, InvPrefImplicit
from ..train import ExplicitTrainManager, ImplicitTrainManager
from ..utils import _show_me_a_list_func, merge_dict
from . import global_config


def default_device() -> torch.device:
    """INVPREF_DEVICE (e.g. ``cuda:3``) or cuda:0; the reference pins a GPU index at import time."""
    return torch.device(os.environ.get("INVPREF_DEVICE", "cuda:0"))


def run_main(implicit, device, model_config, train_config, evaluate_config, data_loader, random_seed,
             silent=False, auto=False, query=True, metric_list=None, use_item_pool=False):
    """``use_item_pool``: rank only the test item pool (Yahoo_InvPref_Implicit.py:87 and MIND_InvPref.py:87 pass
    True, MovieLens_InvPref.py:90 False).  Returns ``(best, best_indexes, result_at_best)`` like the reference
    mains (explicit: ``{metric: value}``; implicit: ``{'metric@k': value}``, utils.py:191-198)."""
    torch.manual_seed(random_seed)                      # seeding order as the reference (:68-71)
    torch.cuda.manual_seed(random_seed)
    torch.cuda.manual_seed_all(random_seed)
    np.random.seed(random_seed)
    Model = InvPrefImplicit if implicit else InvPrefExplicit
    model = Model(user_num=data_loader.user_num, item_num=data_loader.item_num, env_num=model_config['env_num'],
                  factor_num=model_config['factor_num'], reg_only_embed=model_config['reg_only_embed'],
                  reg_env_embed=model_config['reg_env_embed']).to(device)
    if implicit:
        evaluator = ImplicitTestManager(model=model, data_loader=data_loader,
                                        test_batch_size=evaluate_config['test_batch_size'],
                                        top_k_list=evaluate_config['top_k_list'], use_item_pool=use_item_pool)
    else:
        evaluator = ExplicitTestManager(model=model, data_loader=data_loader)
    train_tensor = torch.LongTensor(data_loader.train_data_np).to(device)
    assert train_tensor.shape[1] == 3
    Trainer = ImplicitTrainManager if implicit else ExplicitTrainManager
    tc = train_config
    train_manager = Trainer(
        model=model, evaluator=evaluator, training_data=train_tensor, device=device, batch_size=tc['batch_size'],
        epochs=tc['epochs'], cluster_interval=tc['cluster_interval'], evaluate_interval=tc['evaluate_interval'],
        lr=tc['lr'], invariant_coe=tc['invariant_coe'], env_aware_coe=tc['env_aware_coe'], env_coe=tc['env_coe'],
        L2_coe=tc['L2_coe'], L1_coe=tc['L1_coe'], alpha=tc['alpha'], use_class_re_weight=tc['use_class_re_weight'],
        test_begin_epoch=tc['test_begin_epoch'], begin_cluster_epoch=tc['begin_cluster_epoch'],
        stop_cluster_epoch=tc['stop_cluster_epoch'], use_recommend_re_weight=tc['use_recommend_re_weight'],
        tie_break_rng=tc.get('tie_break_rng', 'numpy'))
    train_tuple, test_tuple, cluster_tuple = train_manager.train(silent=silent, auto=auto)
    merged = merge_dict(test_tuple[0], _show_me_a_list_func)
    metric = evaluate_config['eval_metric']
    if implicit:
        k = evaluate_config['eval_k']
        stand = np.array(merge_dict(merged[metric], _show_me_a_list_func)[k])
        best = np.max(stand)                                            # MovieLens_InvPref.py:123
        label = f'{metric}@{k}'
    else:
        stand = np.array(merged[metric])
        best = np.min(stand)                                            # Coat_InvPref_explicit.py:117
        label = metric
    best_indexes = np.where(stand == best)[0].tolist()
    if not auto:
        print('Best {}:'.format(label), best, best_indexes)
    if query and not auto:
        out_dir = os.path.join(global_config.RESULT_SAVE_PATH, type(model).__name__, f'seed_{random_seed}')
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, 'result.txt'), 'w') as f:
            f.write('best {}: {}, {}\n'.format(label, best, best_indexes))
            f.write(json.dumps(merged, indent=4))
        with open(os.path.join(out_dir, 'config.txt'), 'w') as f:
            f.write('rand seed: ' + str(random_seed) + '\n')
            for cfg in (model_config, train_config, evaluate_config):
                f.write(json.dumps(cfg, indent=4) + '\n')
    if implicit:                                                        # utils.py:191-198
        result = {}
        for m in (metric_list or ['ndcg', 'recall', 'precision']):
            by_k = merge_dict(merged[m], _show_me_a_list_func)
            for kk in evaluate_config['top_k_list']:
                result[f'{m}@{kk}'] = by_k[kk][best_indexes[0]]
        return best, best_indexes, result
    result = {m: merged[m][best_indexes[0]] for m in (metric_list or ['mse', 'rmse', 'mae'])}
    return best, best_indexes, result


def cli(module, implicit, shape=None):
    """``python -m invpref_kdd_2022_b200.drivers.<name> [--epochs N] [--synthetic] [--seeds ...]``."""
    ap = argparse.ArgumentParser(description=module.__doc__)
    ap.add_argument('--epochs', type=int, default=None, help='override TRAIN_CONFIG["epochs"]')
    ap.add_argument('--seeds', type=int, nargs='*', default=None)
    ap.add_argument('--synthetic', action='store_true',
                    help='synthetic interactions of the config\'s shape (train.csv of MovieLens / MIND is not '
                         'in the reference checkout)')
    ap.add_argument('--dataset-root', default=global_config.DATASET_PATH)
    ap.add_argument('--numpy-stream-on-device', action='store_true',
                    help='draw the initial environments and the cluster tie-break rows from numpy\'s global stream '
                         'on the GPU: the same values and the same numpy state as the host draws, without their '
                         'host time')
    args = ap.parse_args()
    device = default_device()
    train_config = dict(module.TRAIN_CONFIG)
    if args.epochs is not None:
        train_config['epochs'] = args.epochs
    if args.numpy_stream_on_device:
        train_config['tie_break_rng'] = 'numpy_device'
    path = args.dataset_root + module.DATASET_PATH
    Loader = dl.YahooImplicitBCELossDataLoader if implicit else dl.ExplicitDataLoader
    if args.synthetic or not os.path.isfile(os.path.join(path, 'train.csv')):
        U, I, N = shape or (6040, 3706, 1_000_000)
        print(f'[{module.__name__}] synthetic interactions U={U} I={I} N={N}')
        tr = dl.synthetic_interactions(U, I, N, implicit)
        te = dl.synthetic_interactions(U, I, max(N // 20, 1000), implicit, seed=7)
        if implicit:
            te = te[te[:, 2] > 0]
        loader = Loader(path, device, train=tr, test=te)
        if implicit and getattr(module, 'HAS_ITEM_POOL_FILE', False):
            # synthetic stand-in for test_item_pool.csv: every test user's pool = its test positives + random items
            loader.set_item_pool(dl.synthetic_item_pool(te, U, I))
    elif implicit:
        loader = Loader(dataset_path=path, device=device,
                        has_item_pool_file=getattr(module, 'HAS_ITEM_POOL_FILE', False))
    else:
        loader = Loader(dataset_path=path, device=device)
    bests = []
    for seed in (args.seeds or module.RANDOM_SEED_LIST):
        print('\nBegin seed:', seed)
        out = module.main(device=device, model_config=module.MODEL_CONFIG, train_config=train_config,
                          evaluate_config=module.EVALUATE_CONFIG, data_loader=loader, random_seed=seed, query=False)
        bests.append(out[0])
    print(json.dumps(module.EVALUATE_CONFIG, indent=4))
    print(json.dumps(module.MODEL_CONFIG, indent=4))
    print(json.dumps(train_config, indent=4))
    print('Best perform mean:', np.mean(bests))
    print('Random seed list:', args.seeds or module.RANDOM_SEED_LIST)
