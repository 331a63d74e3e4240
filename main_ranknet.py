"""RankNet ('sum_session') training entry point -- the flow, variable names and defaults of the reference's
``main_ranknet.py`` (main_ranknet.py:17-172) with its placeholders turned into command-line arguments.

    python main_ranknet.py --synthetic 64,64 --path /tmp/rr_ranknet --gpu 0 --batch_size 4096 --total_epochs 2
"""
import argparse
import logging
import os

import pandas as pd
import torch

from reactranker.data.load_reactions import get_data, Parsing_features
from reactranker.models.base_model import build_model
from reactranker.train.run_train_pairwise import run_train
from reactranker.train.test_ranknet import test
from reactranker.train.utils import build_optimizer, build_lr_scheduler
from main import add_finetune_args, apply_finetune_args, check_finetune_args


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--path", default="runs/reactranker_ranknet")
    ap.add_argument("--data_path", default=None)
    ap.add_argument("--synthetic", default=None, help="G,N: G synthetic groups of N candidates")
    ap.add_argument("--filter_size", type=int, default=3)
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--k_fold", type=int, default=1)
    ap.add_argument("--batch_size", type=int, default=4096)
    ap.add_argument("--total_epochs", type=int, default=30)
    ap.add_argument("--target_name", default="lgk")
    ap.add_argument("--split_strategy", default="random_flag", choices=["random", "random_flag"])
    ap.add_argument("--init_lr", type=float, default=1e-4)
    ap.add_argument("--max_lr", type=float, default=1e-3)
    ap.add_argument("--final_lr", type=float, default=1e-4)
    ap.add_argument("--save_metric", default="all")
    ap.add_argument("--train_strategy", default="sum_session", choices=["sum_session", "accelerate_grad"])
    ap.add_argument("--resume", action="store_true", help="write <path>/<fold>.state.pt after every epoch and continue from it if present")
    ap.add_argument("--deterministic", action="store_true",
                    help="torch.use_deterministic_algorithms(True): bit-identical losses, gradients and weights from the same seed")
    add_finetune_args(ap)
    return check_finetune_args(ap, ap.parse_args())


def main():
    a = parse()
    if a.deterministic:
        torch.use_deterministic_algorithms(True)
    from reactranker_b200 import parallel
    rank, world, local_rank = parallel.world_from_env()        # under torchrun: one process per GPU, windows sharded by group
    if world > 1:
        a.gpu = local_rank
    path = a.path
    os.makedirs(path, exist_ok=True)
    logging.basicConfig(filename=path + ('/output.log' if rank == 0 else '/output.rank{}.log'.format(rank)), level=logging.INFO, format='%(asctime)s - %(message)s', datefmt='%d-%b-%y %H:%M:%S')
    logger = logging.getLogger()
    smiles2graph_dic = Parsing_features()
    if a.synthetic:
        from reactranker_b200 import synthetic
        G, N = (int(v) for v in a.synthetic.split(","))
        ds = synthetic.make_dataset(0, [N] * G)
        for tok, m in ds.mols.items():
            smiles2graph_dic.add(tok, m)
        data = get_data(None)
        data.df = ds.to_dataframe()
    else:
        data = get_data(a.data_path)
        data.read_data()
    data.filter_bacth(filter_szie=a.filter_size)
    k_fold, gpu = a.k_fold, a.gpu
    test_score = []
    train_strategy = a.train_strategy          # main_ranknet.py:62 hard-codes 'sum_session'
    batch_size, total_epochs = a.batch_size, a.total_epochs
    target_name = a.target_name
    smiles_list = ['rsmi_mapped', 'psmi_mapped']
    init_lr, max_lr, final_lr = a.init_lr, a.max_lr, a.final_lr
    save_metric = a.save_metric
    add_features_dim = 1
    add_features_name = 'temp'
    if save_metric == 'all':
        path = [os.path.join(path, i) for i in ["T1", "T25_in_T25", "T25"]]
        for p in path:
            os.makedirs(p, exist_ok=True)
    for ii in range(k_fold):
        seed = ii
        k_fold_str = str(ii) + '.pt'
        path_checkpoints = os.path.join(path, k_fold_str) if save_metric != 'all' else [os.path.join(i, k_fold_str) for i in path]
        split_type = 'reactants' if a.split_strategy == 'random' else 'flag'
        train_data, val_data, test_data = data.split_data(split_size=(0.8, 0.1, 0.1), split_type=split_type, seed=seed)
        train_len = train_data.shape[0]
        torch.manual_seed(seed)
        torch.cuda.manual_seed(seed)
        torch.cuda.manual_seed_all(seed)
        model = build_model(hidden_size=300, mpnn_depth=3, mpnn_diff_depth=3, ffn_depth=3, use_bias=True, dropout=0.2, task_num=1,
                            ffn_last_layer='no_softplus', add_features_dim=add_features_dim)       # main_ranknet.py:113-121
        frozen = apply_finetune_args(a, model, logger)
        torch.cuda.set_device(gpu)
        model = model.cuda(gpu)
        optimizer = build_optimizer(model, freeze=frozen)
        scheduler = build_lr_scheduler(optimizer, warmup_epochs=2, total_epochs=total_epochs, train_data_size=train_len, batch_size=batch_size,
                                       init_lr=init_lr, max_lr=max_lr, final_lr=final_lr)
        run_train(model, scheduler, train_data, val_data, path_checkpoints, optimizer, total_epochs, smiles2graph_dic, batch_size=batch_size,
                  seed=seed, gpu=gpu, train_strategy=train_strategy, task_type='baseline', writer=None, logger=logger, smiles_list=smiles_list,
                  target_name=target_name, save_metric=save_metric, add_features_name=add_features_name,
                  resume_path=os.path.join(a.path, str(ii) + '.state.pt') if a.resume else None)
        if rank != 0:
            continue
        test_path = path_checkpoints[0] if save_metric == 'all' else path_checkpoints
        score, score3, average_pred_in_targ = test(model, test_data, test_path, smiles2graph_dic, batch_size, gpu=gpu, logger=logger,
                                                   smiles_list=smiles_list, add_features_name=add_features_name, target_name=target_name,
                                                   train_strategy=train_strategy)
        test_score.append([score, score3])
    if rank == 0:
        print("test score for k_fold vailidation is: ", test_score)
        logger.info('test score for k_fold vailidation is: {}'.format(test_score))
    if world > 1 and torch.distributed.is_initialized():
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return test_score


if __name__ == "__main__":
    main()
