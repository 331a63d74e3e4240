"""Listwise / pointwise training entry point -- the flow, variable names and defaults of the reference's ``main.py``
(main.py:15-174), with its edit-the-constants placeholders (``user_defined``, ``your_gpu``, the two paths) turned into
command-line arguments.  ``--synthetic G,N`` trains on G synthetic reactant groups of N candidates instead of a CSV
(no RDKit needed): the plumbing case of BASELINE.json configs[0].

    python main.py --data_path reactions.csv --path runs/exp1 --gpu 0 --task_type listnet --batch_size 4096 --total_epochs 30
    python main.py --synthetic 100,20 --path /tmp/rr --gpu 0 --task_type mle --batch_size 100 --total_epochs 2

Fine-tuning (new): start from a pretrained checkpoint and keep sub-modules fixed; frozen layers cost no backward work,

    python main.py --data_path small.csv --path runs/ft --pretrained runs/exp1/T1/0.pt --freeze encoder,diff_encoder --total_epochs 30

Data-parallel over the GPUs of one box (new; the reference is single-device): launch the same command under torchrun,

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 main.py --data_path ... --batch_size 32768

``--batch_size`` stays the GLOBAL batch; every rank plans the same batches and trains on its shard of whole reactant groups on
cuda:LOCAL_RANK (train/step.py).  Rank 0 validates, writes the checkpoints and runs the final test.
"""
import argparse
import logging
import os

import numpy as np
import pandas as pd
import torch

from reactranker.data.load_reactions import get_data, Parsing_features
from reactranker.train.utils import build_optimizer, build_lr_scheduler
from reactranker.models.base_model import build_model
from reactranker_b200.models.base_model import freeze, parse_freeze
from reactranker_b200.utils import load_pretrained
from reactranker.train.train_listwise import train
from reactranker.train.test_listwise import test


# (task_num, build_model task_type, ffn_last_layer) for every key whose loss does not read a single raw / softplus score.  The reference has
# the user edit main.py:114-123 for these; the rows follow what each branch of train_listwise.py:196-285 indexes.
_TWO = (2, None, 'with_softplus')            # -> 'gaussian_with_softplus': (mu, softplus)
_FOUR = (4, None, 'with_softplus')           # -> 'evidential_with_softplus': the NIG head
_MODEL_FOR_TASK = {
    'evidential_ranking': (2, 'evidential_ranking', 'with_softplus'),
    'gauss_regression': _TWO, 'mle_gaussian': _TWO, 'listnet_gauss': _TWO, 'mledis_gaussian': _TWO, 'listnetdis_gauss': _TWO,
    'listnetdis_lognorm': (2, 'listnetdis_lognorm', 'with_softplus'),
    'evidential': _FOUR, 'mle_evidential': _FOUR, 'mledis_evidential': _FOUR, 'listnet_evidential': _FOUR,
    'listnet_uq': (1, 'listnet', 'with_softplus'),               # positive scores
    'dirichlet_uq': (1, 'listnet', 'with_uncertainty'),          # concentrations > 1
}


def make_model(task_type, hidden_size, depth, dropout):
    """The ReactionModel main.py trains for ``task_type`` (predict.py rebuilds it to load a checkpoint)."""
    task_num, model_task, last_layer = _MODEL_FOR_TASK.get(task_type, (1, None, 'with_softplus'))
    return build_model(hidden_size=hidden_size, mpnn_depth=depth, mpnn_diff_depth=depth, ffn_depth=3, use_bias=True, dropout=dropout,
                       task_num=task_num, ffn_last_layer=last_layer, task_type=model_task, add_features_dim=1)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--path", default="runs/reactranker", help="save path (checkpoints, output.log)")
    ap.add_argument("--data_path", default=None)
    ap.add_argument("--val_data_path", default=None)
    ap.add_argument("--test_data_path", default=None)
    ap.add_argument("--synthetic", default=None, help="G,N: G synthetic groups of N candidates")
    ap.add_argument("--filtered_size", type=int, default=3)
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--k_fold", type=int, default=1)
    ap.add_argument("--batch_size", type=int, default=4096)
    ap.add_argument("--total_epochs", type=int, default=30)
    ap.add_argument("--task_type", default="listnet")
    ap.add_argument("--target_name", default="lgk")
    ap.add_argument("--split_strategy", default="random_flag", choices=["random", "scaffold", "random_flag"])
    ap.add_argument("--init_lr", type=float, default=1e-4)
    ap.add_argument("--max_lr", type=float, default=1e-3)
    ap.add_argument("--final_lr", type=float, default=1e-4)
    ap.add_argument("--save_metric", default="all")
    ap.add_argument("--resume", action="store_true", help="write <path>/<fold>.state.pt after every epoch and continue from it if present")
    ap.add_argument("--stop_after", type=int, default=None, help="stop after this many epochs (the schedule still spans --total_epochs)")
    ap.add_argument("--hidden_size", type=int, default=300)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--deterministic", action="store_true",
                    help="torch.use_deterministic_algorithms(True): bit-identical losses, gradients and weights from the same seed")
    add_finetune_args(ap)
    return check_finetune_args(ap, ap.parse_args())


def add_finetune_args(ap):
    """--pretrained / --freeze, shared with main_ranknet.py."""
    ap.add_argument("--pretrained", default=None,
                    help="checkpoint to start from: every state_dict tensor whose name and shape match is copied (utils.load_pretrained)")
    ap.add_argument("--freeze", type=_freeze_arg, default=None, metavar="encoder[,diff_encoder][,ffn:N]",
                    help="keep these pretrained sub-modules fixed (ffn:N = the first N FFN layers); needs --pretrained")


def _freeze_arg(spec):
    try:
        return parse_freeze(spec)
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e))


def check_finetune_args(ap, a):
    if a.freeze is not None and a.pretrained is None:
        ap.error("--freeze needs --pretrained: freezing randomly initialised weights is always a mistake")
    return a


def apply_finetune_args(a, model, logger):
    """--pretrained, then --freeze, on a freshly built model (before .cuda()); returns whether anything is frozen."""
    if a.pretrained is not None:
        skipped = load_pretrained(model, a.pretrained)
        logger.info('Loaded {} tensors from {}; not loaded: {}'.format(len(model.pretrained_names), a.pretrained, skipped))
    if a.freeze is None:
        return False
    frozen = freeze(model, **a.freeze)
    logger.info('Frozen tensors: {}'.format(frozen))
    return True


def main():
    a = parse()
    if a.deterministic:
        torch.use_deterministic_algorithms(True)
    from reactranker_b200 import parallel
    rank, world, local_rank = parallel.world_from_env()
    if world > 1:
        a.gpu = local_rank                      # one process per GPU
    path, data_path, val_data_path, test_data_path = a.path, a.data_path, a.val_data_path, a.test_data_path
    os.makedirs(path, exist_ok=True)
    logging.basicConfig(filename=path + ('/output.log' if rank == 0 else '/output.rank{}.log'.format(rank)), level=logging.INFO,
                        format='%(asctime)s - %(message)s', datefmt='%d-%b-%y %H:%M:%S')
    logger = logging.getLogger()
    writer = None
    if rank == 0:
        try:
            from torch.utils.tensorboard import SummaryWriter
            writer = SummaryWriter(path + '/loss_writer')
        except Exception:
            writer = None
    filtered_size = a.filtered_size
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
        data = get_data(data_path)
        data.read_data()
    data.filter_bacth(filter_szie=filtered_size)
    gpu = a.gpu
    test_score = []

    k_fold, batch_size, total_epochs = a.k_fold, a.batch_size, a.total_epochs
    task_type = a.task_type          # to choose loss function
    target_name = a.target_name
    smiles_list = ['rsmi_mapped', 'psmi_mapped']
    split_strategy = a.split_strategy
    init_lr, max_lr, final_lr = a.init_lr, a.max_lr, a.final_lr
    save_metric = a.save_metric
    add_features_name = 'temp'
    logger.info('Task type is: {}, and target name is: {}'.format(task_type, target_name))
    logger.info('{} fold train with {} epochs every fold. The batch size is: {}'.format(k_fold, total_epochs, batch_size))

    if save_metric == 'all':
        metric_list = ["T1", "T25_in_T25", "T25"]
        path = [os.path.join(path, i) for i in metric_list]
        for p in path:
            os.makedirs(p, exist_ok=True)
    # evidential_ranking / gauss_regression need two outputs; main.py's default build (task_num=1, task_type commented out,
    # main.py:114-123) serves mle / listnet / regression
    # The experimental keys need the head their loss reads (base_model.py:252-264 resolves task_num / task_type / ffn_last_layer to it):
    # make_model looks it up in _MODEL_FOR_TASK.
    for ii in range(k_fold):
        print('**********************************')
        print('**   This is the fold [{}/{}]   **'.format(ii + 1, k_fold))
        print('**********************************')
        seed = ii
        k_fold_str = str(ii) + '.pt'
        path_checkpoints = os.path.join(path, k_fold_str) if save_metric != 'all' else [os.path.join(i, k_fold_str) for i in path]
        if val_data_path is not None and test_data_path is not None:
            train_data, val_data, test_data = pd.read_csv(data_path), pd.read_csv(val_data_path), pd.read_csv(test_data_path)
        elif split_strategy == 'random':
            train_data, val_data, test_data = data.split_data(split_size=(0.8, 0.1, 0.1), split_type='reactants', seed=seed)
        elif split_strategy == 'scaffold':
            train_data, val_data, test_data = data.scaffold_split_data(split_size=(0.8, 0.1, 0.1), balanced=True, seed=seed)
        else:
            train_data, val_data, test_data = data.split_data(split_size=(0.8, 0.1, 0.1), split_type='flag', seed=seed)
        train_len = train_data.shape[0]
        torch.manual_seed(seed)
        torch.cuda.manual_seed(seed)
        torch.cuda.manual_seed_all(seed)
        model = make_model(task_type, a.hidden_size, a.depth, a.dropout)
        logger.info('Model Structure')
        logger.info(model)
        frozen = apply_finetune_args(a, model, logger)
        torch.cuda.set_device(gpu)
        model = model.cuda(gpu)
        optimizer = build_optimizer(model, freeze=frozen)
        scheduler = build_lr_scheduler(optimizer, warmup_epochs=2, total_epochs=total_epochs, train_data_size=train_len, batch_size=batch_size,
                                       init_lr=init_lr, max_lr=max_lr, final_lr=final_lr)
        resume_path = os.path.join(a.path, str(ii) + '.state.pt') if a.resume else None
        train(model, scheduler, train_data, val_data, path_checkpoints, optimizer, a.stop_after or total_epochs, smiles2graph_dic,
              batch_size=batch_size, seed=seed, gpu=gpu, task_type=task_type, writer=writer, logger=logger, target_name=target_name,
              smiles_list=smiles_list, save_metric=save_metric, add_features_name=add_features_name, resume_path=resume_path)
        if rank != 0:                           # rank 0 tests; train() ended with a barrier, so its checkpoints are on disk
            continue
        print(path_checkpoints)
        test_path = path_checkpoints[0] if save_metric == 'all' else path_checkpoints
        score, average_pred_in_targ, score3 = test(model, test_data, test_path, batch_size, smiles2graph_dic, gpu=gpu, smiles_list=smiles_list,
                                                   logger=logger, target_name=target_name, cal_ngcd=False, return_order=False,
                                                   add_features_name=add_features_name)
        test_score.append([score, average_pred_in_targ, score3])
    if rank == 0:
        print("test score for k_fold vailidation is: ", test_score)
        logger.info('test score for k_fold vailidation is: {}'.format(test_score))
    if world > 1 and torch.distributed.is_initialized():
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return test_score


if __name__ == "__main__":
    main()
