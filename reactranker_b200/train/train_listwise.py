"""``train(...)`` for the listwise / pointwise task keys, with the reference's signature, target normalisation, loss
dispatch, optimiser stepping and per-epoch checkpointing (train/train_listwise.py:21-373).

Differences, all on purpose:
* every task key the reference can run is dispatched (``batch_loss``); only ``mle_dirichlet``, which cannot run in the reference
  either, raises ``NotImplementedError``; ``lambdarank`` / ``lambdarank_top`` are keys of this project alone;
* launched under ``torchrun`` (WORLD_SIZE > 1) the same call trains data-parallel: every rank plans the same global batches and takes
  its shard of whole reactant groups (train/step.py, parallel.py); rank 0 validates, checkpoints and prints;
* the reference copies ``encoder.W_i.weight`` to the host EVERY step to look for NaNs (train_listwise.py:190-195); here the
  check is ``torch.isfinite`` on the device, read back once per epoch together with the loss;
* ``gpu=None`` raises: there is no CPU path.
"""
from __future__ import annotations

import copy
import os
from logging import Logger
from typing import Union

import numpy as np
import torch
import torch.nn as nn
from pandas import DataFrame
from torch.optim.lr_scheduler import _LRScheduler
from tqdm import trange

from .. import _lib
from ..data.load_reactions import DataProcessor
from ..utils import load_train_state, save_checkpoint, save_train_state
from .eval import calculate_mse, ranking_metrics
from .step import TrainStep
from .loss import (Dirichlet_uq, ExpMSELoss, GaussDisLoss, LambdaRankLoss, Listnet_For_Gauss, Listnet_with_uq, ListnetLoss, Lognorm, MLEDisLoss,
                   MLEloss, MSELoss, evidential_loss_new, evidential_ranking)

try:  # only used as the default value of ``writer`` in the reference signature
    from torch.utils.tensorboard import SummaryWriter
except Exception:  # pragma: no cover
    SummaryWriter = None

BUILT_TASKS = ("mle", "listnet", "evidential_ranking", "gauss_regression",
               # sums of the terms above, dispatched exactly like train_listwise.py:204-210, 224-227, 263-266, 276-281
               "mle_gaussian", "listnet_gauss", "mle_regression", "listnet_regression", "regression_exploss",
               # distribution-valued ListMLE / ListNet (loss.py:102-141, 233-272) + the Gaussian NLL (196-203, 211-215)
               "mledis_gaussian", "listnetdis_gauss", "listnet_uq",
               # the remaining experimental keys (215-219, 229-260, 269-270)
               "listnetdis_lognorm", "dirichlet_uq", "evidential", "mle_evidential", "mledis_evidential", "listnet_evidential",
               # this project's own: LambdaRank, trained for the validation's NDCG@all / NDCG@25% (loss.LambdaRankLoss)
               "lambdarank", "lambdarank_top")
# 'mle_dirichlet' cannot run in the reference either: no branch of train_listwise.py:128-167 constructs ``dirichlet_loss`` for it and the
# call at 267-268 passes four arguments to a seven-argument forward.
UNBUILT_TASKS = ("mle_dirichlet",)


def batch_loss(task_type, output, scope, targets, gpu, max_coeff=0.0001, epoch=0, epochs=1):
    """The loss dispatch of the reference's step body (train_listwise.py:196-285) for every built key; anything else is the default
    regression (282-285).  Every term is one segmented / pointwise sm_100a kernel returning loss and dL/dscore; sums are autograd sums."""
    if task_type == 'mle':
        return MLEloss()(output, scope, targets, gpu)
    if task_type == 'listnet':
        return ListnetLoss()(output, scope, targets, gpu)
    if task_type == 'evidential_ranking':
        return evidential_ranking()(output, scope, targets, max_coeff, epoch, epochs, gpu)
    if task_type == 'gauss_regression':
        return GaussDisLoss()(output[:, 0], output[:, 1], targets, gpu)
    if task_type == 'mle_gaussian':
        return MLEloss()(output[:, 0], scope, targets, gpu) + GaussDisLoss()(output[:, 0], output[:, 1], targets, gpu)
    if task_type == 'listnet_gauss':
        return ListnetLoss()(output[:, 0], scope, targets, gpu) + GaussDisLoss()(output[:, 0], output[:, 1], targets, gpu)
    if task_type == 'mle_regression':
        return MSELoss()(output, targets) + MLEloss()(output, scope, targets, gpu)
    if task_type == 'listnet_regression':
        return ListnetLoss()(output, scope, targets, gpu) + MSELoss()(output, targets)
    if task_type == 'regression_exploss':
        return ExpMSELoss()(output, targets)
    if task_type == 'mledis_gaussian':           # the variance column is a log-variance for the ranking term (196-203)
        return (MLEDisLoss()(output[:, 0::2], torch.exp(output[:, 1::2]), scope, targets, gpu)
                + GaussDisLoss()(output[:, 0], output[:, 1], targets, gpu))
    if task_type == 'listnet_uq':                # 228-229; needs positive scores (task_type='listnet' -> softplus head)
        return Listnet_with_uq()(output, scope, targets, max_coeff, epoch, epochs, gpu)
    if task_type == 'listnetdis_gauss':          # 211-215
        return (Listnet_For_Gauss()(output[:, 0::2], output[:, 1::2], scope, targets, gpu)
                + GaussDisLoss()(output[:, 0], output[:, 1], targets, gpu))
    if task_type == 'listnetdis_lognorm':        # 215-219: the ListNet term is commented out there, the log-normal NLL is the loss
        return Lognorm()(output[:, 0], output[:, 1], targets, gpu)
    if task_type == 'dirichlet_uq':              # 269-270
        return Dirichlet_uq()(output, scope, targets, max_coeff, epoch, epochs, gpu)
    if task_type in ('evidential', 'mle_evidential', 'mledis_evidential', 'listnet_evidential'):    # 229-260
        mu, lambdas, alphas, betas = (output[:, k::4] for k in range(4))
        if task_type == 'evidential':
            return evidential_loss_new(mu, lambdas, alphas, betas, targets, gpu, lam=0.1)
        if task_type == 'mle_evidential':
            return MLEloss()(output[:, 0], scope, targets, gpu) + evidential_loss_new(mu, lambdas, alphas, betas, targets, gpu, lam=0.2)
        variance = betas / (lambdas * (alphas - 1))
        rank = MLEDisLoss() if task_type == 'mledis_evidential' else Listnet_For_Gauss()
        return rank(mu, variance, scope, targets, gpu) + evidential_loss_new(mu, lambdas, alphas, betas, targets, gpu, lam=0.1)
    if task_type in ('lambdarank', 'lambdarank_top'):    # not keys of the reference, whose fall-through below they would otherwise take
        return LambdaRankLoss(top=task_type == 'lambdarank_top')(output, scope, targets, gpu)
    return MSELoss()(output, targets)


NDCG_METRICS = ['NDCG@1', 'NDCG@2', 'NDCG@25%', 'NDCG@all']


def normalized_targets(train_col, val_col, target_name, normalize_target):
    """Target transform of train_listwise.py:66-115: for every target except ``lgk``/``lgk_bi`` the sign is flipped
    (a lower barrier is the better candidate); ``normalize_target`` may be a bool, a float scale or a ``"lo,hi"`` range."""
    mean, std = train_col.mean(), train_col.std(ddof=0)
    if target_name == 'lgk_bi':
        return train_col, val_col, mean, std
    sign = 1.0 if target_name == 'lgk' else -1.0
    lo_v, hi_v = train_col.min(), train_col.max()
    if isinstance(normalize_target, float):
        f = lambda x: sign * (x * normalize_target) / (hi_v - lo_v)  # noqa: E731
    elif isinstance(normalize_target, str):
        lo_b, hi_b = (int(v) for v in normalize_target.split(','))
        f = lambda x: sign * (x - lo_v) * (hi_b - lo_b) / (hi_v - lo_v) + lo_b  # noqa: E731
    elif normalize_target:
        f = lambda x: sign * (x - mean) / std  # noqa: E731
    else:
        f = lambda x: sign * x  # noqa: E731
    return train_col.map(f), val_col.map(f), mean, std


def train(model: nn.Module, scheduler: _LRScheduler, train_data_ini: DataFrame, val_data_ini: DataFrame, path_checkpoints: str, optimizer,
          epochs: int, smiles2graph_dic, batch_size: int, seed: int, gpu: Union[int, str], task_type: str = 'mle_gaussian',
          writer=SummaryWriter, logger: Logger = None, target_name: str = 'ea', smiles_list: list = None, save_metric=None,
          show_info=False, max_coeff=0.0001, normalize_target=True, add_features_name=None, resume_path=None):
    """``train`` of train_listwise.py:21-372 with one addition: ``resume_path`` (default None = the reference's behaviour).  When given,
    the full training state is written there after every epoch and, if the file already exists, training continues after its epoch."""
    if task_type in UNBUILT_TASKS:
        raise NotImplementedError(f"task_type '{task_type}' is one of the reference's experimental keys; built: {BUILT_TASKS} and 'regression'")
    dev_idx = _lib.require_device(gpu)
    print('Note: Set fixed seed')
    torch.manual_seed(seed)
    model = model.cuda(dev_idx)
    torch.cuda.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    step = TrainStep(model, optimizer, scheduler, task_type, dev_idx, max_coeff)      # joins torchrun's process group when WORLD_SIZE > 1
    main = step.is_main()
    if step.world > 1:
        torch.manual_seed(seed + 1000003 * step.rank)       # every rank draws its own dropout masks; the batch plan is seeded per epoch
        print('Note: data-parallel training, rank {} of {} on cuda:{}'.format(step.rank, step.world, dev_idx))

    train_data, val_data = copy.deepcopy(train_data_ini), copy.deepcopy(val_data_ini)
    score_old = float('inf') if save_metric == 'mse' else ([0, 0, 0] if save_metric == 'all' else float(0))
    data_len = train_data.shape[0] + val_data.shape[0]
    if logger is not None and main:
        logger.info('Note: the length of training and vailidate data is: {}'.format(data_len))
    print("Note: the length of training and vailidate data is", data_len)

    train_std, val_std, mean, std = normalized_targets(train_data[target_name], val_data[target_name], target_name, normalize_target)
    train_data['std' + target_name] = train_std
    val_data['std' + target_name] = val_data[target_name] if save_metric in NDCG_METRICS else val_std
    print('stds is: ', std)
    print('mean is: ', mean)

    train_proc, val_proc = DataProcessor(train_data), DataProcessor(val_data)
    finite = torch.ones((), dtype=torch.bool, device=torch.device("cuda", dev_idx))
    first_epoch = 0
    if resume_path is not None and os.path.exists(resume_path):
        first_epoch, best, _ = load_train_state(resume_path, model, optimizer, scheduler)
        score_old = best if best is not None else score_old
        print('Note: resuming after epoch {} from {}'.format(first_epoch, resume_path))
    for epoch in trange(first_epoch, epochs, disable=not main):
        lr = optimizer.state_dict()['param_groups'][0]['lr']
        if main:
            print('learning rate: ', lr)
        if logger is not None and main:
            logger.info('learning rate is: {}'.format(lr))
        model.train()
        loss = torch.zeros(1)
        # nothing below waits for the GPU (the loss is read once per epoch), so the host plans and featurises batch i+1 while step i runs
        # generate_batch_reactions(..., seed=epoch) as train_listwise.py:177-182 calls it, taken at the planner level (row positions + scope;
        # the gathered SMILES / targets of a row are looked up by whoever trains on it)
        for rows, scope in train_proc.plan_batch_reactions(batch_size=batch_size, seed=epoch):
            # the step body of train_listwise.py:187-290: targets -> FloatTensor.squeeze, featurise, forward, loss dispatch, zero_grad,
            # backward, optimizer.step, scheduler.step -- plus, data-parallel, the shard selection and the gradient all-reduce
            prepared = step.prepare_rows(train_proc, rows, scope, smiles2graph_dic, smiles_list, 'std' + target_name, add_features_name)
            loss = step.run(prepared, epoch, epochs)
            finite &= torch.isfinite(model.encoder.W_i.weight).all()
        if not bool(finite):                       # the reference prints, it does not abort (train_listwise.py:190-195)
            print('*' * 40)
            print('the mean of encoder.W_i.weight is: ', model.state_dict()['encoder.W_i.weight'])
            print('the ffn.ffn.7.weight is: ', model.state_dict().get('ffn.ffn.7.weight'))
            print('*' * 40)
        loss_value = step.global_loss(loss)        # data-parallel: the ranks' terms sum to the batch loss
        if writer is not None and not isinstance(writer, type) and main:
            writer.add_scalar('loss_every_epoch', loss_value)

        # validation, checkpoints and the epoch report are rank 0's; the other ranks receive the metrics (their `score_old` stays in step
        # for the resume state) and wait at the end of the epoch
        mse = float('nan')
        if main:
            if save_metric == 'mse':
                mse = calculate_mse(model, gpu=dev_idx, data_processor=val_proc, smiles2graph_dic=smiles2graph_dic, batch_size=batch_size,
                                    smiles_list=smiles_list, target_name='std' + target_name, add_features_name=add_features_name)
            average_score, average_pred_in_targ, average_top1_in_pred, NDCG_ = ranking_metrics(
                model, gpu=dev_idx, data_processor=val_proc, smiles2graph_dic=smiles2graph_dic, show_info=show_info, smiles_list=smiles_list,
                target_name='std' + target_name, add_features_name=add_features_name)
            metrics = [average_score, average_pred_in_targ, average_top1_in_pred] + list(NDCG_) + [mse]
        else:
            metrics = [0.0] * 8
        metrics = step.broadcast_floats(metrics)
        average_score, average_pred_in_targ, average_top1_in_pred, NDCG_, mse = metrics[0], metrics[1], metrics[2], metrics[3:7], metrics[7]

        def save(path):
            if main:
                save_checkpoint(path, model, mean, std)

        def improved(new, slot=None):
            nonlocal score_old
            old = score_old if slot is None else score_old[slot]
            if new >= old:
                if slot is None:
                    score_old = new
                else:
                    score_old[slot] = new
                return True
            return False

        if save_metric is None or save_metric == 'average_score':
            if improved(average_score):
                save(path_checkpoints)
                print('Note: the checkpint file is updated')
        elif save_metric == 'all':
            for slot, val in enumerate((average_score, average_pred_in_targ, average_top1_in_pred)):
                if improved(val, slot):
                    save(path_checkpoints[slot])
                    print('Note: the checkpint file is updated')
        elif save_metric == 'average_pred_in_targ':
            if improved(average_pred_in_targ):
                save(path_checkpoints)
        elif save_metric == 'average_top1_in_pred':
            if improved(average_top1_in_pred):
                save(path_checkpoints)
        elif save_metric in NDCG_METRICS:
            if improved(NDCG_[NDCG_METRICS.index(save_metric)]):
                save(path_checkpoints)
        elif save_metric == 'mse':                 # train_listwise.py:337-343: keep the checkpoint with the smallest validation MSE
            if mse <= score_old:
                score_old = mse
                save(path_checkpoints)
        else:
            raise Exception('Unknown save metric')

        if writer is not None and not isinstance(writer, type) and main:
            writer.add_scalar("average_score", average_score)
        msg = 'Epoch [{}/{}], train_loss,{:.4f}, top1,{:.4f}, top1_in_pred_top25%,{:.4f}, pred_top25%_in_targ_top25%,{:.4f}'.format(
            epoch + 1, epochs, loss_value, average_score, average_top1_in_pred, average_pred_in_targ)
        if logger is not None and main:
            logger.info(msg)
        if main:
            print('Epoch [{}/{}], average score: {:.4f}'.format(epoch + 1, epochs, average_score))
            print('Epoch [{}/{}], targ_top1_in_pred_top25%: {:.4f}'.format(epoch + 1, epochs, average_top1_in_pred))
            print('Epoch [{}/{}], pred_top25%_in_targ_top25%: {:.4f}'.format(epoch + 1, epochs, average_pred_in_targ))
            print('Epoch [{}/{}], train loss: {:.4f}'.format(epoch + 1, epochs, loss_value))
            print('Epoch [{}/{}], last batch loss, full precision = {!r}'.format(epoch + 1, epochs, loss_value))
            if save_metric in NDCG_METRICS:
                print('Epoch [{}/{}], NDCG: {}'.format(epoch + 1, epochs, NDCG_))
        if resume_path is not None and main:
            save_train_state(resume_path, model, optimizer, scheduler, epoch, mean, std, best=score_old)
        step.barrier()                             # the state file / checkpoints are complete before any rank moves on
