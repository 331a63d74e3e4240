"""Rank candidate reactions with a checkpoint written by ``main.py``: every reactant group of the input is scored, ranked on the device and
written out with the columns of ``reactranker_b200.predict.predict`` (score, score_std, rank, p_top1, top1_freq, mean_rank, and out1 ...
for heads with more than one output), sorted by reactant group and then by rank.

    python predict.py --checkpoint runs/x/0.pt --data_path candidates.csv --out ranked.csv --gpu 0 [--mc_samples 30]
    python predict.py --checkpoint runs/x/0.pt --synthetic 40,10 --out ranked.csv     # the molecules main.py --synthetic trains on

The model arguments (--task_type, --hidden_size, --depth, --dropout) must be the ones the checkpoint was trained with; the molecule
columns (rsmi_mapped, psmi_mapped) and the extra feature (temp) are main.py's.  Real SMILES are featurised with RDKit, as in training;
--synthetic needs none.  --mc_samples T > 1 samples T dropout masks per candidate (MC dropout), seeded by --seed.
"""
import argparse

import numpy as np
import pandas as pd
import torch

from main import _MODEL_FOR_TASK, make_model
from reactranker.data.load_reactions import get_data, Parsing_features
from reactranker_b200.predict import predict
from reactranker_b200.utils import load_checkpoint


def parse(argv=None):
    ap = argparse.ArgumentParser(description="Rank candidate reactions with a trained checkpoint")
    ap.add_argument("--checkpoint", required=True, help="a checkpoint written by main.py (<path>/<fold>.pt)")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--data_path", default=None, help="CSV with rsmi, psmi, rsmi_mapped, psmi_mapped and temp columns; no target needed")
    src.add_argument("--synthetic", default=None, help="G,N: the G synthetic groups of N candidates of main.py --synthetic")
    ap.add_argument("--out", required=True, help="output CSV")
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--mc_samples", type=int, default=1, help="1: one eval-mode pass; T > 1: T dropout samples per candidate")
    ap.add_argument("--seed", type=int, default=0, help="torch.manual_seed before prediction (the MC dropout masks)")
    ap.add_argument("--task_type", default="listnet",
                    help="main.py's --task_type of the checkpoint; these keys have their own head, every other a single score: "
                         + ", ".join(sorted(_MODEL_FOR_TASK)))
    ap.add_argument("--hidden_size", type=int, default=300)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--dropout", type=float, default=0.1)
    return ap.parse_args(argv)


def main(argv=None):
    a = parse(argv)
    smiles2graph_dic = Parsing_features()
    if a.synthetic:
        from reactranker_b200 import synthetic
        G, N = (int(v) for v in a.synthetic.split(","))
        ds = synthetic.make_dataset(0, [N] * G)
        for tok, m in ds.mols.items():
            smiles2graph_dic.add(tok, m)
        data = ds.to_dataframe()
    else:
        reader = get_data(a.data_path)
        reader.read_data()
        data = reader.df
    model = make_model(a.task_type, a.hidden_size, a.depth, a.dropout)
    model.load_state_dict(load_checkpoint(a.checkpoint)['state_dict'])
    torch.cuda.set_device(a.gpu)
    model = model.cuda(a.gpu)
    torch.manual_seed(a.seed)
    ranked = predict(model, data, smiles2graph_dic, a.gpu, smiles_list=['rsmi_mapped', 'psmi_mapped'], add_features_name='temp',
                     mc_samples=a.mc_samples)
    group = pd.factorize(ranked['rsmi'])[0]                    # reactant groups in order of first appearance
    ranked.iloc[np.lexsort((ranked['rank'].values, group))].to_csv(a.out, index=False)
    print(f"{len(ranked)} candidates in {group.max() + 1 if len(group) else 0} reactant groups ranked -> {a.out}")
    return ranked


if __name__ == "__main__":
    main()
