"""Shared body of the four entry points (reference: resume/*.py `catch_inner` / `pipeline`):
build the datasets, create_model, load a checkpoint when resuming, train and / or evaluate."""
import contextlib

from lirec_b200.mixed_utils import update_arg_pars as mixed_arg_update
from lirec_b200.mixed_utils.classification_dataloader import MixedFeaturesDataset
from lirec_b200.utils.arg_pars import opt
from lirec_b200.utils.util_functions import load_ema, load_model, load_optimizer
import lirec_b200.mlp.model
import lirec_b200.mlp.test
import lirec_b200.mlp.train


def released_checkpoint(path):
    """The reference's entry points set `opt.resume = True` and point `opt.resume_str` at the released
    checkpoint (resume/int_rel_ch.py:92, 117-121): they EVALUATE it.  Same here, except that an explicit
    `--resume_str` wins over the default path and `--scratch 1` (ours) turns the script into a training run
    from random init — the released checkpoints are not available offline."""
    if not opt.resume_str:
        opt.resume_str = path
    if int(getattr(opt, "scratch", 0)):
        opt.resume = False


def catch_inner():
    train_dataset = MixedFeaturesDataset(mode="train")
    train_dataset.cache()
    val_dataset = test_dataset = None
    if opt.test:
        val_dataset = MixedFeaturesDataset(mode="val")
        val_dataset.n_classes = train_dataset.n_classes
        val_dataset.cache()
        test_dataset = MixedFeaturesDataset(mode="test")
        test_dataset.n_classes = train_dataset.n_classes
        test_dataset.cache()
    if opt.rels or opt.rels_multitask:
        for d in (train_dataset, val_dataset, test_dataset):
            if d is not None:
                d.init_relships()
    n_classes = train_dataset.n_classes
    n_rels = len(train_dataset.rels_list) - 1
    model, loss, optimizer = lirec_b200.mlp.model.create_model(n_classes, n_rels=n_rels)
    ema = None
    if opt.resume or opt.resume_train:
        model.load_state_dict(load_model(name=opt.model_name))
        if opt.resume_train:
            optimizer.load_state_dict(load_optimizer())
        if opt.ema_decay:
            ema = resume_ema(model)
    if not opt.resume or opt.resume_train:
        lirec_b200.mlp.train.training(train_dataset, ema=ema, model=model, loss=loss, optimizer=optimizer,
                                      name=opt.model_name, val_dataset=val_dataset, test_dataset=test_dataset)
    out = []
    if opt.resume and opt.test:
        with ema.applied() if ema is not None else contextlib.nullcontext():
            out.append(lirec_b200.mlp.test.testing(val_dataset, model=model, loss=loss, total_iter=0, mode="val"))
            out.append(lirec_b200.mlp.test.testing(test_dataset, model=model, loss=loss, total_iter=0, mode="test"))
    return out


def resume_ema(model):
    """--ema_decay with a checkpoint (opt.resume_str) whose live weights `model` already holds: the FlatEMA to
    continue with.  --resume_train restores the checkpoint's "ema" when it has one and otherwise starts the average
    from the loaded weights; --resume (evaluate) needs the checkpoint's average and refuses one without it."""
    ema = lirec_b200.mlp.model.FlatEMA(model, opt.ema_decay)
    state = load_ema()
    if state is not None:
        ema.load_state_dict(state)
        print("restored the weight average of %s (%d updates)" % (opt.resume_str, ema.n_averaged))
    elif opt.resume_train:
        print("%s has no weight average; --ema_decay starts one from its weights (n_averaged = 0)" % opt.resume_str)
    else:
        raise RuntimeError("--resume with --ema_decay evaluates the checkpoint's weight average, but %s has none "
                           "(it was saved without --ema_decay); drop --ema_decay to evaluate its weights"
                           % opt.resume_str)
    return ema


def pipeline(name):
    mixed_arg_update.update(name)
    return catch_inner()
