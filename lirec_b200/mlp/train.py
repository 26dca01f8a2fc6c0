"""Training loop (reference: mlp/train.py:21-107): epochs over the dataset, forward, loss,
zero_grad, backward, Adam step, periodic evaluation and checkpoints in the reference's format.

Differences on purpose: batches are PackedBatches prefetched to the GPU asynchronously; the loss
value is read back every 10 iterations instead of every step (mlp/train.py:59 syncs each step);
with `opt.dp` the clips of every global batch are split over the ranks and the flat gradient buffer
is all-reduced over NCCL before the optimizer step (lirec_b200/dp.py); with --clip_grad_norm the
reduced gradient is clipped to that global L2 norm before the step.  Batches of a single clip
are skipped like the reference does (:55-56)."""
import copy
import time
from datetime import datetime
from os.path import join

import torch

from lirec_b200 import dp
from lirec_b200.mixed_utils.classification_dataloader import packed_loader
from lirec_b200.mlp.model import _FusedLoss, _HotPath, dp_empty_shard_collectives
from lirec_b200.mlp.model import train_step as native_train_step
from lirec_b200.mlp.test import testing
from lirec_b200.utils.arg_pars import opt
from lirec_b200.utils.model_saver import ModelSaver
from lirec_b200.utils.util_functions import Averaging, dir_check


def train_step(model, loss, optimizer, pb, world=1, fused=None, max_norm=0.0):
    """One optimisation step on a device PackedBatch; returns the (device) loss tensor.  `fused`: the
    in-switch reduce+Adam of dp.SwitchReduceAdam.attach (None: NCCL all_reduce, then the optimizer).
    max_norm > 0 (--clip_grad_norm): the reduced gradient is clipped to that global L2 norm before the
    optimizer step (dp.reduce_and_step; needs fused=None); the pre-clip norm stays on the device as
    model._last_grad_norm.
    With lirec_b200's own model and loss the forward, loss and backward run as three native calls
    without the autograd engine (`mlp.model.train_step`, `--native_step 1`, the default); any other
    combination takes the reference's four-call sequence (mlp/train.py:57-63)."""
    if pb.B == 0:
        # EmptyShard: this rank has no clip of a global batch smaller than the world; it contributes a zero
        # gradient with weight 0 but takes part in the exchange, so every rank runs the same collectives
        model._sync_flat()
        model._flat_grad.zero_()
        loss._dp_world = world
        dp_empty_shard_collectives(loss, model._flat.device)
        loss._dp_world = 1
        dp.reduce_and_step(model, optimizer, fused, 0, pb.global_clips, max_norm)
        return model._flat_grad.new_zeros(())
    loss._dp_world = world                       # multi-task losses normalise their relationship term globally
    if fused is not None:                        # bucket 0 of the exchange / Adam overlaps the rest of backward
        gc = getattr(pb.host, "global_clips", None) if getattr(pb, "host", None) is not None else None
        fused.arm(equal_shards=(world == 1 or gc is None or pb.B * world == gc))
    if int(getattr(opt, "native_step", 1)) and isinstance(model, _HotPath) and isinstance(loss, _FusedLoss):
        loss_values = native_train_step(model, loss, pb)
    else:
        output = model(pb)
        loss_values = loss(output, {})
        optimizer.zero_grad()
        loss_values.backward()
    local = global_clips = None
    if world > 1:
        local = pb.B
        global_clips = getattr(pb.host, "global_clips", None) if getattr(pb, "host", None) is not None else None
    loss._dp_world = 1                           # evaluation (mlp/test.py) runs the losses without collectives
    dp.reduce_and_step(model, optimizer, fused, local, global_clips, max_norm)
    return loss_values


def training(train_dataset, **kwargs):
    train_start_time = datetime.now().strftime("%Y%m%d-%H%M%S")
    print("set parameters and model, train start time: %s" % train_start_time)
    model, loss, optimizer = kwargs["model"], kwargs["loss"], kwargs["optimizer"]
    rank, world, fused = 0, 1, None
    # --clip_grad_norm: the fused exchange + Adam and the overlapped gate + head Adam pass both update parameters
    # before the global norm exists, so clipping takes NCCL all_reduce (with --dp) and the optimizer's own step
    max_norm = float(getattr(opt, "clip_grad_norm", 0.0) or 0.0)
    if getattr(opt, "dp", 0):
        rank, world, _ = dp.init_from_env()
        model._sync_flat()
        dp.broadcast_params(model._flat)
        model.set_rank(rank)                               # dropout / sampled-assignment streams differ per rank
        if hasattr(loss, "set_rank"):
            loss.set_rank(rank)
        if int(getattr(opt, "dp_switch_reduce", 1)) and not max_norm:
            fused = dp.SwitchReduceAdam.attach(model, optimizer)     # None without NVSwitch multicast / FlatAdam
    if fused is None and world == 1 and int(getattr(opt, "overlap_adam", 0)) and not max_norm:
        fused = dp.SwitchReduceAdam.attach(model, optimizer, single_gpu=True)    # None unless FlatAdam
    batch_time, data_time, losses = Averaging(), Averaging(), Averaging()
    grad_norm = float("nan")
    print("epochs: %s", opt.epochs)
    model_saver_val = ModelSaver(path=opt.store_root)
    dev = torch.device("cuda", torch.cuda.current_device())
    epoch = 0
    # The dataset's records are a few million long-lived Python objects: parked in the permanent generation, a
    # full collection no longer walks them in the middle of an epoch (tens of milliseconds = a dozen 64-clip steps
    # during which the launch thread holds the GIL and the GPU drains its queue).
    import gc
    gc.collect()
    gc.freeze()
    for epoch in range(opt.epochs):
        model.to(opt.device)
        model.train()
        train_dataset.epoch = epoch
        print("Epoch # %d" % epoch)
        end = time.time()
        counter = 0
        if opt.tr_sum_max and epoch == 20:
            opt.tr_sum_max_flag = True                      # reference: :49-51
        n_batches = (len(train_dataset) + opt.batch_size - 1) // opt.batch_size
        for i, pb in enumerate(packed_loader(train_dataset, opt.batch_size, shuffle=True,
                                             num_workers=opt.num_workers, device=dev, rank=rank, world=world,
                                             seed=opt.seed)):
            data_time.update(time.time() - end)
            if getattr(pb.host, "global_clips", pb.B) == 1:
                continue
            loss_values = train_step(model, loss, optimizer, pb, world, fused, max_norm)
            counter += pb.B
            if i % 10 == 0 and pb.B:
                if max_norm:                                 # the loss and the last pre-clip norm in one read-back
                    lv, grad_norm = torch.stack([loss_values.detach().float().reshape(()),
                                                 model._last_grad_norm]).tolist()
                else:
                    lv = loss_values.item()
                losses.update(lv, pb.B)                      # device->host sync only here
            batch_time.update(time.time() - end)
            end = time.time()
            if i % 10 == 0 and i and rank == 0:
                print("Epoch: [{0}][{1}/{2}]\tTime {bt.val:.3f} ({bt.avg:.3f})\tData {dt.val:.3f} ({dt.avg:.3f})\t"
                      "Loss {loss.val:.4f} ({loss.avg:.4f})\t".format(epoch, i, n_batches, bt=batch_time,
                                                                       dt=data_time, loss=losses)
                      + ("Grad norm {:.4f}\t".format(grad_norm) if max_norm else ""))
        print(counter)
        print("loss: %f" % losses.avg)
        losses.reset()
        if epoch % opt.test_fr == 0:
            testing(train_dataset, model, loss, total_iter=epoch, mode="train", train_start_time=train_start_time)
            if opt.test and kwargs.get("val_dataset", kwargs.get("test_dataset")) is not None:
                val_dataset = kwargs.get("val_dataset", kwargs.get("test_dataset"))
                check_val = testing(val_dataset, model, loss, total_iter=epoch, train_start_time=train_start_time,
                                    mode="val")
                # every rank keeps the same book (the metrics are reduced over ranks), rank 0 alone the payloads
                model_saver_val_hit = model_saver_val.check(check_val)
                if model_saver_val_hit:
                    save_dict = None
                    if rank == 0:
                        save_dict = {"epoch": epoch, "state_dict": copy.deepcopy(model.state_dict()),
                                     "optimizer": copy.deepcopy(optimizer.state_dict().copy())}
                    model_saver_val.update(check_val, save_dict, epoch)
                if model_saver_val_hit and kwargs.get("test_dataset") is not None and \
                        kwargs.get("test_dataset") is not val_dataset:
                    testing(kwargs["test_dataset"], model, loss, total_iter=epoch,     # reference :91-92
                            train_start_time=train_start_time, mode="test")
            print(opt.log_prefix)
        if opt.save_model and opt.save_model_often and epoch % 30 == 0 and rank == 0:
            model_saver_val.save()
    check_str = join(opt.store_root)
    opt.resume_str = join(check_str, "%d.pth.tar" % epoch)
    if opt.save_model and rank == 0:
        save_dict = {"epoch": epoch, "state_dict": model.state_dict(), "optimizer": optimizer.state_dict()}
        dir_check(check_str)
        torch.save(save_dict, opt.resume_str)
    return model
