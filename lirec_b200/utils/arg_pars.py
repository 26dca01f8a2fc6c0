"""General parameters: the reference's flag surface (utils/arg_pars.py:13-184), same names,
types and defaults, parsed at import into the module-global `opt`, plus the flags this
implementation adds (section "B200").

Differences on purpose: unknown command-line arguments are ignored (`parse_known_args`) so the
module can be imported under pytest / torchrun; the reference's quirks are kept (type=bool
flags treat any non-empty string as True, --tr_sum_max_flag is store_false, --sampling_fr has
an int type with a float default).
"""
import argparse

__all__ = ["opt", "build_parser"]

_ROOT = "/meleze/data1/akukleva/moviegraph"

# (flag, kwargs) in the reference's order
_FLAGS = [
    # paths
    ("--project_root", dict(default="/sequoia/data1/akukleva/projects/cvpr20")),
    ("--data_root", dict(default=_ROOT + "/files_to_release/")),
    ("--store_root", dict(default=_ROOT + "/store")),
    ("--dialogs_path", dict(default="/dialogs")),
    ("--frame2time_path", dict(default="/frame2time")),
    ("--labeled_interactions", dict(default="/others/all_train_set.txt")),
    ("--merged_interactions", dict(default="/others/merged_interactions.txt")),
    ("--annotations", dict(default="/others/mg3.pkl")),
    ("--split_path", dict(default="/others/split.json", help="json file with splits: train | val | test")),
    ("--intersected", dict(default="/intersections")),
    ("--relships2_15", dict(default="/others/relships_many2_15.txt")),
    ("--relships_opp", dict(default="/others/relships_15_opp.txt")),
    ("--merged_videos", dict(default="/others/use_vid_for_moviegraphs")),
    ("--inter_class", dict(default="m", help="t | v | m | all")),
    ("--feature_type", dict(default="m", help="m: text + visual | t | v")),
    ("--modality", dict(default="m", help="m | t | v")),
    ("--soft_gt", dict(default=False, type=bool)),
    ("--multilab_weights", dict(default=True)),
    # text
    ("--ext_dialog", dict(default="webvtt")),
    ("--text_features", dict(default="bert_base")),
    ("--contextualization", dict(default="second-to-last")),
    # visual
    ("--visual_features", dict(default="i3d")),
    ("--sampling_fr", dict(default=0.0625, type=int)),
    ("--ext_frame2time", dict(default="matidx")),
    # hyperparameters
    ("--joint_dim", dict(default=512, type=int)),
    ("--pool_features", dict(default="max", help="max | sum | mix | avg")),
    ("--i3d", dict(default="spat")),
    ("--spat_pool", dict(default=True, type=bool)),
    ("--merged", dict(default=True, type=bool)),
    # max margin loss
    ("--margin", dict(default=0.101, type=float)),
    # person tracks
    ("--ftack_ids", dict(default="/ftrack_ids")),
    ("--ftracks", dict(default="/ftracks")),
    ("--tracks", dict(action="store_true")),
    ("--tf_crop", dict(default=True, type=bool)),
    ("--orig_res", dict(default="/others/org_res.txt")),
    ("--tr_maximize", dict(action="store_true")),
    ("--tr_cat_distr", dict(action="store_true")),
    ("--tr_max_neg", dict(action="store_true")),
    ("--tr_margin", dict(default=0.101, type=float)),
    ("--tr_sum_max", dict(action="store_true")),
    ("--tr_sum_max_flag", dict(action="store_false")),
    ("--tr_correct", dict(action="store_true")),
    # relationships
    ("--rels", dict(action="store_true")),
    ("--rels_dim", dict(default=0, type=int)),
    ("--rels_dim_out", dict(default=24, type=int)),
    ("--rels_maximize", dict(default=False, type=bool)),
    ("--rels_multitask", dict(action="store_true")),
    ("--rels_multi_clip", dict(action="store_true")),
    ("--rels_n_clips", dict(default=6, type=int)),
    # gating and aggregation
    ("--lymbda", dict(default=1, type=float)),
    ("--ints", dict(default=0, type=int)),
    ("--ctx", dict(default=0, type=int)),
    ("--gates", dict(default=0, type=int)),
    ("--mid_m_ints", dict(default=6, type=int)),
    ("--mod_check", dict(action="store_true")),
    # network hyperparameters
    ("--seed", dict(default=0, type=int)),
    ("--lr", dict(default=3e-5, type=float)),
    ("--lr_int", dict(default=5, type=int)),
    ("--lr_pfx", dict(default=3, type=int)),
    ("--dropout", dict(default=0.3, type=float)),
    ("--weight_decay", dict(default=1e-5, type=float)),
    ("--epochs", dict(default=100, type=int)),
    ("--batch_size", dict(default=64, type=int)),
    ("--num_workers", dict(default=4)),
    ("--device", dict(default="cuda", help="cuda only: there is no CPU path")),
    # models
    ("--save_model", dict(default=True, type=bool)),
    ("--save_model_often", dict(default=False, type=bool)),
    ("--test", dict(default=True, type=bool)),
    ("--test_fr", dict(default=2, type=int)),
    ("--resume", dict(default=False, type=bool)),
    ("--resume_train", dict(default=False, type=bool)),
    ("--resume_str", dict(default="")),
    ("--model_name", dict(default="")),
    ("--sanity_check", dict(default=False)),
    # ---- B200: flags added by this implementation (defaults keep reference behaviour) ----
    ("--overlap_adam", dict(default=1, type=int, help="1 (single GPU, fused Adam): the Adam pass of the gate + head "
                                                      "parameters runs on a side stream while the encoder stages of "
                                                      "backward are still going (+1.2 % clips/s at 1024-clip batches, "
                                                      "+3 % at 64; bit-identical steps)")),
    ("--prefetch_factor", dict(default=2, type=int, help="batches each loader worker keeps ready")),
    ("--scratch", dict(default=0, type=int, help="1: the resume/*.py entry points train from random init instead of "
                                                 "evaluating the released checkpoint (reference behaviour)")),
    ("--dp", dict(default=0, type=int, help="1: data-parallel over clips, NCCL gradient allreduce")),
    ("--dp_switch_reduce", dict(default=1, type=int, help="1: with --dp and --fused_adam, reduce gradients inside the "
                                                          "NVSwitch fused with Adam (falls back to NCCL without multicast)")),
    ("--fused_adam", dict(default=0, type=int, help="1: flat fused Adam kernel instead of torch.optim.Adam")),
    ("--native_step", dict(default=1, type=int, help="1: forward + loss + backward of a training iteration as three "
                                                     "native calls (no autograd engine round trip); 0: the "
                                                     "reference's model()/loss()/backward() sequence")),
    ("--cache_records", dict(default=1, type=int, help="1: the index-only dataset keeps every deterministic item it has "
                                                       "built and redoes only the train-mode context subsampling per "
                                                       "access (same items, same numpy RNG stream); 0: rebuild always")),
    ("--max_n_tripl", dict(default=20, type=int, help="candidate slots per clip (reference hard-codes 20)")),
    ("--synthetic", dict(default=0, type=int, help="1: independent synthetic MovieGraphs-shaped clips; 2: synthetic "
                                                   "annotation world through the index-only dataset")),
    ("--resident_banks", dict(default=1, type=int, help="1 (default): the split's pooled feature banks stay in HBM "
                                                        "(< 1 GB for MovieGraphs) and batches ship index tables; "
                                                        "0: every batch carries its feature rows host -> device")),
    ("--loss", dict(default="margin", choices=("margin", "bce", "ce"),
                    help="margin: the reference's max-margin losses; bce: multi-label sigmoid BCE (row and track "
                         "forms; --soft_gt adds the co-occurring interactions as positives); ce: softmax "
                         "cross-entropy (row models only)")),
    ("--optimizer", dict(default="adam", choices=("adam", "lamb"),
                         help="adam: the reference's Adam (torch.optim.Adam, or the fused kernel with --fused_adam); "
                              "lamb: fused LAMB (layer-wise trust ratio, decoupled --weight_decay) for large global "
                              "batches, whatever --fused_adam says")),
    ("--clip_grad_norm", dict(default=0.0, type=float,
                              help="> 0: clip the gradient to this global L2 norm before every optimizer step, like "
                                   "torch.nn.utils.clip_grad_norm_ (fused, no host sync; with --dp, the norm of the "
                                   "averaged gradient); turns off the fused exchange + Adam and --overlap_adam. "
                                   "0: off")),
    ("--world_movies", dict(default=6, type=int)),
    ("--world_scenes", dict(default=40, type=int)),
]


def build_parser():
    parser = argparse.ArgumentParser()
    for flag, kw in _FLAGS:
        parser.add_argument(flag, **kw)
    return parser


opt = build_parser().parse_known_args()[0]
# derived dims (reference: mixed_utils/update_arg_pars.py:36-50); set here too so the model can be
# built without calling update()
opt.text_dim, opt.visual_dim, opt.track_dim = 768, 2048, 2048
opt.mlp_dim = opt.text_dim + opt.visual_dim + 2 * opt.track_dim
opt.log_prefix = ""
