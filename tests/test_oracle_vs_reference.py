"""lirec_b200's models against the UNMODIFIED reference's initial parameters, stored with the golden cases
(tests/golden/*.npz, `p_*` arrays): tests/golden/make_golden.py builds every case's model with the reference's
own create_model under torch.manual_seed(<position of the case in its CASES list>), at the reduced dims below."""
import ast
import glob
import os

import numpy as np
import torch

GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz"))
                if not os.path.basename(p).startswith(("dataloader_", "pooling_", "eval_")))
DIMS = dict(text_dim=24, visual_dim=40, track_dim=40, joint_dim=16, mid_m_ints=6)
C, R = 11, 5
# make_golden.py's CASES, in order: a case's position is the torch seed its model was built under
CASE_SEEDS = {stem: seed for seed, stem in enumerate((
    "modalities", "modalities_modality-t_tracks-False", "modalities_modality-v_tracks-False", "modalities_tracks-False",
    "int_rels", "int_ch", "int_ch_tr_correct", "int_ch_tr_max_neg", "int_rel_ch", "int_rel_ch_tr_correct",
    "int_rel_ch_tr_max_neg", "int_rel_ch_tr_correct_tr_max_neg", "modalities_train", "int_rels_train", "int_ch_train",
    "int_rel_ch_train", "int_rels_gates-0_ints-0", "int_rels_gates-0_ints-0_train"))}


def test_same_seed_gives_the_reference_initial_weights(opt_preset):
    """lirec_b200's modules are constructed in the reference's order, so torch.manual_seed(s) yields
    bit-identical initial parameters, for every model class and flag combination of the golden cases (checked on
    CPU: construction does not need the GPU)."""
    import lirec_b200.mlp.model as M
    assert sorted(os.path.basename(p)[:-4] for p in GOLDEN) == sorted(CASE_SEEDS)
    for path in GOLDEN:
        stem = os.path.basename(path)[:-4]
        z = np.load(path)
        preset, over = str(z["meta"][0]), dict(ast.literal_eval(str(z["meta"][1])))
        over.pop("train", None)
        opt_preset(preset, **DIMS, **over)
        torch.manual_seed(CASE_SEEDS[stem])
        if preset == "modalities":
            # create_model (reference mlp/model.py:578-609) builds a MidFusionMultiClip first and replaces it with
            # Modalities when opt.mod_check is set: the first model's draws come before Modalities' own
            M.MidFusionMultiClip(C, R)
            model = M.Modalities(C)
        elif preset == "int_rels":
            model = M.MidFusionMultiClip(C, R)
        else:
            model = M.MidFusionMultiClipMaxTracks(C, R)
        ours = model.state_dict()
        ref = {k[2:]: z[k] for k in z.files if k.startswith("p_")}
        assert list(ours) == list(ref), stem
        for k in ref:
            assert torch.equal(ours[k], torch.from_numpy(ref[k])), (stem, k)
