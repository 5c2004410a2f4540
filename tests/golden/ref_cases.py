"""Case tables shared by the golden generators (which run the REFERENCE builders on keras_shim or on the recording
keras) and the tests that check the oracle and the product against the fixtures they wrote."""

RECEPTION_CASES = {
    # case: (input shape, reception.build kwargs, weight seed, input seed[, frames])
    'reception2d_ctx': ((64, 64, 3), dict(num_joints=16, dim=2, num_blocks=2, ksize=(5, 5), num_context_per_joint=2,
                                          concat_pose_confidence=False), 1234, 1),
    'reception2d_heatmaps': ((64, 64, 3), dict(num_joints=16, dim=2, num_blocks=2, ksize=(3, 3), export_heatmaps=True), 7, 22),
    'reception3d': ((64, 64, 3), dict(num_joints=17, dim=3, num_blocks=2, ksize=(5, 5), concat_pose_confidence=False), 1234, 23),
    # the BASELINE.json configs[1] model at full size (eval_penn_ar_pe_merge.py:51-53 / eval_mpii_singleperson.py:47), 1 frame
    'reception2d_c1_fullsize': ((256, 256, 3), dict(num_joints=16, dim=2, num_blocks=8, ksize=(5, 5), num_context_per_joint=2,
                                                    concat_pose_confidence=False), 1234, 31, 1),
}

# full-size BASELINE configs, inputs regenerated from their seed (the fixture stores seed + checksum, not the frames)
RECEPTION_CASES.update({
    # configs[2]: exp/h36m/eval_h36m.py:42-48 -- 3-D pose, 17 joints, 8 blocks, 256x256
    'reception3d_c3_fullsize': ((256, 256, 3), dict(num_joints=17, dim=3, num_blocks=8, ksize=(5, 5),
                                                    concat_pose_confidence=False), 1234, 41, 1),
    # configs[0]/[1] with every block's heat-maps exported: arg-max pixels of all 8 heads
    'reception2d_c1_heatmaps': ((256, 256, 3), dict(num_joints=16, dim=2, num_blocks=8, ksize=(5, 5), num_context_per_joint=2,
                                                    concat_pose_confidence=False, export_heatmaps=True), 1234, 43, 1),
})
LARGE_INPUT_CASES = ('reception3d_c3_fullsize', 'reception2d_c1_heatmaps', 'spnet_penn_c4_t16', 'spnet_ntu_c5_t16')

SPNET_CASES = {
    # case: (cfg input shape, pose layout name, ModelConfig kwargs, weight seed, batch)
    'spnet_penn_like': ((2, 128, 128, 3), 'pa16j2d',
                        dict(num_actions=[15], num_pyramids=2, action_pyramids=[1, 2], num_levels=4, pose_replica=True,
                             num_pose_features=160, num_visual_features=160), 1234, 1),
    'spnet_ntu_like': ((2, 128, 128, 3), 'pa17j3d',
                       dict(num_actions=[60], num_pyramids=2, action_pyramids=[1, 2], num_levels=4, num_pose_features=192,
                            num_visual_features=192), 1234, 1),
    'spnet_pose_only': ((128, 128, 3), 'pa16j2d', dict(num_pyramids=2, action_pyramids=[], num_levels=4), 5, 2),
    # the BASELINE.json configs[3] architecture (exp/pennaction/eval_penn_multitask.py:37-40) at full resolution; the clip
    # is cut to 2 frames (the clip length only sets the temporal extent of the action head's input)
    'spnet_penn_c4_t2': ((2, 256, 256, 3), 'pa16j2d',
                         dict(num_actions=[15], num_pyramids=6, action_pyramids=[5, 6], num_levels=4, pose_replica=True,
                              num_pose_features=160, num_visual_features=160), 1234, 1),
}

# full clips: x = default_rng(seed_x).uniform(-1, 1, (batch,) + shape) (own generator per case)
SPNET_FULL_CASES = {
    # case: (cfg input shape, pose layout, ModelConfig kwargs, weight seed, batch, input seed)
    # configs[3] (exp/pennaction/eval_penn_multitask.py:37-40 with 8 -> 16 frames): time_stride = 2 in the action head
    'spnet_penn_c4_t16': ((16, 256, 256, 3), 'pa16j2d',
                          dict(num_actions=[15], num_pyramids=6, action_pyramids=[5, 6], num_levels=4, pose_replica=True,
                               num_pose_features=160, num_visual_features=160), 1234, 1, 101),
    # configs[4] (exp/ntu/eval_ntu_multitask.py:35-38 with 8 -> 16 frames), 3-D poses, 60 actions
    'spnet_ntu_c5_t16': ((16, 256, 256, 3), 'pa17j3d',
                         dict(num_actions=[60], num_pyramids=2, action_pyramids=[1, 2], num_levels=4, num_pose_features=192,
                              num_visual_features=192), 1234, 1, 102),
}

# CVPR'18 merge model (exp/pennaction/eval_penn_ar_pe_merge.py:42-62), small geometry
def positive_last_regmap(table, num_blocks):
    """Weight hook of the merge-model cases: |kernel| for the LAST RegMap conv.  Its input is ReLU(x) >= 0, so the
    heat-maps and with them the raw joint confidences are >= 0 and the context aggregation's division by
    sum(pc) (blocks.py:264-267) is perfectly conditioned for every joint -- the action outputs, which consume ALL
    joints' poses, can then be held to the 1e-3 bar instead of being bounded by the worst joint's cancellation."""
    import numpy as np
    out = dict(table)
    for name in table:
        if name.startswith('RegMap%d/' % num_blocks) and name.endswith('/kernel'):
            out[name] = np.abs(table[name])
    return out


MERGE_CASE = dict(input_shape=(64, 64, 3), num_frames=4, num_actions=15, num_joints=16, num_blocks=4, seed=3,
                  reception=dict(num_joints=16, dim=2, num_blocks=4, num_context_per_joint=2, ksize=(5, 5)))

# the 3-D variant of the merge model (action.py:208-297 via build_merge_model(pose_dim=3)); 20 joints (pa20j3d):
# the PoseAR net pools and re-upsamples the joint axis, which only closes for joint counts divisible by 4
MERGE3D_CASE = dict(input_shape=(64, 64, 3), num_frames=4, num_actions=15, num_joints=20, num_blocks=2, depth_maps=8, seed=9,
                    reception=dict(num_joints=20, dim=3, num_blocks=2, depth_maps=8, ksize=(5, 5)))


# builder arguments the BASELINE configs do not use, recorded on the recording keras (reference_dropin/
# run_reference_backbone.py sweep -> ref_dropin_models.json.gz; tests/test_keras_compat.py): reception.build at 128x128 ...
RECORDED_SWEEP_RECEPTION = (
    dict(dim=2, num_context_per_joint=None, num_blocks=1, ksize=(3, 3)),
    dict(dim=2, num_context_per_joint=1, num_blocks=2, ksize=(5, 5), export_heatmaps=True),
    dict(dim=2, num_context_per_joint=2, num_blocks=2, ksize=(3, 3), concat_pose_confidence=False, alpha=0.5,
         export_vfeat_block=1),
    dict(dim=3, depth_maps=8, num_blocks=2, ksize=(3, 3)),
    dict(dim=3, num_blocks=1, ksize=(5, 5), export_heatmaps=True),         # refused by both
    dict(dim=4, num_blocks=1))                                             # the reference's own ValueError
# ... and spnet.build: (input shape, pose layout, ModelConfig kwargs over SWEEP_SPNET_BASE)
SWEEP_SPNET_BASE = dict(num_pyramids=2, num_levels=4, num_actions=[15], action_pyramids=[1, 2])
RECORDED_SWEEP_SPNET = (
    ((128, 128, 3), 'pa16j2d', dict(num_actions=[], action_pyramids=[], num_levels=3)),
    ((128, 128, 3), 'pa17j3d', dict(num_actions=[], action_pyramids=[], predict_rootz=True, growth=64)),
    ((4, 128, 128, 3), 'pa16j2d', dict(pose_replica=True, kernel_size=(3, 3))),
    ((4, 128, 128, 3), 'pa20j3d', dict(num_actions=[15, 60], sam_alpha=2)),
    ((16, 128, 128, 3), 'pa17j3d', dict(action_pyramids=[2], image_div=4)),
    ((16, 128, 128, 3), 'pa16j2d', dict(num_pyramids=3, action_pyramids=[1, 3], num_pose_features=160,
                                        num_visual_features=96)),
    ((4, 128, 128, 3), 'pa16j2d', dict(downsampling_type='conv')))         # transposed conv: refused by both

# the same kind of options executed numerically on keras_shim (make_option_sweep_golden.py -> ref_option_sweep.npz;
# tests/test_reference_golden.py): reception.build at 64x64 on 2 frames, spnet.build on one item; inputs are drawn in
# this order from one default_rng(OPTION_SWEEP_INPUT_SEED), weights are the product's synthetic ones (seed 1234)
OPTION_SWEEP_INPUT_SEED = 2020
OPTION_SWEEP_RECEPTION = RECORDED_SWEEP_RECEPTION[:4]
OPTION_SWEEP_SPNET = (
    ((128, 128, 3), 'pa16j2d', dict(num_actions=[], action_pyramids=[], num_levels=3)),
    ((128, 128, 3), 'pa17j3d', dict(num_actions=[], action_pyramids=[], predict_rootz=True, growth=64)),
    ((4, 128, 128, 3), 'pa16j2d', dict(pose_replica=True, kernel_size=(3, 3))),
    ((4, 128, 128, 3), 'pa20j3d', dict(num_actions=[15, 60], sam_alpha=2)),
    ((8, 128, 128, 3), 'pa17j3d', dict(action_pyramids=[2], image_div=4)),
    ((4, 128, 128, 3), 'pa16j2d', dict(num_pyramids=3, action_pyramids=[1, 3], num_pose_features=160,
                                       num_visual_features=96)))


def option_sweep_inputs():
    """[(kind, build kwargs / (shape, layout, kwargs), x float64)] of the numeric option sweep, in drawing order."""
    import numpy as np
    rng = np.random.default_rng(OPTION_SWEEP_INPUT_SEED)
    out = [('reception', kw, rng.uniform(-1, 1, (2, 64, 64, 3))) for kw in OPTION_SWEEP_RECEPTION]
    for shape, layout, extra in OPTION_SWEEP_SPNET:
        kw = dict(SWEEP_SPNET_BASE)
        kw.update(extra)
        out.append(('spnet', (shape, layout, kw), rng.uniform(-1, 1, (1,) + shape)))
    return out


OPTION_SWEEP_SAMPLE = 4096      # outputs with more elements are stored as this many values at fixed positions


def option_sweep_sample_index(size):
    """Positions (in the flattened output) of the values ref_option_sweep.npz keeps of a large output."""
    import numpy as np
    return np.sort(np.random.default_rng(0).choice(size, OPTION_SWEEP_SAMPLE, replace=False))


def option_sweep_store(blob, key, out):
    """Output `key` of the option sweep into `blob`: whole, or its shape and a fixed sample of its values."""
    import numpy as np
    out = np.asarray(out, dtype=np.float64)
    if out.size <= OPTION_SWEEP_SAMPLE:
        blob[key] = out
    else:
        blob[key + '_shape'] = np.array(out.shape)
        blob[key + '_sample'] = out.ravel()[option_sweep_sample_index(out.size)]
