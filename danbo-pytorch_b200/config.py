"""Flag handling for the path: the reference's argparse defaults (run_nerf.py:186-572) for the flags this package reads,
the values its shipped configs set on top of them, and a reader for its `key = value` config files (configs/**.txt).
tests/test_oracle_vs_reference.py checks all three against the reference's own parser on the shipped configs."""
import argparse

# the reference CLI's own defaults (expname / basedir: conveniences, the reference requires them)
DEFAULTS = dict(
    expname='danbo', basedir='./logs', no_reload=False, ft_path=None, finetune=False, finetune_light=False,
    nerf_type='nerf', gnn_backbone='PoolPNGCN', agg_backbone='mlp', agg_type='softmax', agg_W=16, agg_D=3,
    node_W=32, gcn_D=4, gcn_fc_D=1, voxel_res=4, voxel_feat=4, multires_voxel=5, multires_graph=5,
    multires_views=4, multires=10, netdepth=8, netwidth=256, netwidth_view=None, mask_root=False,
    mask_vol_prob=False, opt_vol_scale=False, vol_cal_scale=False, attenuate_feat=False,
    attenuate_invalid=False, align_bones='align', use_volume_near_far=False, single_net=False,
    opt_framecode=False, framecode_size=16, n_framecodes=None, density_type='relu', density_scale=1.0,
    raw_noise_std=0.0, ray_noise_std=0.0, perturb=1.0, N_samples=64, N_importance=0, N_rand=4096,
    N_sample_images=8, chunk=65536, netchunk=65536, lrate=0.0005, lrate_decay=250, lrate_decay_rate=0.1,
    decay_unit=1000, weight_decay=None, loss_fn='MSE', coarse_weight=1.0, rgb_loss_coef=1.0,
    soft_softmax_loss_coef=0.01, vol_scale_penalty=0.01, use_background=False, use_viewdirs=False,
    lindisp=False, ext_scale=0.001, kp_dist_type='reldist', view_type='relray', ray_tr_type='local',
    pts_tr_type='local', bone_type='reldir', graph_input_type='quat', use_cutoff=False, opt_posecode=False,
    gnn_concat=False, no_adj=False, adj_self_one=False, align_corners=False, opt_pose=False, i_embed=0,
    multires_bones=0, cutoff_mm=500, cutoff_viewdir=False, cutoff_inputs=False, cutoff_shift=False,
    cut_to_dist=False, cutoff_bones=False, normalize_cutoff=False, opt_cutoff=False, freq_schedule=False,
    netwidth_fine=256,
)

# what configs/*/danbo_base.txt and danbo_fast.txt set on top of the CLI defaults (identical in both files)
DANBO_CONFIG = dict(
    nerf_type='danbo', gnn_backbone='FGNNcat', agg_backbone='vox_MIXGNN', agg_type='sigmoid', agg_W=32,
    node_W=128, voxel_res=16, voxel_feat=5, multires_voxel=6, multires=1, mask_root=True, mask_vol_prob=True,
    opt_vol_scale=True, vol_cal_scale=True, attenuate_feat=True, single_net=True, opt_framecode=True,
    framecode_size=128, raw_noise_std=1.0, N_rand=3072, N_sample_images=16, chunk=4096, lrate_decay=500000,
    decay_unit=1, loss_fn='L1', soft_softmax_loss_coef=0.001, vol_scale_penalty=0.001, use_background=True,
    use_viewdirs=True, view_type='identity', ray_tr_type='world', bone_type='Nope', graph_input_type='rot6d',
    cutoff_shift=True, cut_to_dist=True,
)

PRESETS = {
    "danbo_base": dict(DANBO_CONFIG, N_samples=96, N_importance=48),
    "danbo_fast": dict(DANBO_CONFIG, N_samples=32, N_importance=16, use_volume_near_far=True),
    "danbo_cfg3": dict(DANBO_CONFIG, N_samples=64, N_importance=16),               # BASELINE config #3 (SURVEY F11)
    # configs/h36m_zju/anerf_base.txt (BASELINE config #4)
    "anerf_base": dict(
        nerf_type='nerf', netwidth=448, netwidth_fine=448, multires=7, multires_views=4, bone_type='reldir',
        kp_dist_type='reldist', view_type='relray', ray_tr_type='local', use_cutoff=True, cutoff_viewdir=True,
        cutoff_inputs=True, cutoff_shift=True, cut_to_dist=True, N_samples=96, N_importance=48,
        use_volume_near_far=False, single_net=True, opt_framecode=True, framecode_size=128, raw_noise_std=1.0,
        N_rand=3072, N_sample_images=16, chunk=4096, lrate_decay=500000, decay_unit=1, loss_fn='L1',
        use_background=True, use_viewdirs=True),
}


# flags of this package that the reference does not have: the 2D keypoint reprojection term of pose fitting and
# --opt_pose training (training.kp2d_batch); kp2d_coef = 0 leaves it off
PACKAGE_DEFAULTS = dict(kp2d_sigma=100.0, kp2d_coef=0.0)


def _coerce(v):
    if v in ("True", "False"):
        return v == "True"
    if v == "None":
        return None
    for cast in (int, float):
        try:
            return cast(v)
        except ValueError:
            pass
    if v.startswith("[") and v.endswith("]"):
        return [x.strip() for x in v[1:-1].split(",")]
    return v


def read_config_file(path):
    out = {}
    for line in open(path):
        line = line.split("#")[0].strip()
        if "=" in line:
            k, v = [s.strip() for s in line.split("=", 1)]
            out[k] = _coerce(v)
    return out


def make_args(preset=None, config_file=None, **overrides):
    d = dict(DEFAULTS, **PACKAGE_DEFAULTS)
    if config_file is not None:
        d.update(read_config_file(config_file))
    if preset is not None:
        d.update(PRESETS[preset])
    d.update(overrides)
    return argparse.Namespace(**d)
