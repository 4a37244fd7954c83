"""CPU checks of the entry-point host logic: the reference's command-line surface, checkpoint key handling, and the
context-parallel condition broadcast (gloo, world size 2)."""
import os

import pytest
import torch

# option strings of cosmos_predict1/diffusion/inference/gen3c_single_image.py:35-99 + inference_utils.py:53-171, stored
# here so that the check needs no copy of the reference (its video-input options --input_image_or_video_path and
# --num_input_frames are not taken by this entry point)
REFERENCE_OPTIONS = [
    "--checkpoint_dir", "--tokenizer_dir", "--video_save_name", "--video_save_folder", "--prompt", "--batch_input_path",
    "--negative_prompt", "--num_steps", "--guidance", "--num_video_frames", "--height", "--width", "--fps", "--seed",
    "--num_gpus", "--disable_prompt_upsampler", "--offload_diffusion_transformer", "--offload_tokenizer",
    "--offload_text_encoder_model", "--offload_prompt_upsampler", "--offload_guardrail_models", "--disable_guardrail",
    "--disable_prompt_encoder", "--prompt_upsampler_dir", "--input_image_path", "--trajectory", "--camera_rotation",
    "--movement_distance", "--noise_aug_strength", "--save_buffer", "--filter_points_threshold", "--foreground_masking"]


def test_command_line_surface_matches_reference():
    from gen3c_b200.inference import gen3c_single_image as m

    p = m.create_parser()
    have = {s for a in p._actions for s in a.option_strings}
    assert set(REFERENCE_OPTIONS) <= have
    d = p.parse_args([])
    assert (d.num_steps, d.guidance, d.num_video_frames, d.height, d.width, d.fps, d.seed) == (35, 1, 121, 704, 1280, 24, 1)
    assert (d.trajectory, d.camera_rotation, d.movement_distance, d.filter_points_threshold) == ("left", "center_facing", 0.3, 0.05)
    assert d.tokenizer_dir == "Cosmos-Tokenize1-CV8x8x8-720p" and d.checkpoint_dir == "checkpoints"
    with pytest.raises(AssertionError):
        m.validate_args(p.parse_args(["--num_video_frames", "100"]))
    m.validate_args(p.parse_args(["--num_video_frames", "361"]))


def test_non_strict_load_reports_shapes_and_skips_te_state():
    from gen3c_b200 import inference_utils as iu

    net = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    sd = {"0.weight": torch.ones(3, 4), "1.weight": torch.ones(5, 5), "0._extra_state": torch.zeros(1), "2.weight": torch.ones(1)}
    res = iu.non_strict_load_model(net, sd)
    assert res.missing_keys == ["1.weight"] and res.unexpected_keys == ["2.weight"]
    assert res.incorrect_shapes == [("1.weight", (5, 5), (2, 3))]
    assert float(net[0].weight.sum()) == 12.0


def _bcast_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from gen3c_b200.model_gen3c import VideoExtendCondition
        from gen3c_b200.parallel import broadcast_condition

        # rank 1 starts with different values AND a different shape: the robust broadcast resizes it
        c = VideoExtendCondition(crossattn_emb=torch.full((1, 4, 8), float(rank)), video_cond_bool=bool(rank == 0),
                                 gt_latent=torch.full((1, 2, 3 + rank, 2, 2), 7.0 + rank), fps=None)
        c = broadcast_condition(c, cp_group=dist.group.WORLD)
        out.put((rank, float(c.crossattn_emb.mean()), tuple(c.gt_latent.shape), float(c.gt_latent.mean()), c.video_cond_bool,
                 c.fps))
    finally:
        dist.destroy_process_group()


def test_broadcast_condition_gloo_world2():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29650 + os.getpid() % 300
    ps = [ctx.Process(target=_bcast_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in ps:
        p.start()
    got = sorted(out.get(timeout=120) for _ in range(2))
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0][1:] == got[1][1:] == (0.0, (1, 2, 3, 2, 2), 7.0, True, None)
