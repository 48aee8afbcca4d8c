"""The handle's un-guided forward (ca_forward, driven through NativeModel.forward) against model.py's `forward`: the same
kernels in the same order, so the two agree to the rounding of the host-built tables through eager, captured and
replayed calls, draw the same numbers from the global generator, and keep the CuriosityModule's ring buffer alike."""
import pytest
import torch

from oracle import cogaim_oracle as orc

pytestmark = pytest.mark.gpu


def _close(p, q):
    assert torch.allclose(p, q, rtol=1e-4, atol=1e-6), (p - q).abs().max()


@pytest.mark.parametrize("with_exif", [True, False])
def test_handle_forward_matches_the_model(cuda_device, with_exif):
    from cognitive_aim_depth_estimation_b200.model import create_model
    from cognitive_aim_depth_estimation_b200.native import NativeModel
    sd = orc.build_state_dict(0)
    m = create_model({"model": {}}, {"num_cameras": 71}, device=cuda_device)
    m.load_state_dict(sd)
    nat = NativeModel(sd, device=cuda_device, fold_layernorm=m._ln_folded())
    B = 3
    x = orc.synthetic_images(B, 518, seed=5).cuda()
    ex = {k: v.cuda() for k, v in orc.synthetic_exif(B, seed=6).items()} if with_exif else None
    # (return_attention, CuriosityModule runs of the model's forward): a fresh model runs it twice (no attention stored
    # yet), then once, or twice when it returns the attention; each path is called eagerly, captured, then replayed
    calls = [(False, 2), (False, 1), (False, 1), (False, 1), (True, 2), (True, 2), (True, 2)]
    side = torch.cuda.Stream()  # the handle captures nothing on the legacy default stream
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i, (ret, runs) in enumerate(calls):
            torch.manual_seed(30 + i)
            a = m.forward(x, ex, return_attention=ret)
            fused = m.fusion_features
            drawn = torch.get_rng_state()
            torch.manual_seed(30 + i)
            depth, conf, att, nat_fused = nat.forward(x, ex, runs=runs)
            assert torch.equal(torch.get_rng_state(), drawn), i
            _close(a[0], depth)
            _close(a[1], conf)
            if ret:
                _close(a[2], att)
            assert ((fused - nat_fused).norm() / fused.norm()).item() < 1e-4, i
    torch.cuda.synchronize()
    n = B * sum(runs for _, runs in calls)
    assert int(nat.history_pointer) == int(m.curiosity_module.history_pointer) == n
    assert torch.allclose(nat.exploration_history[:n], m.curiosity_module.exploration_history[:n], rtol=1e-4, atol=1e-7)
    nat.close()
