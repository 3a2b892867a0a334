"""CPU: the module tree / state_dict contract. The state_dict keys and shapes of the UNMODIFIED reference SoftGroup class
(instantiated on this repo's spconv/ops shims; tests/golden/ref_host.json) must equal ours one to one (checkpoints load
unchanged, softgroup/util/utils.py:111-145)."""
import torch

from softgroup_b200.configs import model_cfg
from softgroup_b200.model import SoftGroup


def test_state_dict_names():
    m = SoftGroup(**model_cfg('scannet'))
    sd = m.state_dict()
    for k in ['input_conv.0.weight', 'unet.blocks.block0.conv_branch.2.weight', 'unet.conv.2.weight',
              'unet.deconv.2.weight', 'unet.blocks_tail.block0.i_branch.0.weight', 'unet.u.u.u.u.u.u.blocks.block1.conv_branch.5.weight',
              'tiny_unet.blocks.block0.conv_branch.0.running_mean', 'semantic_linear.3.weight', 'offset_linear.1.running_var',
              'cls_linear.weight', 'mask_linear.2.bias', 'iou_score_linear.bias', 'output_layer.0.weight']:
        assert k in sd, k
    assert tuple(sd['input_conv.0.weight'].shape) == (32, 3, 3, 3, 6)
    assert tuple(sd['unet.conv.2.weight'].shape) == (64, 2, 2, 2, 32)
    assert tuple(sd['unet.deconv.2.weight'].shape) == (32, 2, 2, 2, 64)
    assert tuple(sd['unet.blocks_tail.block0.i_branch.0.weight'].shape) == (32, 1, 1, 1, 64)
    n_subm = sum(1 for k, v in sd.items() if k.endswith('weight') and v.dim() == 5 and v.shape[1] == 3)
    assert n_subm == 53 + 12  # backbone + tiny U-Net


def test_reference_class_on_our_shims_has_identical_state_dict(host_gold):
    want = host_gold['state_dict']
    ours = SoftGroup(**model_cfg('scannet'))
    b = ours.state_dict()
    assert [k for k, _ in want] == list(b.keys())
    for k, shape in want:
        assert list(b[k].shape) == shape, k
    ours.load_state_dict({k: torch.zeros(shape, dtype=b[k].dtype) for k, shape in want})  # strict


def test_model_survives_deepcopy_and_pickle():
    """The per-thread scratch (threading.local) and the compiled plans (ctypes arrays, raw pointers) stay out of the module's
    state: copy.deepcopy and torch.save(module) work and the copies rebuild them on demand."""
    import copy
    import io
    from softgroup_b200.configs import model_cfg
    from softgroup_b200.model import SoftGroup
    m = SoftGroup(**model_cfg('scannet', channels=16, num_blocks=3))
    m2 = copy.deepcopy(m)
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    for c in (m2, m3):
        assert c._plans == {} and hasattr(c, '_tls')
        assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), c.state_dict().values()))
