"""Every model of the registry builds, runs a forward/backward at a reduced resolution and has the parameter count of
the architecture it names (the reference benchmarks torchvision's resnet/vgg/densenet, its own inceptionv4 and
transformers' BERT: dear/imagenet_benchmark.py:70-82, dear/bert_benchmark.py:60-75)."""
import pytest
import torch

from dear_pytorch_b200.models.registry import available, create, input_size

# torchvision / transformers parameter counts of the named architectures
EXPECTED = {"resnet18": 11_689_512, "resnet34": 21_797_672, "resnet50": 25_557_032, "resnet101": 44_549_160,
            "resnet152": 60_192_808, "vgg11": 132_863_336, "vgg16": 138_357_544, "vgg19": 143_667_240,
            "densenet121": 7_978_856, "densenet169": 14_149_480, "densenet201": 20_013_928}


def test_registry_lists_the_reference_models():
    names = set(available())
    assert {"resnet50", "vgg16", "densenet121", "inceptionv4", "bert", "bert_base", "mnist"} <= names
    assert input_size("inceptionv4") == 299 and input_size("resnet50") == 224


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_parameter_counts_match_the_named_architecture(name):
    with torch.device("meta"):
        model = create(name)
    assert sum(p.numel() for p in model.parameters()) == EXPECTED[name]


@pytest.mark.parametrize("name,size", [("resnet18", 64), ("vgg11", 32), ("densenet121", 64), ("inceptionv4", 96), ("mnist", 28)])
def test_forward_backward_at_reduced_resolution(name, size):
    torch.manual_seed(0)
    model = create(name)
    ch = 1 if name == "mnist" else 3
    x = torch.randn(2, ch, size, size)
    if name.startswith("vgg"):                         # the classifier expects 7x7 features: keep the spec'd input
        x = torch.randn(1, 3, 224, 224)
    out = model(x)
    assert out.shape[0] == x.shape[0] and torch.isfinite(out).all()
    out.float().square().mean().backward()
    assert all(p.grad is not None for p in model.parameters() if p.requires_grad)


def test_fused_variants_keep_the_state_dict():
    for name in ("resnet50", "densenet121"):
        with torch.device("meta"):
            a, b = create(name), create(name, fused_bn=True)
        assert list(a.state_dict().keys()) == list(b.state_dict().keys())
    from dear_pytorch_b200.models import bert
    cfg = bert.BertConfig(hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128, vocab_size=100)
    with torch.device("meta"):
        a, b = bert.BertForPreTraining(cfg), bert.BertForPreTraining(cfg, fused_ln=True, tc_ffn=True)
    assert list(a.state_dict().keys()) == list(b.state_dict().keys())
    with torch.device("meta"):
        large = bert.BertForPreTraining(bert.BERT_LARGE)
    assert sum(p.numel() for p in large.parameters()) == 336_232_258      # the count bench.py reports for BERT-large


def test_bert_matches_transformers_bert_for_pretraining():
    """Same architecture as the model the reference trains (dear/bert_benchmark.py:72-83): load the weights of a small
    ``transformers.BertForPreTraining`` through the converter and compare both heads, with and without key padding; the
    converter round-trips."""
    transformers = pytest.importorskip("transformers")
    from dear_pytorch_b200.models import bert as B
    cfg = dict(vocab_size=90, hidden_size=32, num_hidden_layers=3, num_attention_heads=4, intermediate_size=64,
               max_position_embeddings=24)
    torch.manual_seed(0)
    hf = transformers.BertForPreTraining(transformers.BertConfig(**cfg)).eval()
    with torch.no_grad():                                  # the zero-initialised biases / unit LayerNorms prove nothing
        for p in hf.parameters():
            p.add_(0.05 * torch.randn_like(p))
    ours = B.BertForPreTraining(B.BertConfig(**cfg)).eval()
    assert ours.vocab_size == 96                           # padded to a multiple of 8 like the reference does (:77-78)
    ours.load_state_dict(B.from_hf_state_dict(hf.state_dict(), cfg["num_hidden_layers"], ours.vocab_size))
    ids = torch.randint(0, 90, (3, 20))
    types = torch.randint(0, 2, (3, 20))
    mask = torch.ones(3, 20, dtype=torch.long)
    mask[1, 13:] = 0
    mask[2, 5:] = 0
    with torch.no_grad():
        for m in (None, mask):
            ref = hf(input_ids=ids, token_type_ids=types, attention_mask=m)
            scores, nsp = ours(ids, types, m)
            torch.testing.assert_close(scores[..., :90], ref.prediction_logits, rtol=1e-4, atol=1e-4)
            torch.testing.assert_close(nsp, ref.seq_relationship_logits, rtol=1e-4, atol=1e-4)
    back = B.to_hf_state_dict(ours.state_dict(), cfg["num_hidden_layers"], 90)
    missing = hf.load_state_dict(back, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys)
    for k, v in hf.state_dict().items():
        if k in back:
            assert torch.equal(back[k], v), k


@pytest.mark.parametrize("name", ["resnet18", "resnet50", "vgg11", "densenet121"])
def test_cnn_matches_torchvision(name):
    """The reference benchmarks torchvision's models by name (dear/imagenet_benchmark.py:78-82): same parameters, same
    function.  ResNet / VGG even share the state-dict keys; DenseNet's module tree is flatter here, with the tensors in
    the same order."""
    tv = pytest.importorskip("torchvision")
    torch.manual_seed(0)
    ref = getattr(tv.models, name)()
    with torch.no_grad():
        for m in ref.modules():                            # non-trivial BatchNorm statistics and affine parameters
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5); m.weight.uniform_(0.5, 1.5); m.bias.normal_(0, 0.1)
    ours = create(name)
    src = ref.state_dict()
    if set(src) == set(ours.state_dict()):
        ours.load_state_dict(src)
    else:
        mine = ours.state_dict()
        assert [tuple(v.shape) for v in mine.values()] == [tuple(v.shape) for v in src.values()]
        ours.load_state_dict(dict(zip(mine.keys(), src.values())))
    x = torch.randn(2, 3, 64, 64)
    ref.eval(); ours.eval()
    with torch.no_grad():
        torch.testing.assert_close(ours(x), ref(x), rtol=1e-4, atol=1e-4)
    ref.train(); ours.train()
    if name.startswith("vgg"):
        torch.manual_seed(1); a = ours(x)
        torch.manual_seed(1); b = ref(x)                   # same dropout masks
    else:
        a, b = ours(x), ref(x)
    torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4)
    for (ka, va), (kb, vb) in zip(ours.state_dict().items(), ref.state_dict().items()):
        if "running" in ka:
            torch.testing.assert_close(va, vb, rtol=1e-5, atol=1e-6)      # the training forward updated the same statistics


def seeded_state_dict(sd):
    """Deterministic values for a state dict, drawn in its order from its shapes and attribute names only, so two modules
    whose tensors line up one to one receive the same values: He-scaled convolution / linear weights, non-trivial
    BatchNorm statistics and affine parameters."""
    g = torch.Generator().manual_seed(0)
    out = {}
    for k, v in sd.items():
        if not v.is_floating_point():
            out[k] = v.clone()
        elif v.dim() > 1:
            out[k] = torch.randn(v.shape, generator=g) * (2.0 / v[0].numel()) ** 0.5
        elif k.endswith(("running_var", "weight")):
            out[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            out[k] = torch.randn(v.shape, generator=g) * 0.1
    return out


def inceptionv4_input():
    return torch.randn(2, 3, 299, 299, generator=torch.Generator().manual_seed(1))


def test_inceptionv4_matches_the_reference_file():
    """The reference ships its own Inception-v4 (dear/inceptionv4.py, the Cadene implementation).  Its tensors line up
    with ours one to one (896, same order and shapes), and with the same values both compute the same function.  The
    reference's shapes and its logits for seeded weights and inputs are stored in tests/golden/ (written by
    tests/golden/make_inceptionv4_reference.py)."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "inceptionv4_reference.json")) as f:
        golden = json.load(f)
    ours = create("inceptionv4").eval()
    mine = ours.state_dict()
    assert len(mine) == 896
    assert [list(v.shape) for v in mine.values()] == golden["state_dict_shapes"]
    ours.load_state_dict(seeded_state_dict(mine))
    with torch.no_grad():
        torch.testing.assert_close(ours(inceptionv4_input()), torch.tensor(golden["logits"]), rtol=1e-3, atol=1e-3)
