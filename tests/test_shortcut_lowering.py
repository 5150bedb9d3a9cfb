"""Lowering of ResNet50's projection shortcuts into block 0's conv3 (no GPU): with `shortcut_stages` the listed stages emit no
downsample op, their conv3 reads the block input as a shortcut segment, and every byte any op reads -- the shortcut input
included -- was written by an earlier op and still holds what that op wrote when it is read."""
import numpy as np
import pytest

from pd_fusion_b200 import _lib
from pd_fusion_b200.backbone import _parse_stages, conv_list, lower_resnet


def _check_dataflow(ops, extents):
    """Tag every byte with the index of the op that last wrote it; return, per op, the set of writer names of each range it read."""
    tag = {k: np.full(v, -1, dtype=np.int64) for k, v in extents.items()}
    tag["input"][:] = -2
    names = [o[0] for o in ops]
    reads = []
    esz = 2
    for i, (name, f, refs, _) in enumerate(ops):
        seen, ranges = {}, []

        def read(key, nbytes):
            buf, off = refs[key]
            t = tag[buf][off:off + nbytes]
            assert len(t) == nbytes and (t != -1).all(), (name, key, "read before written")
            seen[key] = {("input" if w == -2 else names[w]) for w in np.unique(t)}
            ranges.append((buf, off, off + nbytes))

        in_bytes = f["n"] * f["h"] * f["w"] * f["c"] * (4 if (f["kind"] == _lib.OP_AVGPOOL and f.get("out_f32")) else esz)
        read("d_in", in_bytes)
        if "d_residual" in refs:
            if f.get("sc_c"):
                sc_h, sc_w = f["sc_hw"] >> 16, f["sc_hw"] & 0xFFFF
                read("d_residual", f["n"] * sc_h * sc_w * f["sc_c"] * esz)
            else:
                read("d_residual", f["n"] * f["ho"] * f["wo"] * f["k"] * esz)
        reads.append(seen)

        def write(key, nbytes):
            buf, off = refs[key]
            assert off + nbytes <= extents[buf], (name, key)
            for rb, r0, r1 in ranges:              # an op never overwrites what it reads
                assert rb != buf or r1 <= off or off + nbytes <= r0, (name, key, "overwrites its own input")
            tag[buf][off:off + nbytes] = i

        if f["kind"] == _lib.OP_AVGPOOL:
            write("d_out", f["n"] * f["c"] * 4)
        elif f["kind"] == _lib.OP_MAXPOOL:
            write("d_out", f["n"] * f["ho"] * f["wo"] * f["c"] * esz)
        else:
            write("d_out", f["n"] * f["ho"] * f["wo"] * f["k"] * (4 if f.get("out_f32") else esz))
        if "d_out3" in refs:
            write("d_out3", f["n"] * f["ho"] * f["wo"] * f["k3"] * esz)
    assert (tag["output"] >= 0).all()
    return reads


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("chain", [(), (1, 2, 3)])
@pytest.mark.parametrize("chunks", [[2, 2, 4, 4, 7], [7, 7, 7, 7, 7]])
def test_shortcut_lowering_dataflow(fused, chain, chunks):
    n, S = 7, 70                                 # odd stage sizes: 18 -> 18 -> 9 -> 5 -> 3
    ops, extents, _ = lower_resnet("resnet50", n, S, bf16=True, fused_stem=fused, chunks=chunks, chain_stages=chain,
                                   shortcut_stages=(1, 2, 3, 4))
    assert not any("downsample" in o[0] for o in ops)
    reads = _check_dataflow(ops, extents)
    down = {cv["block"]: cv for cv in conv_list("resnet50") if cv["role"] == "down"}
    fused_convs = set()
    for (name, f, refs, wname), seen in zip(ops, reads):
        if not f.get("sc_c"):
            assert "_shortcut" not in f
            continue
        fused_convs.add(name)
        k = int(name[5])
        blk = name.rsplit(".", 1)[0]
        assert name.endswith(".0.conv3") and f["_shortcut"] == down[blk]["name"] and f["sc_c"] == down[blk]["cin"]
        assert f["k"] == down[blk]["cout"] and f["r"] == 1 and f["stride"] == 1 and f["relu"] == 1 and not f.get("out_f32")
        sc_h, sc_w = f["sc_hw"] >> 16, f["sc_hw"] & 0xFFFF
        assert sc_h == sc_w and (f["ho"] == sc_h if k == 1 else f["ho"] == (sc_h - 1) // 2 + 1)
        # the shortcut input is the stage input, still as the previous stage's last conv3 (or the stem) wrote it
        prev = "layer1.2.conv3" if k == 2 else "layer2.3.conv3" if k == 3 else "layer3.5.conv3" if k == 4 else None
        assert seen["d_residual"] == ({prev} if prev else ({"stem.fused"} if fused else {"maxpool"})), (name, seen["d_residual"])
    assert fused_convs == {f"layer{k}.0.conv3" for k in range(1, 5)}


def test_shortcut_stages_default_off_and_selective():
    """lower_resnet defaults to no shortcut stage (the downsample ops stay), a subset fuses only those stages, resnet18 and the
    fp32 path are unaffected."""
    base, ext, _ = lower_resnet("resnet50", 3, 64, bf16=True, fused_stem=True, chunks=[3] * 5)
    assert sum("downsample" in o[0] for o in base) == 4 and not any(o[1].get("sc_c") for o in base)
    part, ext2, _ = lower_resnet("resnet50", 3, 64, bf16=True, fused_stem=True, chunks=[3] * 5, shortcut_stages=(1, 2))
    assert {o[0] for o in part if "downsample" in o[0]} == {"layer3.0.downsample.0", "layer4.0.downsample.0"}
    assert {o[0] for o in part if o[1].get("sc_c")} == {"layer1.0.conv3", "layer2.0.conv3"}
    assert len(part) == len(base) - 2
    _check_dataflow(part, ext2)
    for arch, bf16 in (("resnet18", True), ("resnet50", False)):
        a = lower_resnet(arch, 3, 64, bf16=bf16, fused_stem=bf16, chunks=[3] * 5)
        b = lower_resnet(arch, 3, 64, bf16=bf16, fused_stem=bf16, chunks=[3] * 5, shortcut_stages=(1, 2, 3, 4))
        assert a == b


def test_parse_stages(monkeypatch):
    monkeypatch.delenv("PDFUSION_B200_SHORTCUT", raising=False)
    assert _parse_stages("PDFUSION_B200_SHORTCUT", (1, 2)) == (1, 2)
    for v, want in (("none", ()), ("", ()), ("1,2,3", (1, 2, 3)), ("4", (4,))):
        monkeypatch.setenv("PDFUSION_B200_SHORTCUT", v)
        assert _parse_stages("PDFUSION_B200_SHORTCUT", (1, 2)) == want
