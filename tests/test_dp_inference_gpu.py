"""Data-parallel survival inference on the GPU.

First the property the split rests on: how much a patient's eval-mode prediction and GradCAM maps depend on which other
patients share its batch.  They are not bit-identical.  On a B200, the same 11 patients forwarded in batches of 4
instead of 11 give predictions that differ by up to 1.6e-4 (the largest prediction is 0.20), and maps that differ by up
to 0.016: the maps are normalised per sample, (cam - min) / max, which magnifies the fp16 rounding of the trunk
activations wherever a cam's range is small next to its level.  So predictions and maps are compared within bounds, and
the C-indices exactly against the gathered predictions themselves.  Then inference_survival over ranks started with
mp.spawn (NCCL, one GPU per rank, when enough GPUs are visible; otherwise every rank on cuda:0 over gloo, so the test
runs on any machine with a GPU)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist

from tests.dp_helpers import spawn_ranks

pytestmark = pytest.mark.gpu
CIN, SPATIAL, BATCH, RESAMPLES = 2, (64, 64, 32), 4, 64
PRED_TOL = 1e-3      # max |prediction difference| between batch compositions (measured: 1.6e-4)
MAP_TOL = 5e-2       # max |map difference|, maps in [0, 1] (measured: 0.016); the bound tests/test_gradcam_batched_gpu.py
                     # holds the batched maps to against the reference's golden maps


def _model(blend, dev):
    from mmnn_sts_b200.models.densenet import DenseNet121
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    from oracle import synth
    m = MultiModalModel(DenseNet121(spatial_dims=3, in_channels=CIN, out_channels=2, feature_channels=12, dropout_prob=0.0),
                        ["x"] * 20, 2, 12, blend=blend)
    m.load_state_dict(synth.make_state_dict(131, in_channels=CIN))
    return m.to(dev).eval()


@pytest.mark.parametrize("blend", [False, True])
def test_eval_outputs_do_not_depend_on_batch_composition(blend):
    """The same 11 patients in batches of 11, 4 and 1: predictions (every head) and maps within PRED_TOL / MAP_TOL."""
    from mmnn_sts_b200.utils.utils import attention_maps
    from oracle import synth
    dev = torch.device("cuda", 0)
    m = _model(blend, dev)
    image, clinical, _, _ = synth.make_batch(132, 11, CIN, SPATIAL)
    res = {}
    for bs in (11, 4, 1):
        outs, maps = [], []
        for s in range(0, 11, bs):
            o, mp = attention_maps(m, {"image": image[s:s + bs].to(dev), "clinical": clinical[s:s + bs].to(dev)})
            outs.append(o); maps.append(mp)
        res[bs] = (torch.cat(outs, dim=-2), torch.cat(maps))
    worst = []
    for bs in (4, 1):
        dp = float((res[bs][0] - res[11][0]).abs().max())
        dm = float((res[bs][1] - res[11][1]).abs().nan_to_num().max())
        same_nan = torch.equal(res[bs][1].isnan(), res[11][1].isnan())
        print("blend", blend, "batch", bs, "vs 11: max |prediction diff|", dp, "max |map diff|", dm,
              "max |prediction|", float(res[11][0].abs().max()))
        worst.append((bs, dp, dm, same_nan))
    assert all(dp <= PRED_TOL and dm <= MAP_TOL and same_nan for _, dp, dm, same_nan in worst), worst


def _batches(image, clinical, events, durations, ids):
    return [({"image": image[ids[s:s + BATCH]], "clinical": clinical[ids[s:s + BATCH]]}, events[ids[s:s + BATCH]],
             durations[ids[s:s + BATCH]]) for s in range(0, len(ids), BATCH)]


def _worker(rank, world, port, blend, n, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    nccl = torch.cuda.device_count() >= world
    dev = torch.device("cuda", rank if nccl else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl" if nccl else "gloo", rank=rank, world_size=world)
    try:
        from mmnn_sts_b200 import distributed as D
        from mmnn_sts_b200.main import (_draw_resamples, bootstrap_cindices, getCIndices, inference_survival,
                                        predict_risks)
        from oracle import synth
        m = _model(blend, dev)
        image, clinical, events, durations = synth.make_batch(133, n, CIN, SPATIAL)
        if n < BATCH:
            events = torch.ones_like(events)              # so that the few patients still form an admissible pair
        # one process over every patient in global order
        ref_maps = {}

        def ref_cb(i, maps):
            for k in range(maps.shape[0]):
                ref_maps[i * BATCH + k] = maps[k].clone()

        everyone = torch.arange(n)
        ref = inference_survival(m, _batches(image, clinical, events, durations, everyone), dev, num_resamples=RESAMPLES,
                                 seed=134, gradcam=ref_cb)
        # this rank's strided shard, ragged last batch
        ids = D.shard_patients(n, rank, world)
        mine = _batches(image, clinical, events, durations, ids)
        got_maps = {}

        def cb(i, maps):
            for k in range(maps.shape[0]):
                got_maps[int(ids[i * BATCH + k])] = maps[k].clone()

        g = dist.group.WORLD
        got = inference_survival(m, mine, dev, num_resamples=RESAMPLES, seed=134, gradcam=cb, group=g, patient_ids=ids)
        assert got.preds.shape == (n, 2), "preds shape"
        # gather and order exact: this rank's rows are its own forward, bit for bit
        if len(ids):
            local, _, _ = predict_risks(m, mine, dev)
            assert torch.equal(got.preds[ids.to(dev)], local), "gathered rows of this rank"
        assert float((got.preds - ref.preds).abs().max()) <= PRED_TOL, "preds vs one process"
        # C-indices exact against one process counting the gathered predictions with the same resamples
        ev, du = events.to(dev), durations.to(dev)
        idx = torch.as_tensor(_draw_resamples(n, RESAMPLES, 134), device=dev)
        want = bootstrap_cindices(got.preds, ev, du, idx)
        assert np.array_equal(got.per_resample, want[0], equal_nan=True), "per_resample"
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in ((got.mean, want[1]), (got.std, want[2]))), "mean / std"
        assert sorted(got_maps) == sorted(ids.tolist()), "maps of this rank's patients"
        assert all(torch.allclose(got_maps[p], ref_maps[p], rtol=0, atol=MAP_TOL, equal_nan=True) for p in got_maps), "maps"
        c, preds = inference_survival(m, mine, dev, bootstrap=False, group=g, patient_ids=ids)
        assert torch.equal(preds, got.preds) and c == getCIndices(got.preds, ev, du), "bootstrap=False"
        ret[rank] = ("ok", "nccl" if nccl else "gloo", len(ids), got.preds.cpu().numpy(), got.per_resample, got.mean,
                     got.std, c)
    except BaseException as ex:                           # reported by the parent
        ret[rank] = (repr(ex)[:2000],)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,blend,n", [(2, True, 37), (2, False, 37), (3, False, 2)])
def test_data_parallel_inference_equals_one_process(world, blend, n):
    """37 patients over 2 ranks (19 / 18, batches of 4 with a ragged last batch), and 2 patients over 3 ranks (the last
    rank forwards nothing).  Every rank must return the same result."""
    import torch.multiprocessing as mp
    with mp.Manager() as mgr:
        ret = mgr.dict()
        spawn_ranks(_worker, world, (blend, n, ret))
        res = dict(ret)
    assert sorted(res) == list(range(world)) and all(res[r][0] == "ok" for r in res), {r: res[r][0] for r in res}
    print("backend", res[0][1], "patients per rank", [res[r][2] for r in range(world)])
    assert [res[r][2] for r in range(world)] == [len(range(r, n, world)) for r in range(world)]
    for r in range(1, world):
        assert np.array_equal(res[r][3], res[0][3])
        for k in (4, 5, 6):
            assert np.array_equal(res[r][k], res[0][k], equal_nan=True)
        assert res[r][7] == res[0][7]
