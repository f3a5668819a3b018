"""GPU: the streaming session over region groups (pb_variant_stream_*) and the multi-GPU product path built on it.

* 1 GPU: a session over ragged group sizes — host-staged and device-resident — gives the records of the one-shot call
  bit for bit (the head kernel writes them itself), whatever the group boundaries are.
* 2 GPUs (skipped on a 1-GPU box): DistributedVariantCaller under both schedules; the gathered, order-restored records on
  BOTH ranks equal the 1-rank result of the same region list bit for bit (VERDICT r1 item 3)."""
import os
import numpy as np
import pytest

from pepper_b200 import synth

pytestmark = pytest.mark.gpu


def _workload():
    reads, regions = synth.make_variant_workload(6, 4000, 30, synth.ONT, seed=51)
    return synth.tile_workload(reads, regions, 12)            # 72 regions, ~8 k candidates


def test_stream_session_matches_one_shot_call():
    import torch
    from oracle import nets
    from pepper_b200.abi import HostReads, regions_array, PRED_RECORD
    from pepper_b200.dist import records_from_calls
    from pepper_b200.pipeline import VariantCaller, DeviceReads
    reads, regions = _workload()
    params = synth.ont_params()
    caller = VariantCaller(nets.make_variant_weights(5))
    want = caller.call(reads, regions, params, want_images=True)
    wrec = records_from_calls(want)
    n_reg = regions.n_regions
    cuts = [0, 1, 8, 9, 40, n_reg]                            # ragged groups, incl. a single-region one
    cap = len(want) + 64
    hr = HostReads(reads, pin=True)
    regs, keep = regions_array(regions)
    ref = np.ascontiguousarray(regions.ref, dtype=np.uint8)
    dreads = DeviceReads(reads, regions)
    for mode in ("host", "device"):
        rec_t = torch.zeros(cap * PRED_RECORD.itemsize, dtype=torch.uint8, device="cuda")
        s = caller.stream(params, cap, d_records=rec_t.data_ptr())

        def stage(i):
            if mode == "host":
                s.stage_host(hr, regs, cuts[i], cuts[i + 1], ref, cuts[i])
            else:
                s.stage_device(dreads, cuts[i], cuts[i + 1], cuts[i])
        stage(0)
        for i in range(len(cuts) - 1):
            s.run(flush=False)
            if i + 2 < len(cuts):
                stage(i + 1)
            s.sync()
        n = s.end()
        assert n == len(want)
        got = s.fetch(n, want_images=True)
        assert np.array_equal(got.images, want.images) and np.array_equal(got.positions, want.positions)
        assert np.array_equal(got.region_of, want.region_of) and got.keys == want.keys
        assert np.array_equal(got.probs, want.probs)          # same kernels on the same rows; chunk boundaries do not matter
        rec = rec_t.cpu().numpy()[:n * PRED_RECORD.itemsize].view(PRED_RECORD)
        assert np.array_equal(rec, wrec), mode
    # capacity too small: the session reports the need instead of overrunning
    from pepper_b200._lib import PepperB200Error
    from pepper_b200.abi import PB_ERR_CAPACITY
    s = caller.stream(params, 100)
    s.stage_device(dreads, 0, n_reg, 0)
    with pytest.raises(PepperB200Error) as ei:
        s.run(flush=True)
    assert ei.value.rc == PB_ERR_CAPACITY
    caller.close()


def _rank_main(rank, world, port, q, paths=None):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from oracle import nets
    from pepper_b200.abi import HostReads
    from pepper_b200.dist import DistributedVariantCaller
    from pepper_b200.pipeline import DeviceReads
    reads, regions = _workload()
    params = synth.ont_params()
    out = {}
    for schedule in ("static", "dynamic"):
        dvc = DistributedVariantCaller(nets.make_variant_weights(5), rank, capacity=20000, schedule=schedule, group_regions=5)
        for src_name in ("host", "device"):
            src = HostReads(reads, pin=True) if src_name == "host" else DeviceReads(reads, regions, device=rank)
            n = dvc.run(src, regions, params, seq_off=reads.seq_off)
            out[(schedule, src_name)] = (dvc.buffer.to_host().copy(), n, dict(dvc.phase_ms), dvc.buffer.registered)
        if paths is not None:                  # the same job given as files every rank opens (frontend.VariantFileSource)
            from pepper_b200.frontend import VariantFileSource
            bam, fa, iv = paths
            src = VariantFileSource(bam, fa, "ctg", iv, int(params["min_snp_baseq"]), device=rank)
            n = dvc.run(src, None, params)
            out[(schedule, "files")] = (dvc.buffer.to_host().copy(), n, dict(dvc.phase_ms), dvc.buffer.registered)
            src.close()
        dvc.close()
    q.put((rank, out))
    dist.destroy_process_group()


def test_two_rank_gather_equals_one_rank(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import nets
    from pepper_b200 import synth_files
    from pepper_b200.dist import records_from_calls
    from pepper_b200.frontend import VariantFromFiles, variant_intervals
    from pepper_b200.pipeline import VariantCaller
    reads, regions = _workload()
    caller = VariantCaller(nets.make_variant_weights(5))
    want = records_from_calls(caller.call(reads, regions, synth.ont_params()))
    caller.close()
    # the from-files job: 36 intervals of a small BAM; its 1-rank answer through the single-GPU front end
    rec, genome = synth.simulate_contig_records(40000, 30, synth.ONT, 29)
    bam, fa = str(tmp_path / "d.bam"), str(tmp_path / "d.fa")
    synth_files.write_bam(bam, [("ctg", genome.shape[0])], {0: rec})
    synth_files.write_fasta(fa, [("ctg", genome)])
    iv = variant_intervals(1000, 37000, 1000)
    with VariantFromFiles(bam, fa, nets.make_variant_weights(5)) as vf:
        want_files = records_from_calls(vf.call_stream("ctg", iv, synth.ont_params(), batch=5))
    assert want_files.shape[0] > 100
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, q, (bam, fa, iv))) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
    for key in res[0]:
        n_tot, g_tot = 0, 0
        from_files = key[1] == "files"
        for rank in range(world):
            rec, n, phases, registered = res[rank][key]
            assert np.array_equal(rec, want_files if from_files else want), (key, rank)
            n_tot += n
            g_tot += phases["groups"]
            assert (phases["network_ms"] > 0) == (n > 0)           # under the dynamic schedule a rank may end up with no group at all
        from pepper_b200.dist import plan_groups, plan_groups_tapered
        n_units = len(iv) if from_files else 72
        n_groups = len(plan_groups_tapered(n_units, 5, world)) if key[0] == "dynamic" else len(plan_groups(n_units, 5))
        assert n_tot == (want_files if from_files else want).shape[0] and g_tot == n_groups           # every group of the plan run exactly once
