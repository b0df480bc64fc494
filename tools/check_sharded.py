"""torchrun --nproc-per-node N tools/check_sharded.py : the view-sharded multi-GPU schedule (NCCL max all-reduce +
sum reduce-scatter + result all-gather) against the single-GPU schedule on the same inputs (rank 0 computes both):
the depth map and its confidence map (prob_map_up)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
import atvsnet_b200 as A

rank, world, lr = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
os.environ['NCCL_DEBUG'] = 'WARN'
torch.cuda.set_device(lr)
dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', lr))
nv, D, h, w = 5, 32, 48, 64
A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:%d' % lr)
cams = torch.from_numpy(A.synthetic.orbit_cams(nv, h, w, D)[None]).cuda()
feats = torch.from_numpy(A.synthetic.smooth_features(nv, h, w, 32, seed=3)[None]).cuda()
res = {}
for prec in ('fp32', 'fp16'):
    A.FLAGS.precision = prec
    sh = A.pipeline.run_multiview(feats, cams, D, siamese=False, group=dist.group.WORLD, rank=rank, world=world,
                                  confidence=True)
    torch.cuda.synchronize()
    if rank == 0:
        one = A.pipeline.run_multiview(feats, cams, D, siamese=False, confidence=True)
        rng_ = float(cams[0, 0, 1, 3, 1]) * (D - 1)
        res[prec] = dict(depth_mae_over_range=float((sh['depth_up'] - one['depth_up']).abs().mean()) / rng_,
                         depth_max_over_range=float((sh['depth_up'] - one['depth_up']).abs().max()) / rng_,
                         prob_mae=float((sh['prob_map_up'] - one['prob_map_up']).abs().mean()),
                         prob_frac_over_1e5=float(((sh['prob_map_up'] - one['prob_map_up']).abs() > 1e-5).float().mean()),
                         cost_rel=float((sh['cost_volume_agg'].float() - one['cost_volume_agg'].float()).abs().max() /
                                        one['cost_volume_agg'].float().abs().max()))
if rank == 0:
    print(json.dumps(dict(world=world, **res)))
    assert res['fp32']['depth_max_over_range'] < 1e-5 and res['fp32']['cost_rel'] < 1e-5, res
    assert res['fp16']['depth_mae_over_range'] < 2e-3, res
    # confidence (in [0, 3]) to the same bounds as the depth, except that fp32 counts the pixels off by more than 1e-5
    # instead of taking the max: where the estimate sits on an integer plane index, a last-bit difference in the depth
    # moves the 4-tap window of get_propability_map by one plane
    assert res['fp32']['prob_frac_over_1e5'] < 1e-3 and res['fp16']['prob_mae'] < 2e-3, res
dist.barrier()
dist.destroy_process_group()
