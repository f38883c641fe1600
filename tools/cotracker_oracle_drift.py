import os, sys, torch, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'sam-pt_b200'))
from oracle import cotracker_ref as R
from sampt_b200 import synth
def run(threads, scale=None, P=64):
    torch.set_num_threads(threads)
    sd = synth.condition_cotracker(synth.make_state_dict(R.cotracker_state_dict_shapes(), 7202), vis_bias=0.6)
    if scale is not None:
        w, b = sd["updateformer.flow_head.weight"].clone(), sd["updateformer.flow_head.bias"].clone()
        w[:2] *= scale; b[:2] *= scale
        sd["updateformer.flow_head.weight"], sd["updateformer.flow_head.bias"] = w, b
    v = synth.make_video_dict(50, 480, 854, P)
    im = torch.stack(v["image"])[None]
    with torch.no_grad():
        return R.cotracker_point_tracker_forward(sd, im, v["query_points"].reshape(1,-1,3))
for scale in (None, 1/3.0):
    t8, v8 = run(8, scale)
    t3, v3 = run(3, scale)
    d = (t8 - t3).abs()
    print("scale", scale, "oracle(8 thr) vs oracle(3 thr): max |dtraj| =", d.max().item(), "per-frame max:", [round(x,6) for x in d.amax(dim=(0,2,3)).tolist()][::7], "vis equal", torch.equal(v8, v3))
