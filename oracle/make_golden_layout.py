"""Parameter layout of the reference's networks -> tests/golden/reference_layout.json.

    python oracle/make_golden_layout.py <reference checkout>

Builds the reference's own lib/net/pointnet2_msg.py::Pointnet2MSG (input_channels=0) and lib/net/point_rcnn.py::PointRCNN
(tools/cfgs/default.yaml, RPN + RCNN, TEST mode) on the CPU, on top of pointrcnn_b200.dropin (the reference's CUDA
extensions are not built), and stores every state_dict entry's name and shape in order, plus the parameter count.
"""
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main(ref):
    warnings.filterwarnings("ignore")
    sys.path[:0] = [ref, os.path.join(ref, "lib", "net"), ROOT]
    import pointrcnn_b200.dropin as d
    d.activate(compat=True)
    from lib.config import cfg, cfg_from_file
    cfg_from_file(os.path.join(ref, "tools", "cfgs", "default.yaml"))
    import lib.net.pointnet2_msg as pointnet2_msg
    cfg.RPN.ENABLED = True
    cfg.RCNN.ENABLED = True
    from lib.net.point_rcnn import PointRCNN

    def layout(net):
        return [[k, list(v.shape)] for k, v in net.state_dict().items()]
    rcnn = PointRCNN(num_classes=2, use_xyz=True, mode="TEST")
    out = {"Pointnet2MSG(input_channels=0)": layout(pointnet2_msg.Pointnet2MSG(input_channels=0)),
           "PointRCNN(num_classes=2, mode=TEST)": layout(rcnn),
           "PointRCNN parameters": sum(p.numel() for p in rcnn.parameters())}
    path = os.path.join(ROOT, "tests", "golden", "reference_layout.json")
    with open(path, "w") as f:      # one state_dict entry per line
        f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), "[\n" + ",\n".join(json.dumps(e) for e in v) + "\n]"
                                               if isinstance(v, list) else json.dumps(v)) for k, v in out.items()) + "\n}\n")
    print(path)


if __name__ == "__main__":
    main(sys.argv[1])
