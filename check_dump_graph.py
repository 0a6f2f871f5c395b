import sys
import bench
from sslam_b200.pipeline import FrontEnd
seen = {}
_capture, _dump = FrontEnd.capture, bench.dump_outputs


def capture(self, fn, *a, **kw):
    replay, out = _capture(self, fn, *a, **kw)
    seen["feats"], seen["lists"] = out[0], out[1:4]
    return replay, out


def dump(path, per_frame, per_pair, descriptors):
    f = seen["feats"]
    same = (per_frame["keypoints"] is f["keypoints_pixel"] and per_frame["scores"] is f["scores"]
            and descriptors is f["descriptors"] and per_pair["pairs"].data_ptr() != 0)
    sys.stderr.write(f"DUMP_FROM_GRAPH_BANK={same}\n")
    assert same
    _dump(path, per_frame, per_pair, descriptors)


FrontEnd.capture, bench.dump_outputs = capture, dump
sys.argv = ["bench.py"] + sys.argv[1:]
bench.main()
