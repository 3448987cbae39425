"""Which loops of the NMS segment kernel do the oracle-checked tests of the suite reach?

Runs the given test files in this process with ``ops.nms`` wrapped: after every eager call it reads the kernel's four
work counters back from the workspace (layout and dealing restated in tests/test_gpu_nms_stage.py) and records whether
the segment list ran on tickets (more entries than segment CTAs) and whether the packed CTAs strided over more than one
group each.  Graph captures are passed through unread.

    python -m profiles.nms_dealing_probe OUT.json tests/test_gpu_random.py tests/test_gpu_parity.py ...
"""
import json
import os
import sys

import pytest
import torch

from pytorch_yolo_b200 import ops
from tests.test_gpu_nms_stage import DEFAULT_RESIDENCY, PACK_SLOT_BITS, SMALL_SEG, read_work_count


def main():
    out_path, files = sys.argv[1], sys.argv[2:]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    calls = []
    orig = ops.nms

    def probed(buf, nms_thres, out, out_row, out_ptrs=None, step=None, seg_warps_per_sm=0):
        orig(buf, nms_thres, out, out_row, out_ptrs=out_ptrs, step=step, seg_warps_per_sm=seg_warps_per_sm)
        if torch.cuda.is_current_stream_capturing() or buf.batch == 0:
            return
        wc = read_work_count(buf)
        res = seg_warps_per_sm if 1 <= seg_warps_per_sm <= 32 else DEFAULT_RESIDENCY
        seg_ctas = min(buf.batch * buf.nc, sms * res)
        pack_ok = buf.mpc >= SMALL_SEG and buf.cap <= 1 << PACK_SLOT_BITS and buf.nc <= 0xFFFF
        packed = seg_ctas if pack_ok else 0
        calls.append(dict(test=os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0], batch=buf.batch, nc=buf.nc,
                          mpc=buf.mpc, residency=res, work_count=wc, seg_ctas=seg_ctas, packed_ctas=packed,
                          tickets=wc[3] > seg_ctas, stride=wc[2] > packed))

    ops.nms = probed
    rc = pytest.main(["-q", "-m", "gpu", "-p", "no:cacheprovider", *files])
    ops.nms = orig
    summary = dict(calls=len(calls), with_tickets=sum(c["tickets"] for c in calls),
                   with_stride=sum(c["stride"] for c in calls),
                   max_segs_over_ctas=max((c["work_count"][3] / c["seg_ctas"] for c in calls), default=0),
                   max_groups_over_ctas=max((c["work_count"][2] / max(1, c["packed_ctas"]) for c in calls), default=0),
                   pytest_exit=int(rc), files=files)
    with open(out_path, "w") as f:
        json.dump(dict(summary=summary, engaged=[c for c in calls if c["tickets"] or c["stride"]]), f, indent=1)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
