"""Child process of tests/test_gpu_bgzf_inflate.py: tests/shim_bam_driver.py (typing() with HGT_NATIVE_INTAKE=1 on BAM
alignment files) with sam_intake.inflate_bgzf counted.  Prints shim_bam_driver.py's lines and then
"INFLATE_CALLS <calls> <kernels>": the GPU inflate calls typing() made and the kernels the context launched inside them.

usage: shim_bgzf_driver.py <golden name> <work dir>"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)


def main():
    import _hgt_path
    _hgt_path.load()
    import shim_bam_driver
    from hisatgenotype_b200 import _lib, sam_intake

    inflate = sam_intake.inflate_bgzf
    kernels = []

    def counted(streams, device=None):
        ctx = _lib.ctx(device)
        k0 = _lib.lib().hgt_launch_count(ctx)
        out = inflate(streams, device)
        kernels.append(_lib.lib().hgt_launch_count(ctx) - k0)
        return out

    sam_intake.inflate_bgzf = counted  # read_alignment looks the name up at call time
    shim_bam_driver.main()
    print("INFLATE_CALLS %d %d" % (len(kernels), sum(kernels)))


if __name__ == "__main__":
    main()
