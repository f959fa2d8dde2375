"""Child process of tests/test_gpu_bam_intake.py: the native run of shim_driver.py (HGT_NATIVE_INTAKE=1, the stand-in
samtools exits 97) with a BAM alignment file.  shim_driver.py writes each test's alignments as SAM; just before typing()
reads that file, it is rewritten in place as a BAM of the same records (tests/bam_writer.py), so typing() takes the native
BAM path.  Prints shim_driver.py's SHIM_RESULT line and then "BAM_FILES <n>", the number of files typed as BAM.

usage: shim_bam_driver.py <golden name> <work dir>"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)


def main():
    import _hgt_path
    _hgt_path.load()
    import shim_driver
    from bam_writer import write_bam
    from hisatgenotype_b200 import typing_core

    converted = []
    typing = typing_core.typing

    def typing_on_bam(*args, **kwargs):
        aln = args[typing_core._TYPING_PARAMS.index("alignment_fname")]
        with open(aln, "rb") as f:
            text = f.read().decode()
        refs, lines = [], []
        for line in text.splitlines():
            if line.startswith("@SQ"):
                tags = dict(t.split(":", 1) for t in line.split("\t")[1:])
                refs.append((tags["SN"], int(tags["LN"])))
            elif line and not line.startswith("@"):
                lines.append(line)
        with open(aln, "wb") as f:
            f.write(write_bam(lines, refs, block=4096))
        converted.append(aln)
        return typing(*args, **kwargs)

    typing_core.typing = typing_on_bam  # typing_dispatch (the drop-in's typing) looks the name up at call time
    sys.argv = [sys.argv[0], sys.argv[1], sys.argv[2], "native"]
    shim_driver.main()
    print("BAM_FILES %d" % len(converted))


if __name__ == "__main__":
    main()
