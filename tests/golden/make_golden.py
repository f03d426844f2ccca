"""Regenerates tests/golden/ from a checkout of the reference (swift-png), given as the only argument:

    python tests/golden/make_golden.py PATH-TO-SWIFT-PNG

The tests never read the reference itself, so everything they need from its fixtures is committed here:

  pngsuite/*.png            the reference's PngSuite inputs (Sources/PNGIntegrationTests/Inputs/Common)
  invalid/*.png             its malformed inputs              (.../Inputs/Invalid)
  pngsuite_rgba.json        sha256 + size of each golden      (.../RGBA/<name>.png.rgba, RGBA16 LE)
  ios/*.png                 the CgBI inputs (.../Inputs/iOS) and ios_rgba.json: sha256 of the same
                            RGBA goldens after pixel.premultiplied(as: UInt8.self), which is what
                            Roundtripping.swift:206-211 compares those inputs against
  gzip/*.gz                 the gzip fixtures                 (Sources/LZ77/docs.docc/GzipCompression)
  encode/*.png (+ .json)    a subset of the reference encoder's committed level-9 outputs
                            (Tests/Outputs) with the matching Tests/Baselines inputs, and
                            sha256 digests of the concatenated IDAT payload for all 28
  outputs/*.png             more of those level-9 outputs, without their inputs: the smallest one of
                            each 8-bit pixel layout encode/ does not hold (all 28 are 4.4 MB)
"""
import hashlib
import json
import os
import shutil
import struct
import sys
import zlib

REF = sys.argv[1]
HERE = os.path.dirname(os.path.abspath(__file__))
IT = os.path.join(REF, "Sources", "PNGIntegrationTests")


def idat_of(path):
    data = open(path, "rb").read()
    at, out = 8, []
    while at < len(data):
        (n,) = struct.unpack(">I", data[at:at + 4])
        if data[at + 4:at + 8] == b"IDAT":
            out.append(data[at + 8:at + 8 + n])
        at += 12 + n
    return b"".join(out)


def main():
    for sub, dst in (("Inputs/Common", "pngsuite"), ("Inputs/Invalid", "invalid")):
        os.makedirs(os.path.join(HERE, dst), exist_ok=True)
        for f in sorted(os.listdir(os.path.join(IT, sub))):
            shutil.copyfile(os.path.join(IT, sub, f), os.path.join(HERE, dst, f))
    digests = {}
    for f in sorted(os.listdir(os.path.join(IT, "Inputs/Common"))):
        raw = open(os.path.join(IT, "RGBA", f + ".rgba"), "rb").read()
        digests[f] = {"sha256": hashlib.sha256(raw).hexdigest(), "bytes": len(raw)}
    json.dump(digests, open(os.path.join(HERE, "pngsuite_rgba.json"), "w"), indent=0, sort_keys=True)
    # iOS (CgBI) inputs: golden = RGBA<UInt16>.premultiplied(as: UInt8.self) of the common golden
    # (PNG.RGBA.swift:141-155: shift 8, q = 257, premultiply on the high bytes, alpha requantised)
    import numpy as np
    os.makedirs(os.path.join(HERE, "ios"), exist_ok=True)
    ios = {}
    for f in sorted(os.listdir(os.path.join(IT, "Inputs/iOS"))):
        shutil.copyfile(os.path.join(IT, "Inputs/iOS", f), os.path.join(HERE, "ios", f))
        px = np.frombuffer(open(os.path.join(IT, "RGBA", f + ".rgba"), "rb").read(), dtype="<u2")
        px = px.reshape(-1, 4).astype(np.uint32) >> 8
        a = px[:, 3:4]
        out = np.concatenate([(px[:, :3] * a + 127) // 255, a], axis=1) * 257
        raw = out.astype("<u2").tobytes()
        ios[f] = {"sha256": hashlib.sha256(raw).hexdigest(), "bytes": len(raw)}
    json.dump(ios, open(os.path.join(HERE, "ios_rgba.json"), "w"), indent=0, sort_keys=True)
    gz = os.path.join(REF, "Sources", "LZ77", "docs.docc", "GzipCompression")
    os.makedirs(os.path.join(HERE, "gzip"), exist_ok=True)
    for f in sorted(os.listdir(gz)):
        if f.endswith(".gz"):
            shutil.copyfile(os.path.join(gz, f), os.path.join(HERE, "gzip", f))
    # encoder goldens: digests for all, files for a small subset
    enc = {}
    os.makedirs(os.path.join(HERE, "encode"), exist_ok=True)
    keep = {"rgba8-color-photographic.png", "v8-monochrome-nonphotographic.png",
            "rgb16-color-nonphotographic.png", "indexed8-color-photographic.png"}
    sampled = {"va8-monochrome-nonphotographic.png", "rgb8-monochrome-nonphotographic.png"}
    os.makedirs(os.path.join(HERE, "outputs"), exist_ok=True)
    outs = os.path.join(REF, "Tests", "Outputs")
    for f in sorted(os.listdir(outs)):
        if not f.endswith(".png"):
            continue
        payload = idat_of(os.path.join(outs, f))
        filtered = zlib.decompress(payload)
        whole = open(os.path.join(outs, f), "rb").read()
        enc[f] = {"idat_sha256": hashlib.sha256(payload).hexdigest(), "idat_bytes": len(payload),
                  "file_sha256": hashlib.sha256(whole).hexdigest(), "file_bytes": len(whole),
                  "filtered_sha256": hashlib.sha256(filtered).hexdigest(),
                  "filtered_bytes": len(filtered)}
        if f in keep:
            shutil.copyfile(os.path.join(outs, f), os.path.join(HERE, "encode", "out-" + f))
            shutil.copyfile(os.path.join(REF, "Tests", "Baselines", f),
                            os.path.join(HERE, "encode", "in-" + f))
        if f in sampled:
            shutil.copyfile(os.path.join(outs, f), os.path.join(HERE, "outputs", f))
    json.dump(enc, open(os.path.join(HERE, "encode.json"), "w"), indent=0, sort_keys=True)


if __name__ == "__main__":
    main()
