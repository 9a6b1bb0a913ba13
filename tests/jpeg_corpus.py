"""Seeded JPEG corpus shared by tests/test_jpeg_cpu.py and tests/test_gpu_jpeg.py."""
import cv2
import numpy as np

from oracle import synth


def corpus(seed=0):
    """The seeded corpus the tests compare with cv2: ``(image, imencode params, tag)`` over qualities 50 / 90 / 100, sampling
    4:4:4 / 4:2:2 / 4:2:0 / 4:4:0 / 4:1:1, grayscale, restart intervals 1 and 7, optimised Huffman tables, sizes from 1x1 to
    720x1280, smooth and noisy content."""
    rng = np.random.default_rng(seed)
    samp = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
            "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}

    def image(h, w, noisy, k):
        if noisy:
            return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        return synth.smooth_image(h, w, seed=seed * 1000 + k)

    out = []
    k = 0
    for h, w in ((1, 1), (2, 2), (3, 17), (37, 61)):
        for q in (50, 90, 100):
            for s, f in samp.items():
                for noisy in (False, True):
                    k += 1
                    out.append((image(h, w, noisy, k), [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, f],
                                "%dx%d q%d %s %s" % (h, w, q, s, "noisy" if noisy else "smooth")))
    for h, w in ((3, 17), (37, 61), (70, 45)):
        for q in (50, 90, 100):
            k += 1
            g = cv2.cvtColor(image(h, w, q == 90, k), cv2.COLOR_BGR2GRAY)
            out.append((g, [cv2.IMWRITE_JPEG_QUALITY, q], "%dx%d q%d gray" % (h, w, q)))
    for rst in (1, 7):
        for s in ("420", "444", "411"):
            for h, w in ((37, 61), (130, 97)):
                k += 1
                out.append((image(h, w, k % 2 == 0, k), [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp[s],
                                                         cv2.IMWRITE_JPEG_RST_INTERVAL, rst], "%dx%d rst%d %s" % (h, w, rst, s)))
    for s in ("420", "422", "440"):
        k += 1
        out.append((image(61, 37, s == "422", k), [cv2.IMWRITE_JPEG_QUALITY, 75, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp[s],
                                                   cv2.IMWRITE_JPEG_OPTIMIZE, 1], "61x37 optimize %s" % s))
    big = [((513, 513), 90, "420", False, 0), ((513, 513), 50, "411", True, 0), ((513, 513), 100, "440", False, 0),
           ((720, 1280), 90, "420", False, 0), ((720, 1280), 90, "422", False, 7)]
    for (h, w), q, s, noisy, rst in big:
        k += 1
        p = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp[s]]
        if rst:
            p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
        out.append((image(h, w, noisy, k), p, "%dx%d q%d %s rst%d" % (h, w, q, s, rst)))
    return out
