"""CPU-only: the decode-only plug-ins of method ids 6 (BZIP2) and 7 (LZMA) -- their ids, compress() refusing, b''
decoding to b'' -- how the facade loads them (known for decompress, outside the chunk trial), and the
`decompress --methods` flag of the CLI."""
import pytest


def test_bz2_lzma_plugin_surface_facade_and_cli(capsys):
    import main as cli
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200.adaptive_compressor import AdaptiveCompressor
    from adaptive_compression_b200.compression_methods import BZip2Compression, LZMACompression
    assert BZip2Compression().type_id == 6 == L.BZIP2 and LZMACompression().type_id == 7 == L.LZMA
    for m in (BZip2Compression(), LZMACompression()):
        with pytest.raises(NotImplementedError):
            m.compress(b"abc")
        assert m.decompress(b"", 5) == b"" and not m.should_use(bytes(5000)) and m.calculate_overhead() == 0
    c = AdaptiveCompressor(chunk_size=4096, methods=[1, 2, 3, 6, 7])
    assert [m.type_id for m in c.compression_methods] == [1, 2, 3, 6, 7, 255]
    assert c._method_mask() == (1 << 1) | (1 << 2) | (1 << 3)
    assert "takes no part in the chunk trial" in capsys.readouterr().out
    c = AdaptiveCompressor(methods=[7, 5, 1, 6])
    assert [m.type_id for m in c.compression_methods] == [1, 5, 6, 7, 255]
    assert [m.type_id for m in AdaptiveCompressor().compression_methods] == [1, 2, 3, 4, 255]
    args = cli.build_parser().parse_args(["decompress", "a.ambc", "b.bin", "--methods", "deflate,bzip2,lzma"])
    assert cli.parse_methods(args.methods) == [5, 6, 7] and (args.input, args.output) == ("a.ambc", "b.bin")
    assert cli.build_parser().parse_args(["decompress", "a", "b"]).methods is None
    assert cli.METHOD_LABELS[6] == "BZIP2" and cli.METHOD_LABELS[7] == "LZMA"
