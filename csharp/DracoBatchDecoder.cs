// csharp/DracoBatchDecoder.cs -- the reference-side binding of libdracob200.so.
//
// Drop this file into src/Draco/IO/ of B3zaleel/draco-sharp (namespace Draco.IO, next to DracoDecoder.cs).
// It keeps the reference's result types -- Draco (src/Draco/Draco.cs:9-15), DracoHeader (DracoHeader.cs:5-23),
// PointCloud (IO/PointCloud/PointCloud.cs:11-12), Mesh (IO/Mesh/Mesh.cs:7-40), PointAttribute / GeometryAttribute
// (IO/Attributes/PointAttribute.cs:7-63, GeometryAttribute.cs:10-17) and DataBuffer (IO/Core/DataBuffer.cs:7-23) --
// and adds ONE new entry point, DecodeBatch, that runs the attribute-decode hot path of every buffer on the GPU:
//
//   DracoDecoder.Decode            per buffer, CPU, single thread      (unchanged; still throws on point clouds)
//   DracoBatchDecoder.DecodeBatch  many buffers, B200, no CPU fallback (this file)
//
// The P/Invoke declarations are 1:1 with include/dracob200.h (blittable structs, no marshalling logic); the
// Python ctypes harness (draco_sharp_b200/_native.py) binds the very same symbols and is what the parity tests
// drive, because the build image has no .NET SDK (this file is therefore compiled by the maintainer, not by us).
//
// Meshes: Edgebreaker connectivity stays on the host (it is inherently sequential).  The wrapper runs the
// reference's own MeshEdgeBreakerDecoder up to the ATTRIBUTES section through the small hook shown at the bottom
// (IHostConnectivity), then hands CornerTable.{Opposite,Vertex} and the traversal maps of every attributes
// decoder to dcb_set_mesh_maps -- exactly the inputs of MeshPredictionSchemeData (MeshPredictionSchemeData.cs:5-24).
using System.Runtime.InteropServices;
using Draco.IO.Attributes;
using Draco.IO.Core;
using Draco.IO.Enums;

namespace Draco.IO;

public sealed class DracoBatchDecoder : IDisposable
{
    private const string Lib = "dracob200"; // runtimes/linux-x64/native/libdracob200.so

    // ---- include/dracob200.h ----
    [StructLayout(LayoutKind.Sequential)]
    private struct BufferInfo
    {
        public int Status, GeometryType, EncoderMethod, VersionMajor, VersionMinor, Flags;
        public uint NPoints;
        public int NAttrDecoders, NAttrs, NeedsConnectivity, Device, Reserved;
        public ulong AttrSectionOff;
    }

    [StructLayout(LayoutKind.Sequential)]
    private unsafe struct AttrInfo
    {
        public int AttType, DataType, NumComponents, Normalized;
        public uint UniqueId;
        public int SeqDecoderType, DecoderId, PredMethod, Transform, Scheme, PrecisionBits;
        public uint NEntries;
        public ulong OutBytes, OutOff, DbgOff;
        public int XfA, XfB;
        public fixed float QMin[4];
        public float QRange;
        public int QBits, Resolved;
    }

    [StructLayout(LayoutKind.Sequential)]
    private struct FaceInfo
    {
        public ulong OutOff, OutBytes, NFaces;
        public int Source, Reserved;
    }

    [DllImport(Lib)] private static extern int dcb_version();
    [DllImport(Lib)] private static extern int dcb_device_count();
    [DllImport(Lib)] private static extern IntPtr dcb_error_string(int code);
    [DllImport(Lib)] private static extern int dcb_create(int[]? deviceIds, int nDevices, out IntPtr ctx);
    [DllImport(Lib)] private static extern void dcb_destroy(IntPtr ctx);
    [DllImport(Lib)] private static extern unsafe int dcb_index(IntPtr ctx, byte** bufs, ulong* lens, int nBufs, out IntPtr batch);
    [DllImport(Lib)] private static extern int dcb_get_buffer_info(IntPtr batch, int buf, out BufferInfo info);
    [DllImport(Lib)] private static extern int dcb_get_attr_info(IntPtr batch, int buf, int attr, out AttrInfo info);
    [DllImport(Lib)] private static extern ulong dcb_batch_out_bytes(IntPtr batch);
    [DllImport(Lib)] private static extern int dcb_set_attr_section(IntPtr batch, int buf, ulong attrSectionOff, uint nPoints);
    [DllImport(Lib)] private static extern int dcb_set_limits(IntPtr ctx, ulong maxPointsPerBuffer, ulong pointsPerByte);
    // the four arrays are BORROWED by the library until the decode call returns: raw pointers of pinned arrays
    [DllImport(Lib)] private static extern unsafe int dcb_set_mesh_maps(IntPtr batch, int buf, int attrDecoder, uint* opposite, uint* cornerToVertex,
        ulong nCorners, uint* dataToCorner, ulong nEntries, int* vertexToData, ulong nVertices);
    [DllImport(Lib)] private static extern int dcb_host_connectivity(IntPtr batch, int buf);
    [DllImport(Lib)] private static extern int dcb_mesh_faces(IntPtr batch, int buf, uint[]? faces, ulong capFaces, out ulong nFaces);
    [DllImport(Lib)] private static extern int dcb_mesh_map(IntPtr batch, int buf, int attrDecoder, int which, uint[]? dst, ulong cap, out ulong n);
    [DllImport(Lib)] private static extern int dcb_index_finish(IntPtr ctx, IntPtr batch);
    [DllImport(Lib)] private static extern int dcb_set_output_order(IntPtr batch, int order);
    [DllImport(Lib)] private static extern unsafe int dcb_set_mesh_faces(IntPtr batch, int buf, uint* faces, ulong nFaces);
    [DllImport(Lib)] private static extern int dcb_set_face_output(IntPtr batch, int mode);
    [DllImport(Lib)] private static extern int dcb_get_face_info(IntPtr batch, int buf, out FaceInfo info);
    [DllImport(Lib)] private static extern unsafe int dcb_decode(IntPtr ctx, IntPtr batch, byte* hostOut, byte* hostDbg, uint flags);
    [DllImport(Lib)] private static extern unsafe int dcb_decode_scatter(IntPtr ctx, IntPtr batch, byte** outs, int nOuts, uint flags);
    [DllImport(Lib)] private static extern int dcb_status(IntPtr batch, int buf);
    [DllImport(Lib)] private static extern void dcb_batch_free(IntPtr batch);

    private IntPtr _ctx;

    /// <param name="deviceIds">CUDA ordinals to shard buffers over (default: the current device).</param>
    public DracoBatchDecoder(int[]? deviceIds = null)
    {
        var rc = dcb_create(deviceIds, deviceIds?.Length ?? 0, out _ctx);
        if (rc != 0)
        {
            // DCB_ERR_NO_DEVICE included: there is deliberately no CPU fallback behind this class.
            throw new InvalidOperationException($"libdracob200: {Marshal.PtrToStringAnsi(dcb_error_string(rc))}");
        }
    }

    /// <summary>Per-buffer plausibility limits (dcb_set_limits): a forged point count fails its own buffer.</summary>
    public void SetLimits(ulong maxPointsPerBuffer = 0, ulong pointsPerByte = 4096) => Check(dcb_set_limits(_ctx, maxPointsPerBuffer, pointsPerByte));

    /// <summary>Host connectivity hook for meshes; null = the library's own host Edgebreaker helper is used.</summary>
    public IHostConnectivity? Connectivity { get; set; }

    /// <summary>
    /// Decodes every buffer. A malformed buffer yields a null entry and its exception in <paramref name="errors"/>
    /// (the same exception type DracoDecoder.Decode would have thrown for it); it never poisons its neighbours.
    /// <paramref name="pointOrder"/>: attributes of Edgebreaker meshes arrive with one value per point (DCB_ORDER_POINTS,
    /// the point-to-value map applied on the GPU) and carry the identity mapping; otherwise they hold the unique entries
    /// and <see cref="IHostConnectivity.ApplyPointMapping"/> supplies the map.
    /// <paramref name="facesInArena"/>: the faces of every mesh come out of the output arena (DCB_FACES_ARENA; plain
    /// sequential indices decoded on the GPU) and the decode runs into one arena instead of the per-attribute scatter.
    /// </summary>
    public unsafe Draco?[] DecodeBatch(IReadOnlyList<ReadOnlyMemory<byte>> buffers, out Exception?[] errors, bool pointOrder = false,
                                       bool facesInArena = false)
    {
        int n = buffers.Count;
        var result = new Draco?[n];
        errors = new Exception?[n];
        var pins = new System.Buffers.MemoryHandle[n];
        // heap, not stack: batches of 200,000 buffers are a normal case (BASELINE configs[4])
        var ptrs = (byte**)NativeMemory.Alloc((nuint)Math.Max(n, 1), (nuint)sizeof(byte*));
        var lens = (ulong*)NativeMemory.Alloc((nuint)Math.Max(n, 1), (nuint)sizeof(ulong));
        byte** outs = null;
        var mapPins = new List<GCHandle>();  // connectivity maps stay pinned until the decode has consumed them
        IntPtr batch = IntPtr.Zero;
        try
        {
            for (int k = 0; k < n; ++k)
            {
                pins[k] = buffers[k].Pin();
                ptrs[k] = (byte*)pins[k].Pointer;
                lens[k] = (ulong)buffers[k].Length;
            }
            Check(dcb_index(_ctx, ptrs, lens, n, out batch));
            if (pointOrder) Check(dcb_set_output_order(batch, 1));  // DCB_ORDER_POINTS
            if (facesInArena) Check(dcb_set_face_output(batch, 1));  // DCB_FACES_ARENA, before the connectivity step

            // meshes: connectivity on the host, maps to the GPU
            var hostMeshes = new Mesh.Mesh?[n];
            bool anyMesh = false;
            for (int k = 0; k < n; ++k)
            {
                Check(dcb_get_buffer_info(batch, k, out var bi));
                if (bi.Status != 0 || bi.NeedsConnectivity == 0) continue;
                anyMesh = true;
                if (Connectivity == null)
                {
                    // no C# hook installed: the library's own host Edgebreaker decoder (still CPU work, still
                    // MeshEdgeBreakerDecoder.DecodeConnectivity's algorithm); faces come back through dcb_mesh_faces
                    Check(dcb_host_connectivity(batch, k));
                    continue;
                }
                HostConnectivity hc;
                try
                {
                    hc = Connectivity.DecodeConnectivity(buffers[k]);
                }
                catch (Exception e)
                {
                    // one malformed mesh fails alone: without an attribute section the library reports
                    // DCB_ERR_CONNECTIVITY for this buffer after dcb_index_finish; keep the host's own exception
                    errors[k] = e;
                    continue;
                }
                hostMeshes[k] = hc.Mesh;
                Check(dcb_set_attr_section(batch, k, (ulong)hc.AttributesSectionOffset, (uint)hc.Mesh.PointsCount));
                for (int d = 0; d < hc.Decoders.Count; ++d)
                {
                    var m = hc.Decoders[d];
                    uint* Pin<T>(T[] a) where T : unmanaged
                    {
                        var h = GCHandle.Alloc(a, GCHandleType.Pinned);
                        mapPins.Add(h);
                        return (uint*)h.AddrOfPinnedObject();
                    }
                    Check(dcb_set_mesh_maps(batch, k, d, Pin(m.Opposite), Pin(m.CornerToVertex), (ulong)m.Opposite.Length,
                        Pin(m.DataToCorner), (ulong)m.DataToCorner.Length, (int*)Pin(m.VertexToData), (ulong)m.VertexToData.Length));
                }
                // Edgebreaker meshes only: the library refuses faces for sequential meshes (their attributes are already in point
                // order).  A hook that exports no faces leaves the buffer to fail alone with DCB_ERR_MAPS.
                if ((pointOrder || facesInArena) && bi.EncoderMethod == 1 && hc.Faces != null)  // Mesh.Faces as point ids, borrowed (pinned) like the maps
                {
                    var h = GCHandle.Alloc(hc.Faces, GCHandleType.Pinned);
                    mapPins.Add(h);
                    Check(dcb_set_mesh_faces(batch, k, (uint*)h.AddrOfPinnedObject(), (ulong)hc.Faces.Length / 3));
                }
            }
            if (anyMesh) Check(dcb_index_finish(_ctx, batch));

            // one DataBuffer per attribute: the GPU writes straight into their pinned byte arrays
            byte[]? arena = null;
            var attrs = new List<(int buf, AttrInfo info, byte[] data, GCHandle pin)>();
            for (int k = 0; k < n; ++k)
            {
                Check(dcb_get_buffer_info(batch, k, out var bi));
                for (int a = 0; a < bi.NAttrs; ++a)
                {
                    Check(dcb_get_attr_info(batch, k, a, out var ai));
                    var data = new byte[bi.Status == 0 ? (int)ai.OutBytes : 0];
                    attrs.Add((k, ai, data, GCHandle.Alloc(data, GCHandleType.Pinned)));
                }
            }
            try
            {
                outs = (byte**)NativeMemory.Alloc((nuint)Math.Max(attrs.Count, 1), (nuint)sizeof(byte*));
                if (facesInArena)
                {
                    // dcb_decode_scatter has no slot for faces: one arena, sliced into the DataBuffers afterwards.  A .NET
                    // array holds at most Array.MaxLength bytes (about 2 GB): larger batches must be split by the caller
                    // (checked below rather than truncated)
                    ulong arenaBytes = dcb_batch_out_bytes(batch);
                    if (arenaBytes > (ulong)Array.MaxLength)
                        throw new InvalidOperationException($"DecodeBatch(facesInArena): output arena of {arenaBytes} bytes exceeds one .NET array; split the batch");
                    arena = new byte[arenaBytes];
                    fixed (byte* p = arena) Check(dcb_decode(_ctx, batch, p, null, 0));
                    foreach (var a in attrs)
                        if (a.data.Length > 0) Array.Copy(arena, (long)a.info.OutOff, a.data, 0, a.data.Length);
                }
                else
                {
                    for (int i = 0; i < attrs.Count; ++i)
                        outs[i] = attrs[i].data.Length > 0 ? (byte*)attrs[i].pin.AddrOfPinnedObject() : null;
                    Check(dcb_decode_scatter(_ctx, batch, outs, attrs.Count, 0));
                }
            }
            finally
            {
                foreach (var a in attrs) a.pin.Free();
            }

            // wrap into the reference's types
            int cursor = 0;
            for (int k = 0; k < n; ++k)
            {
                Check(dcb_get_buffer_info(batch, k, out var bi));
                int status = dcb_status(batch, k);
                int first = cursor;
                cursor += bi.NAttrs;
                if (status != 0)
                {
                    errors[k] ??= ToException(status);  // a host connectivity exception, if any, is the more precise one
                    continue;
                }
                PointCloud.PointCloud pc = hostMeshes[k] ?? (bi.GeometryType == 1 ? new Mesh.Mesh() : new PointCloud.PointCloud());
                pc.PointsCount = (int)bi.NPoints;
                if (hostMeshes[k] == null && pc is Mesh.Mesh arenaMesh && arena != null)
                {
                    // faces from the output arena: u32 point ids, 3 per face (dcb_get_face_info); offsets stay 64-bit until
                    // the slice, which the array bounds check
                    Check(dcb_get_face_info(batch, k, out var fi));
                    var ids = MemoryMarshal.Cast<byte, uint>(arena.AsSpan(checked((int)fi.OutOff), checked((int)fi.OutBytes)));
                    for (long f = 0; f < (long)fi.NFaces; ++f)
                        arenaMesh.SetFace((int)f, new[] { (int)ids[(int)(3 * f)], (int)ids[(int)(3 * f + 1)], (int)ids[(int)(3 * f + 2)] });
                }
                else if (hostMeshes[k] == null && pc is Mesh.Mesh mesh)
                {
                    // the library decoded the connectivity: its faces (Mesh.SetFace, MeshEdgeBreakerDecoder.cs:622-636)
                    Check(dcb_mesh_faces(batch, k, null, 0, out ulong nFaces));
                    var faces = new uint[nFaces * 3];
                    Check(dcb_mesh_faces(batch, k, faces, nFaces, out nFaces));
                    for (int f = 0; f < (int)nFaces; ++f)
                        mesh.SetFace(f, new[] { (int)faces[3 * f], (int)faces[3 * f + 1], (int)faces[3 * f + 2] });
                }
                bool pointRows = pointOrder && bi.GeometryType == 1 && bi.EncoderMethod == 1;
                var list = new List<PointAttribute>();
                for (int a = 0; a < bi.NAttrs; ++a)
                {
                    var (_, ai, data, _) = attrs[first + a];
                    var buffer = new DataBuffer();
                    buffer.Update(data); // DataBuffer.Update<byte> (DataBuffer.cs:13-18)
                    long stride = (long)Constants.DataTypeLength((DataType)ai.DataType) * ai.NumComponents;
                    var ga = new GeometryAttribute((GeometryAttributeType)ai.AttType, buffer, (byte)ai.NumComponents,
                        (DataType)ai.DataType, ai.Normalized != 0, stride, 0) { UniqueId = ai.UniqueId };
                    var pa = new PointAttribute(ga);
                    pa.Reset(0);                        // keeps DataType / NumComponents, then:
                    pa.ResetBuffer(buffer, stride, 0);  // ... attach the decoded bytes (GeometryAttribute.cs:55-60)
                    typeof(PointAttribute).GetProperty(nameof(PointAttribute.UniqueEntriesCount))!.SetValue(pa, pointRows ? (uint)(ai.OutBytes / (ulong)stride) : ai.NEntries);
                    if (bi.GeometryType == 0 || pointRows) pa.SetIdentityMapping(); // LinearSequencer / point order: row p is point p
                    else Connectivity?.ApplyPointMapping(k, ai.DecoderId, pa); // MeshTraversalSequencer.UpdatePointToAttributeIndexMapping
                    pc.AddAttribute(pa);
                    list.Add(pa);
                }
                result[k] = new Draco
                {
                    Header = new DracoHeader((byte)bi.VersionMajor, (byte)bi.VersionMinor, (byte)bi.GeometryType,
                        (byte)bi.EncoderMethod, (ushort)bi.Flags),
                    ConnectedData = pc,
                    Attributes = list,
                };
            }
            return result;
        }
        finally
        {
            if (batch != IntPtr.Zero) dcb_batch_free(batch);
            foreach (var h in mapPins) h.Free();
            foreach (var p in pins) p.Dispose();
            NativeMemory.Free(ptrs);
            NativeMemory.Free(lens);
            if (outs != null) NativeMemory.Free(outs);
        }
    }

    // per-buffer status codes mirror the reference's exception sites (include/dracob200.h)
    private static Exception ToException(int status) => status switch
    {
        -1 => new EndOfStreamException(),
        -3 or -15 => new NotSupportedException(Marshal.PtrToStringAnsi(dcb_error_string(status))),
        _ => new InvalidDataException(Marshal.PtrToStringAnsi(dcb_error_string(status))),
    };

    private static void Check(int rc)
    {
        if (rc != 0) throw new InvalidOperationException($"libdracob200: {Marshal.PtrToStringAnsi(dcb_error_string(rc))} ({rc})");
    }

    public void Dispose()
    {
        if (_ctx != IntPtr.Zero) dcb_destroy(_ctx);
        _ctx = IntPtr.Zero;
    }
}

/// <summary>
/// What the host side contributes for meshes. The default implementation (INTEGRATION.md) subclasses
/// MeshEdgeBreakerTraversal*Decoder, calls DecodeConnectivity, reads u8 numAttributesDecoders + the
/// CreateAttributesDecoder triples (MeshEdgeBreakerDecoder.cs:640-708) so the sequencers exist, runs
/// GenerateSequence on each (MeshTraversalSequencer.cs:13-31) and exports the tables below.
/// </summary>
public interface IHostConnectivity
{
    HostConnectivity DecodeConnectivity(ReadOnlyMemory<byte> buffer);
    void ApplyPointMapping(int bufferIndex, int attributesDecoder, PointAttribute attribute);
}

public sealed class HostConnectivity
{
    public required Mesh.Mesh Mesh { get; init; }
    public required long AttributesSectionOffset { get; init; }             // DecoderBuffer position after DecodeConnectivity
    public required IReadOnlyList<HostDecoderMaps> Decoders { get; init; }  // one per attributes decoder
    public uint[]? Faces { get; init; }                                      // Mesh.Faces, 3 point ids per face: needed for point order only
}

public sealed class HostDecoderMaps
{
    public required uint[] Opposite { get; init; }        // CornerTable.Opposite(c) or the attribute corner table's (seams cut)
    public required uint[] CornerToVertex { get; init; }  // CornerTable.Vertex(c)
    public required uint[] DataToCorner { get; init; }    // MeshAttributeIndicesEncodingData.EncodedAttributeValueIndexToCornerMap
    public required int[] VertexToData { get; init; }     // MeshAttributeIndicesEncodingData.VertexToEncodedAttributeValueIndexMap
}
