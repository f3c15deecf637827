// AmbientOcclusionNative.cs -- the C# host a MiniEngineAO maintainer would drop next to
// Assets/MiniEngineAO/AmbientOcclusion.cs to route the compute path through libmeao (include/meao.h).
//
// SOURCE ONLY: this image has no C# toolchain (dotnet / mono / mcs / csc are absent, SURVEY.md 8c), so
// this file is neither compiled nor tested here; the Python host miniengineao_b200/ambient_occlusion.py
// is its executable twin and exercises exactly the same entry points.
//
// What changes relative to the reference component:
//   * the parameter surface (AmbientOcclusion.cs:20-68), CheckPropertiesChanged (:104-113) and the
//     LateUpdate re-plan triggers (:329-350) are kept verbatim in spirit;
//   * PushDownsampleCommands / PushRenderCommands x4 / PushUpsampleCommands x4 (:604-785) are replaced
//     by ONE CommandBuffer.IssuePluginEvent that replays libmeao's captured CUDA graph;
//   * texture interop (D3D <-> CUDA) is engine specific and out of scope: the plugin consumes / produces
//     linear device buffers (cudaGraphicsD3D11RegisterResource would map the depth and AO textures).

using System;
using System.Runtime.InteropServices;
using UnityEngine;
using UnityEngine.Rendering;

namespace MiniEngineAO
{
    internal static class MeaoNative
    {
        const string Lib = "meao";   // libmeao.so / meao.dll

        [StructLayout(LayoutKind.Sequential)]
        public struct MeaoParams
        {
            public float noise_filter_tolerance, blur_tolerance, upsample_tolerance, thickness_modifier, intensity;
            public int debug, ambient_only;
        }

        [StructLayout(LayoutKind.Sequential)]
        public struct MeaoCamera
        {
            public float near_clip, far_clip, tan_half_fov_h;
            public int reversed_z;
        }

        [StructLayout(LayoutKind.Sequential)]
        public struct MeaoDeviceCfg { public int device; public uint flags; }

        // Variants the reference ships in its shaders but never selects (meao.h: MeaoVariants); all zero = reference behaviour.
        [StructLayout(LayoutKind.Sequential)]
        public struct MeaoVariants { public int single_pass_stereo, sample_exhaustively, high_quality_mask, single_scale; }

        [DllImport(Lib)] public static extern int meao_create(ref MeaoDeviceCfg cfg, out IntPtr ctx);
        [DllImport(Lib)] public static extern void meao_destroy(IntPtr ctx);
        [DllImport(Lib)] public static extern IntPtr meao_last_error(IntPtr ctx);
        [DllImport(Lib)] public static extern int meao_set_params(IntPtr ctx, ref MeaoParams p);
        [DllImport(Lib)] public static extern int meao_set_variants(IntPtr ctx, ref MeaoVariants v);
        [DllImport(Lib)] public static extern int meao_set_camera(IntPtr ctx, ref MeaoCamera c);
        [DllImport(Lib)] public static extern int meao_resize(IntPtr ctx, int width, int height);
        [DllImport(Lib)] public static extern int meao_render(IntPtr ctx, IntPtr depthDev, int depthKind, IntPtr aoOutDev, IntPtr stream);
        [DllImport(Lib)] public static extern int meao_render_host(IntPtr ctx, float[] depth, int depthKind, byte[] aoOut);
        [DllImport(Lib)] public static extern int meao_reserve_batch(IntPtr ctx, int frames);
        [DllImport(Lib)] public static extern int meao_render_batch(IntPtr ctx, IntPtr depthDev, int depthKind, int frames, IntPtr aoOutDev, IntPtr stream);
        [DllImport(Lib)] public static extern int meao_get_batch_buffer(IntPtr ctx, int frame, int bufferId, IntPtr hostOut, UIntPtr hostBytes);
        [DllImport(Lib)] public static extern int meao_bind_event(IntPtr ctx, int eventId, IntPtr depthDev, int depthKind, IntPtr aoOutDev, IntPtr stream);
        [DllImport(Lib)] public static extern IntPtr meao_get_render_event_func();
        [DllImport(Lib)] public static extern int meao_composite_framebuffer(IntPtr ctx, IntPtr aoDev, IntPtr colorDev, int colorFormat, IntPtr stream);
        [DllImport(Lib)] public static extern int meao_composite_gbuffer(IntPtr ctx, IntPtr aoDev, IntPtr gbuffer0Dev, IntPtr gbuffer3Dev, int gbuffer3Format, IntPtr stream);
        [DllImport(Lib)] public static extern int meao_composite_debug(IntPtr ctx, IntPtr viewR8Dev, IntPtr colorDev, int colorFormat, IntPtr stream);   // AO.cs:826-829
        [DllImport(Lib)] public static extern int meao_get_buffer(IntPtr ctx, int bufferId, IntPtr hostOut, UIntPtr hostBytes);
        [DllImport(Lib)] public static extern int meao_debug_view(IntPtr ctx, int bufferId, IntPtr outR8Dev, IntPtr stream);   // AO.cs:787-820

        public static void Check(IntPtr ctx, int rc)
        {
            if (rc < 0) throw new InvalidOperationException("libmeao: " + Marshal.PtrToStringAnsi(meao_last_error(ctx)));
        }
    }

    [ExecuteInEditMode]
    [RequireComponent(typeof(Camera))]
    public sealed class AmbientOcclusionNative : MonoBehaviour
    {
        // ---- exposed properties: same names, ranges and defaults as AmbientOcclusion.cs:20-68 ----
        [SerializeField, Range(-8, 0)] float _noiseFilterTolerance = 0;
        public float noiseFilterTolerance { get { return _noiseFilterTolerance; } set { _noiseFilterTolerance = value; } }

        [SerializeField, Range(-8, -1)] float _blurTolerance = -4.6f;
        public float blurTolerance { get { return _blurTolerance; } set { _blurTolerance = value; } }

        [SerializeField, Range(-12, -1)] float _upsampleTolerance = -12;
        public float upsampleTolerance { get { return _upsampleTolerance; } set { _upsampleTolerance = value; } }

        [SerializeField, Range(1, 10)] float _thicknessModifier = 1;
        public float thicknessModifier { get { return _thicknessModifier; } set { _thicknessModifier = value; } }

        [SerializeField, Range(0, 2)] float _intensity = 1;
        public float intensity { get { return _intensity; } set { _intensity = value; } }

        [SerializeField, Range(0, 17)] int _debug;

        [SerializeField] bool _ambientOnly = true;
        public bool ambientOnly { get { return _ambientOnly; } set { _ambientOnly = value; } }

        // ---- not in the reference inspector: the shader variants Render.compute / Upsample.compute ship but AO.cs never selects ----
        [SerializeField] bool _sampleExhaustively;             // Render.compute:144-159, AmbientOcclusion.cs:709-715 (FIXME there)
        [SerializeField, Range(0, 15)] int _highQualityMask;   // bit k-1: Render kernel "main" on level k + Upsample "main_premin*"
        int _drawCountPerFrame;                                // AmbientOcclusion.cs:289, 349-355: single-pass stereo detection
        void OnPreRender() { _drawCountPerFrame++; }
        bool singlePassStereoEnabled                           // AmbientOcclusion.cs:392-401
        {
            get { return _camera != null && _camera.stereoEnabled && _camera.targetTexture == null && _drawCountPerFrame == 1; }
        }

        const int kEventId = 0x4d41;   // "MA"

        Camera _camera;
        IntPtr _ctx = IntPtr.Zero;
        CommandBuffer _renderCommand;
        IntPtr _depthDev = IntPtr.Zero, _aoDev = IntPtr.Zero;   // mapped by the engine-specific interop layer
        IntPtr _stream = IntPtr.Zero;                           // cudaStream_t the plugin event renders on (ABI 3; Zero = legacy default stream)

        void LateUpdate()
        {
            if (_camera == null)
            {
                _camera = GetComponent<Camera>();
                _camera.depthTextureMode = DepthTextureMode.Depth;          // AmbientOcclusion.cs:447
            }
            if (_ctx == IntPtr.Zero)
            {
                var cfg = new MeaoNative.MeaoDeviceCfg { device = 0, flags = 0 };
                MeaoNative.Check(IntPtr.Zero, MeaoNative.meao_create(ref cfg, out _ctx));
            }

            // CheckPropertiesChanged + CheckBaseDimensions live inside the plugin: the setters return 1
            // when the plan was dirtied (AmbientOcclusion.cs:104-113, 338-341).
            var p = new MeaoNative.MeaoParams
            {
                noise_filter_tolerance = _noiseFilterTolerance, blur_tolerance = _blurTolerance,
                upsample_tolerance = _upsampleTolerance, thickness_modifier = _thicknessModifier,
                intensity = _intensity, debug = _debug, ambient_only = _ambientOnly ? 1 : 0
            };
            var rebuild = MeaoNative.meao_set_params(_ctx, ref p) == 1;

            var cam = new MeaoNative.MeaoCamera
            {
                near_clip = _camera.nearClipPlane, far_clip = _camera.farClipPlane,          // :563
                tan_half_fov_h = 1 / _camera.projectionMatrix[0, 0],                         // :570-573
                reversed_z = SystemInfo.usesReversedZBuffer ? 1 : 0                          // :564
            };
            MeaoNative.Check(_ctx, MeaoNative.meao_set_camera(_ctx, ref cam));
            var stereo = singlePassStereoEnabled;
            var variants = new MeaoNative.MeaoVariants
            {
                single_pass_stereo = stereo ? 1 : 0,                                         // :680
                sample_exhaustively = _sampleExhaustively ? 1 : 0, high_quality_mask = _highQualityMask,
                single_scale = 0                                                             // BASELINE configs[0] plumbing mode; the component never selects it
            };
            rebuild |= MeaoNative.meao_set_variants(_ctx, ref variants) == 1;
            rebuild |= MeaoNative.meao_resize(_ctx, _camera.pixelWidth * (stereo ? 2 : 1), _camera.pixelHeight) == 1;   // :338-341
            rebuild |= !Application.isPlaying;                                               // :345
            _drawCountPerFrame = 0;                                                          // :349

            if (rebuild || _renderCommand == null) RebuildCommandBuffers();
        }

        void RebuildCommandBuffers()
        {
            if (_renderCommand == null) _renderCommand = new CommandBuffer { name = "SSAO" };   // :481-482
            else _camera.RemoveCommandBuffer(CameraEvent.BeforeImageEffects, _renderCommand);
            _renderCommand.Clear();
            // (engine-specific: map _CameraDepthTexture and the R8 AO render texture to _depthDev / _aoDev)
            MeaoNative.Check(_ctx, MeaoNative.meao_bind_event(_ctx, kEventId, _depthDev, 0 /* MEAO_DEPTH_RAW_F32 */, _aoDev, _stream));
            // one plugin event replaces the ten DispatchCompute calls recorded by :511-531
            _renderCommand.IssuePluginEvent(MeaoNative.meao_get_render_event_func(), kEventId);
            _camera.AddCommandBuffer(CameraEvent.BeforeImageEffects, _renderCommand);          // :421
        }

        // Offline use (e.g. baking AO for a recorded depth sequence): `frames` camera-sized depth frames stacked tightly in device
        // memory -> as many R8 AO frames, one graph replay.  Reserve the largest batch once, outside per-frame work.
        public void RenderBatch(IntPtr depthDev, int depthKind, int frames, IntPtr aoOutDev, IntPtr stream)
        {
            MeaoNative.Check(_ctx, MeaoNative.meao_render_batch(_ctx, depthDev, depthKind, frames, aoOutDev, stream));
        }

        void OnDisable()
        {
            if (_renderCommand != null && _camera != null)
                _camera.RemoveCommandBuffer(CameraEvent.BeforeImageEffects, _renderCommand);
        }

        void OnDestroy()
        {
            if (_ctx != IntPtr.Zero) { MeaoNative.meao_destroy(_ctx); _ctx = IntPtr.Zero; }    // :357-381
            if (_renderCommand != null) { _renderCommand.Dispose(); _renderCommand = null; }
        }
    }
}
