// GpuWalker.cs -- the reference's Walker surface (Walker/Walker.cs:25-223) for walker `index` of a GpuEnvironment batch.
// Source only (no .NET toolchain in the build image); see INTEGRATION.md.
//
// The physical body lives in the library (wb_env_batch); this class keeps the method names and meanings of Walker.cs so that
// Environment-style code reads the same: CreateCreature / Reset / Update are handled inside the fused step (they are kept as
// methods so call sites compile unchanged), GetState / GetPosition / GetChangeInPosition / GetJoints read the walker's record.
using System;
using System.Collections.Generic;
using Microsoft.Xna.Framework;
using NEA.Native;
using NEA.Rendering;
using NEA.Walker.PPO;

namespace NEA.Walker;

public sealed class GpuWalker
{
    private readonly GpuEnvironment _environment;
    private readonly int _index;
    private readonly GpuPPOAgent _brain;          // the shared brain, or null when every walker owns one
    private readonly GpuPopulation _population;   // brainPerWalker: this walker's agent is agent _index
    public bool Terminal => (_environment.Flags(_index) & 32) != 0;      // WB_FLAG_TERMINAL: Walker.Terminal (Walker.cs:23)

    internal GpuWalker(GpuEnvironment environment, int index, GpuPPOAgent brain, GpuPopulation population = null)
    {
        _environment = environment;
        _index = index;
        _brain = brain;
        _population = population;
    }

    // Walker.CreateCreature (Walker.cs:40-46): the library builds bodies, joints, association lists and gravity at wb_env_create
    public void CreateCreature() { }

    // Walker.Update (Walker.cs:49-54) is the Observe phase of the fused step: position / previous position / Terminal latch
    public void Update() { }

    // Walker.GetActions (Walker.cs:58-62)
    public PPO.Matrix GetActions(PPO.Matrix state, out PPO.Matrix logProbabilities)
        => _population == null
            ? _brain.SampleActions(state, out logProbabilities, out _, out _)
            : _population.SampleAction(_index, PPO.Matrix.GetRepresentation(state), _environment.Observations(), out logProbabilities);

    // Walker.TakeActions (Walker.cs:66-75): this walker's four torques; the library clips like Environment.cs:78
    public void TakeActions(PPO.Matrix actions)
    {
        if (actions.GetHeight() != Wb.Act) return;
        for (int k = 0; k < Wb.Act; k++) _environment.StageAction(_index, k, actions.GetValue(k, 0));
    }

    // Walker.Train (Walker.cs:79-82)
    public void Train(Trajectory trajectory, Renderer renderer)
    {
        if (_population == null) _brain.Train(trajectory, renderer);
        else _population.Train(new[] { (_index, trajectory) }, renderer);
    }

    // Walker.GetState (Walker.cs:132-152): the 12-float observation the last step produced
    public PPO.Matrix GetState() => PPO.Matrix.FromValues(_environment.Observation(_index));

    // Walker.GetPosition / GetChangeInPosition (Walker.cs:113-122): the Body's cached centroid and its change over the last step
    public Vector2 GetPosition() => _environment.Position(_index);
    public Vector2 GetChangeInPosition() => _environment.Position(_index) - _environment.PreviousPosition(_index);

    // Walker.GetJoints (Walker.cs:107-110), reduced to what callers read: the two joint points (Joint.GetPointA / GetPointB,
    // Joint.cs:44-53) and the current torque (Joint.GetTorque, :64-67) of the four joints in creation order (Walker.cs:182-187)
    public List<(Vector2 pointA, Vector2 pointB, float torque)> GetJoints()
    {
        float[] r = _environment.Record(_index);     // 92 floats, layout in include/walker_b200.h
        Vector2 V(int body, int vertex) { int f = 2 * (Offsets[body] + vertex); return new Vector2(r[f], r[f + 1]); }
        return new List<(Vector2, Vector2, float)>
        {
            (V(Body, 1), V(LLU, 4), r[88]), (V(Body, 1), V(RLU, 4), r[89]), (V(LLU, 2), V(LLL, 3), r[90]), (V(RLU, 2), V(RLL, 3), r[91]),
        };
    }

    // vertices of the five bodies for Renderer.RenderRigidObject (Rendering/Renderer.cs:90-99), list order LLL, LLU, Body, RLL, RLU
    public List<List<Vector2>> GetBodyVectors()
    {
        float[] r = _environment.Record(_index);
        var bodies = new List<List<Vector2>>();
        for (int b = 0; b < 5; b++)
        {
            var verts = new List<Vector2>();
            for (int i = 0; i < (b == Body ? 5 : 6); i++) verts.Add(new Vector2(r[2 * (Offsets[b] + i)], r[2 * (Offsets[b] + i) + 1]));
            bodies.Add(verts);
        }
        return bodies;
    }

    // Walker.Reset (Walker.cs:212-223): the fused step resets a terminal walker itself (auto_reset); an explicit call resets now
    public void Reset() => _environment.ResetWalker(_index);

    private const int LLL = 0, LLU = 1, Body = 2, RLL = 3, RLU = 4;
    private static readonly int[] Offsets = { 0, 6, 12, 17, 23 };      // first vertex of each body inside the record
}
