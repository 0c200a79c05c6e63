"""Loop steppers: decide when an iterative method such as ICP has converged (counterpart of pypose.utils.stepper)."""
import torch


class ReduceToBason:
    r'''Stops a loop when the relative loss decrease stays below ``decreasing`` for ``patience`` steps in a row, when
    the loss falls below ``tol``, or after ``steps`` steps.

    Args:
        steps (``int``): maximum number of steps.
        patience (``int``, optional): number of consecutive steps without a relative decrease of at least
            ``decreasing`` that stops the loop. Default: ``5``.
        decreasing (``float``, optional): relative loss decrease that resets the patience count. Default: ``1e-3``.
        tol (``float``, optional): loss below which the loop stops. Default: ``1e-5``.
        verbose (``bool``, optional): print the loss at every step and the reason for stopping. Default: ``False``.

    A batched loss meets a condition only when every element meets it.  Call ``reset()`` before re-using a stepper;
    it restarts the step count and forgets the last loss, but the patience count carries over, as in PyPose.

    Example:
        >>> stepper = ReduceToBason(steps=5, patience=2, decreasing=0.1)
        >>> x = 0.9
        >>> while stepper.continual():
        ...     x = x ** 2
        ...     stepper.step(x)
    '''
    def __init__(self, steps, patience=5, decreasing=1e-3, tol=1e-5, verbose=False):
        self.max_steps, self.patience, self.decreasing, self.tol = steps, patience, decreasing, tol
        self.verbose = verbose
        self.patience_count = 0
        self.reset()

    def reset(self):
        self.steps, self.last, self._continual = 0, torch.tensor(float('inf')), True

    def continual(self):
        return self._continual

    def step(self, loss):
        r'''Records the loss (``float`` or ``torch.Tensor``, possibly batched) of the latest iteration.'''
        if self.verbose:
            print(f"ReduceToBason step {self.steps} loss {loss!s}")
        loss = loss if torch.is_tensor(loss) else torch.tensor(loss)
        self.steps += 1
        stalled = bool(torch.all((self.last - loss) / loss < self.decreasing))
        self.patience_count = self.patience_count + 1 if stalled else 0
        self.last = loss
        # every condition that holds is reported, in this order
        for met, reason in ((bool(torch.all(loss < self.tol)), "Loss tol reached"),
                            (self.steps >= self.max_steps, "Maximum steps reached"),
                            (self.patience_count >= self.patience, "Maximum patience steps reached")):
            if met:
                self._continual = False
                if self.verbose:
                    print(f"ReduceToBason: {reason}, Quiting..")
